"""Where each T2 frame's TS bytes start in a chain's input streams (Chain.ts_bytes, plp_ts_bytes, ts_bytes_per_frame,
history_bytes), against the rule stated once more here: a stream starts on a packet boundary; a FECFRAME carries
Kbch / 8 - 10 payload bytes (the BB header takes 80 bits), 13 fewer when it opens an in-band signalling cycle (one cycle
= the PLP's FEC blocks per T2 frame); in high-efficiency mode the sync byte in front of each 187 payload bytes is not
carried, and a frame starts right behind the last payload byte of the one before.  Host-side plan only: no device."""
import pytest

import dvbt2ll_b200 as T
from dvbt2ll_b200 import configs as K

# Kbch by (framesize, code rate): EN 302 755 tables 6(a) and 6(b)
KBCH = {K.FECFRAME_NORMAL: {K.C1_2: 32208, K.C3_5: 38688, K.C2_3: 43040, K.C3_4: 48408, K.C4_5: 51648, K.C5_6: 53840},
        K.FECFRAME_SHORT: {K.C1_2: 7032, K.C3_5: 9552, K.C2_3: 10632, K.C3_4: 11712, K.C4_5: 12432, K.C5_6: 13152,
                           K.C1_3: 5232, K.C2_5: 6312}}


def ts_pos(fecframes, payload, cycle, hieff):
    """TS byte index at which FECFRAME `fecframes` of a PLP starts (cycle None: no in-band signalling)."""
    n = fecframes * payload - (13 * len(range(0, fecframes, cycle)) if cycle else 0)
    if not hieff or n == 0:
        return n
    last = n - 1                              # index of the last payload byte before the frame, in payload bytes
    return 188 * (last // 187) + 1 + last % 187 + 1


def plps_of(cfg):
    """(FEC blocks per T2 frame, payload bytes per FECFRAME) of each PLP of the chain built from cfg."""
    if cfg.get("plps"):
        qs = T.plp_params(cfg)
    else:
        qs = [dict(cfg, fecblocks=n) for n in (cfg.get("plp_fecblocks") or [cfg["fecblocks"]])]
    return [(q["fecblocks"], KBCH[q["framesize"]][q["rate"]] // 8 - 10) for q in qs]


def plp(blocks, framesize, rate, constellation, rotation):
    return dict(fecblocks=blocks, framesize=framesize, rate=rate, constellation=constellation, rotation=rotation)


S, N = K.FECFRAME_SHORT, K.FECFRAME_NORMAL
TWO_K = dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_2K, pilotpattern=K.PILOT_PP2, guardinterval=K.GI_1_8, numdatasyms=30,
             l1constellation=K.L1_MOD_QPSK, version=K.VERSION_131)
CASES = {
    "c1": dict(K.CONFIGS["c1"]),
    "c1-3blocks": dict(K.CONFIGS["c1"], fecblocks=3),
    "c1-1block": dict(K.CONFIGS["c1"], fecblocks=1),
    "c2": dict(K.CONFIGS["c2"]),
    "c2-7blocks": dict(K.CONFIGS["c2"], fecblocks=7),
    # create_multiplp: PLPs of the frame's own parameters
    "c1-2plp": dict(K.CONFIGS["c1"], plp_fecblocks=[3, 5], fecblocks=8),
    "c1-3plp": dict(K.CONFIGS["c1"], plp_fecblocks=[2, 1, 4], fecblocks=7, tiblocks=1),
    # per-PLP ModCod: framesize, rate, constellation and rotation of every PLP its own
    "c1-mix": dict(K.CONFIGS["c1"], plps=[plp(4, S, K.C4_5, K.MOD_256QAM, 1), plp(1, S, K.C1_2, K.MOD_QPSK, 0)]),
    "c1-fectype": dict(K.CONFIGS["c1"], plps=[dict(fecblocks=4), plp(1, N, K.C2_3, K.MOD_256QAM, 1)]),
    "2k-mix": dict(TWO_K, plps=[plp(7, S, K.C3_5, K.MOD_64QAM, 1), plp(2, S, K.C1_2, K.MOD_QPSK, 0)]),
}


@pytest.mark.parametrize("inband", [0, 1])
@pytest.mark.parametrize("inputmode", [K.INPUTMODE_NORMAL, K.INPUTMODE_HIEFF])
@pytest.mark.parametrize("name", sorted(CASES))
def test_chain_stream_positions(name, inputmode, inband):
    cfg = K.resolve(dict(CASES[name], inputmode=inputmode, inband=inband))
    if inband:
        cfg.update(version=K.VERSION_131)
    ch = T.Chain(cfg, max_frames=1)
    plps = plps_of(cfg)
    assert ch.num_plp == len(plps)
    hieff = inputmode == K.INPUTMODE_HIEFF

    def want(p, first_frame, n_frames):
        fpl, payload = plps[p]
        cycle = fpl if inband else None
        return (ts_pos((first_frame + n_frames) * fpl, payload, cycle, hieff)
                - ts_pos(first_frame * fpl, payload, cycle, hieff))

    assert ch.ts_bytes_per_frame == want(0, 0, 1)
    for first_frame in range(22):
        assert ch.history_bytes(first_frame) == (187 if first_frame > 0 and not hieff else 0)
        for n_frames in (1, 2, 3):
            assert ch.ts_bytes(first_frame, n_frames) == want(0, first_frame, n_frames), (first_frame, n_frames)
            for p in range(len(plps)):
                assert ch.plp_ts_bytes(p, first_frame, n_frames) == want(p, first_frame, n_frames), (p, first_frame)
