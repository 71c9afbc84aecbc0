"""Every FEC frame size, code rate, constellation and rotation through the fused chain, 16 PLPs and eight constellation
tables per T2 frame.

Seven per-PLP-ModCod chains of 16 one-block PLPs each carry two codes x the 8 (constellation, rotation) pairs, so that
together they hold each of the 14 x 4 x 2 = 112 modes once.  Each sits on its own FFT size (32K twice, normal and
extended carriers), so k_ofdm's several-table form runs with the largest table set (4 constellations x rotation on/off:
680 entries, bases up to 676) at every transform size, the 2-CTA 32K split included.  A 16-PLP chain of the frame's own
parameters runs all its PLPs as one FEC group (one LDPC and one mapper launch), with in-band type B signalling and
high-efficiency input mode, so a PLP's frames start at a packet phase that depends on its FEC block count.

The checker is tests/plp_oracle.py through the helpers of tests/test_plp_modcod.py (and tests/miso_oracle.py for MISO
group 2); the drop-in mapper is compared with oracle/t2oracle.py over every mode as well."""
import numpy as np
import pytest

import dvbt2ll_b200 as T
from dvbt2ll_b200 import configs as K
from common import cells_equal, max_err_over_rms, mer_db
import test_miso as MI
import test_plp_modcod as PM

S, N = K.FECFRAME_SHORT, K.FECFRAME_NORMAL
RATES = {N: (K.C1_2, K.C3_5, K.C2_3, K.C3_4, K.C4_5, K.C5_6),
         S: (K.C1_3, K.C2_5, K.C1_2, K.C3_5, K.C2_3, K.C3_4, K.C4_5, K.C5_6)}
RATE_NAMES = {K.C1_2: "1_2", K.C3_5: "3_5", K.C2_3: "2_3", K.C3_4: "3_4", K.C4_5: "4_5", K.C5_6: "5_6", K.C1_3: "1_3",
              K.C2_5: "2_5"}
CODES = [(fs, r) for fs in (N, S) for r in RATES[fs]]
MODES = [(fs, r, con, rot) for fs, r in CODES for con in range(4) for rot in (0, 1)]
NCH, NFR = 2, 2


def frame(fft, gi, pp, carriers, numdatasyms, **kw):
    """The c1 base with one TI block per frame, QPSK L1-post (room for 16 PLPs' signalling) and the given OFDM."""
    return K.resolve(dict(K.CONFIGS["c1"], fftsize=fft, guardinterval=gi, pilotpattern=pp, carriermode=carriers,
                          numdatasyms=numdatasyms, tiblocks=1, l1constellation=K.L1_MOD_QPSK, **kw))


def mode_plps(*codes):
    """One FEC block of each code x (constellation, rotation): 16 PLPs for two codes."""
    return [dict(fecblocks=1, framesize=fs, rate=r, constellation=con, rotation=rot)
            for fs, r in codes for con in range(4) for rot in (0, 1)]


# the fewest data symbols the frame holds the 16 PLPs in
MODE_CHAINS = {
    "1k": frame(K.FFTSIZE_1K, K.GI_1_16, K.PILOT_PP4, K.CARRIERS_NORMAL, 205, plps=mode_plps((N, K.C1_2), (S, K.C1_2))),
    "2k": frame(K.FFTSIZE_2K, K.GI_1_8, K.PILOT_PP2, K.CARRIERS_NORMAL, 108, plps=mode_plps((N, K.C3_5), (S, K.C3_5))),
    "4k": frame(K.FFTSIZE_4K, K.GI_1_32, K.PILOT_PP7, K.CARRIERS_NORMAL, 50, plps=mode_plps((N, K.C2_3), (S, K.C2_3))),
    "8k-ext": frame(K.FFTSIZE_8K, K.GI_1_16, K.PILOT_PP8, K.CARRIERS_EXTENDED, 25,
                    plps=mode_plps((N, K.C3_4), (S, K.C3_4))),
    "16k-ext": frame(K.FFTSIZE_16K, K.GI_1_128, K.PILOT_PP7, K.CARRIERS_EXTENDED, 13,
                     plps=mode_plps((N, K.C4_5), (S, K.C4_5))),
    "32k-ext": frame(K.FFTSIZE_32K, K.GI_1_128, K.PILOT_PP7, K.CARRIERS_EXTENDED, 6,
                     plps=mode_plps((N, K.C5_6), (S, K.C5_6))),
    "32k": frame(K.FFTSIZE_32K, K.GI_1_16, K.PILOT_PP4, K.CARRIERS_NORMAL, 3, plps=mode_plps((S, K.C1_3), (S, K.C2_5))),
}
# 16 PLPs of the frame's own parameters (short 4/5, 256QAM rotated) with unequal block counts: one FEC group
GROUP_BLOCKS = [1, 2, 1, 3, 1, 1, 2, 4, 1, 1, 1, 2, 1, 3, 1, 1]
GROUP16 = frame(K.FFTSIZE_4K, K.GI_1_32, K.PILOT_PP7, K.CARRIERS_NORMAL, 15, inband=1, version=K.VERSION_131,
                inputmode=K.INPUTMODE_HIEFF, plp_fecblocks=GROUP_BLOCKS, fecblocks=sum(GROUP_BLOCKS))
CHAINS = dict(MODE_CHAINS, group16=GROUP16)
# the 8K extended chain as a MISO frame, transmitter group 2
MISO_CHAIN = K.resolve(dict(MODE_CHAINS["8k-ext"], preamble=K.PREAMBLE_T2_MISO, misogroup=1))


def table_size(con):
    return 4 << (2 * con)


def lut_bases(plps):
    """First table entry of each PLP: one table per distinct (constellation, rotation), in the order of a stable sort of
    the PLPs by constellation, largest first."""
    bases, at, n = [0] * len(plps), {}, 0
    for p in sorted(range(len(plps)), key=lambda i: -plps[i]["constellation"]):
        key = (plps[p]["constellation"], plps[p]["rotation"])
        if key not in at:
            at[key] = n
            n += table_size(key[0])
        bases[p] = at[key]
    return bases


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_chains_cover_every_mode_once():
    modes = [(q["framesize"], q["rate"], q["constellation"], q["rotation"]) for c in MODE_CHAINS.values() for q in c["plps"]]
    assert len(modes) == 112 and sorted(modes) == sorted(MODES)
    assert len(set(MODES)) == 112
    # every transform size, and 32K twice (normal and extended carriers)
    ffts = sorted((c["fftsize"], c["carriermode"]) for c in MODE_CHAINS.values())
    assert ffts == sorted([(K.FFTSIZE_1K, 0), (K.FFTSIZE_2K, 0), (K.FFTSIZE_4K, 0), (K.FFTSIZE_8K, 1), (K.FFTSIZE_16K, 1),
                           (K.FFTSIZE_32K, 1), (K.FFTSIZE_32K, 0)])
    assert all(len(c["plps"]) == 16 for c in MODE_CHAINS.values())


@pytest.mark.parametrize("name", sorted(MODE_CHAINS))
def test_fewest_data_symbols(name):
    """The frames are full: one data symbol fewer and the 16 PLPs no longer fit."""
    cfg = MODE_CHAINS[name]
    T.Chain(cfg, max_frames=1)
    with pytest.raises(ValueError):
        T.Chain(dict(cfg, numdatasyms=cfg["numdatasyms"] - 1), max_frames=1)


@pytest.mark.parametrize("name", sorted(CHAINS))
def test_plan_matches_oracle(name):
    PM.check_plan_matches_oracle(name, CHAINS[name])


@pytest.mark.parametrize("name", sorted(CHAINS))
def test_l1post_fields_at_standard_offsets(name):
    """K_sig = 213 + 137 * 16 = 2405 bits; every field of PLP 15 at its offset."""
    import plp_oracle as O
    cfg = CHAINS[name]
    assert O.l1post_sig_bits(cfg) == 2405
    PM.check_l1post_fields(cfg)


@pytest.mark.parametrize("name", sorted(CHAINS))
def test_constellation_tables(name):
    """chain.luts: { tables, single-table form, copies in shared memory (0 before any run), first entry per PLP }.  Eight
    tables in the largest-first order of chain_create, bases 0 .. 676; one table for the single-group chain."""
    import plp_oracle as O
    cfg = CHAINS[name]
    ch = T.Chain(cfg, max_frames=1)
    plps = O.plp_list(cfg)
    luts = ch.plan("chain.luts", np.int32)
    assert luts.size == 3 + 16 and luts[2] == 0
    bases = [int(b) for b in luts[3:]]
    if name == "group16":
        assert luts[0] == 1 and bases == [0] * 16
        return
    assert luts[0] == 8
    assert bases == lut_bases(plps)
    assert sorted(set(bases)) == [0, 256, 512, 576, 640, 656, 672, 676]


def test_miso_plan():
    """The MISO frame: every symbol has the even cell count of the oracle's carrier map, and group 2's carrier codes
    build over the chain's eight tables."""
    import miso_oracle as MO
    ch = T.Chain(MISO_CHAIN, max_frames=1)
    assert np.array_equal(np.diff(ch.plan("ofdm.sym_data_start", np.int32)), MO.symbol_cells(MISO_CHAIN))
    ch.set_miso(1)
    assert ch.plan("chain.miso_code", np.int32).size == ch.plan("chain.code", np.int32).size
    assert int(ch.plan("chain.luts", np.int32)[0]) == 8


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CHAINS))
def test_chain_matches_oracle(name):
    """2 channels x 2 T2 frames (both L1-post variants): taps, cells through each PLP's own table, baseband and a
    channel alone against the batch (test_plp_modcod.check_chain_matches_oracle); then the LUT copies k_ofdm kept."""
    ch = PM.check_chain_matches_oracle(name, CHAINS[name], NCH, NFR)
    copies = int(ch.plan("chain.luts", np.int32)[2])
    assert copies in (1, 2, 4, 8, 16, 32), copies


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["1k", "32k-ext", "32k"])
def test_int16_sink(name):
    """k_ofdm's int16 form with eight tables: within 1 LSB of the complex64 output x 0.2 x 32767."""
    ch = T.Chain(MODE_CHAINS[name], max_frames=NCH * NFR)
    ts, _ = PM._streams(ch, NCH, NFR, seed=9)
    ref = ch.run_host(ts, NCH, NFR).copy()
    ch.set_sink(1, 0.2)
    got = ch.run_host(ts, NCH, NFR)
    want = np.clip(np.rint(ref.view(np.float32).astype(np.float64) * 0.2 * 32767.0), -32768, 32767).reshape(NCH, -1, 2)
    assert got.shape == want.shape and got.dtype == np.int16
    # the kernel folds the gain into its normalisation factor: the last bit of the product may round the other way
    assert np.abs(got.astype(np.int64) - want.astype(np.int64)).max() <= 1


@pytest.mark.gpu
def test_miso_dual_call():
    """k_ofdm's MISO forms with eight tables: group 1 of the dual call byte-equal to a TX1 chain, group 2 against
    tests/miso_oracle.py at MER >= 90 dB, and within 1 LSB of it on the int16 sink."""
    cfg = MISO_CHAIN
    _, ts, streams, want1 = MI._run(MI.tx(cfg, 0), nch=1, nfr=NFR, on=None)
    ch = T.Chain(cfg, max_frames=NFR)
    out1, out2 = ch.run_host_miso(ts, 1, NFR)
    assert np.array_equal(out1.view(np.uint32), want1.view(np.uint32))
    _, want2 = MI._checker(cfg, streams, 0, NFR)
    assert mer_db(out2[0], want2) >= 90.0
    assert max_err_over_rms(out2[0], want2) <= 1e-5
    gain = 0.2
    ch.set_sink(1, gain)
    _, out2 = ch.run_host_miso(ts, 1, NFR)
    w = np.stack([want2.real, want2.imag], axis=-1).astype(np.float64) * gain * 32767
    assert np.abs(out2[0].astype(np.int64) - np.clip(np.rint(w), -32768, 32767)).max() <= 1


@pytest.mark.gpu
def test_group16_equals_plps():
    """The single-group chain (dvbt2ll_chain_create_multiplp) and the same frame given as 16 `plps` entries
    (dvbt2ll_chain_create_plps) emit the same bytes."""
    a = T.Chain(GROUP16, max_frames=NCH * NFR)
    b = T.Chain(dict(GROUP16, plps=[dict(fecblocks=n) for n in GROUP_BLOCKS]), max_frames=NCH * NFR)
    ts, _ = PM._streams(a, NCH, NFR, seed=3)
    x = a.run_host(ts, NCH, NFR).copy()
    y = b.run_host(ts, NCH, NFR)
    assert np.array_equal(x.view(np.uint32), y.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["group16", "2k"])
def test_offset_batch_equals_tail(name):
    """Frames 1..2 fed from each PLP's own stream position plp_ts_bytes(p, 0, 1) (with the history bytes in front)
    equal the tail of a batch of frames 0..2, for two channels."""
    cfg = CHAINS[name]
    nfr = 3
    ch = T.Chain(cfg, max_frames=NCH * nfr)
    P, spf = ch.num_plp, ch.samples_per_frame
    ts, streams = PM._streams(ch, NCH, nfr, seed=11)
    full = ch.run_host(ts, NCH, nfr).copy()
    hist = ch.history_bytes(1)
    starts = [ch.plp_ts_bytes(p, 0, 1) for p in range(P)]
    assert len({s % 188 for s in starts}) > 1          # the PLPs' frames start at different packet phases
    rows = [streams[c, p][starts[p] - hist:starts[p] + ch.plp_ts_bytes(p, 1, nfr - 1)] for c in range(NCH) for p in range(P)]
    width = max(r.size for r in rows)
    rows = np.stack([np.pad(r, (0, width - r.size)) for r in rows])
    out = ch.run_host(rows, NCH, nfr - 1, first_frame=1)
    assert np.array_equal(out.view(np.uint32), full[:, spf:].view(np.uint32))


# ---------------------------------------------------------------------------------------------------------------------
# The drop-in mapper over every mode
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fs,rate", CODES, ids=["%s-%s" % ("normal" if fs else "short", RATE_NAMES[r]) for fs, r in CODES])
def test_dropin_mapper_every_mode(fs, rate):
    """interleavermod_bc (k_map / k_map_n<8|12|16> / k_map_qtr) for every constellation x rotation of the code, three
    FECFRAMEs of random bits each, against oracle/t2oracle.py's bit interleaver and mapper."""
    from oracle import t2oracle as O
    n = O.fec_params(fs, rate)["nldpc"]
    rng = np.random.default_rng(1000 + 10 * fs + rate)
    fec = rng.integers(0, 2, 3 * n, dtype=np.uint8)
    for con in range(4):
        for rot in (0, 1):
            cells, _ = T.interleavermod_bc(fs, rate, con, rot).work(fec, 3)
            want = O.interleavermod(fec.reshape(3, n), fs, rate, con, rot).reshape(-1)
            assert cells_equal(cells, want), (fs, rate, con, rot)
