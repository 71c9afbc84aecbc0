"""Several PLPs per T2 frame (SURVEY 8(f) item 4: the reference is single-PLP, lib/framemapperfint_cc_impl.cc:152).

The checker for num_plp > 1 is the numpy restatement (oracle/t2oracle.py: per-PLP L1-post entries, K_sig = 213 + 137 P,
per-PLP cell / time interleaving, PLPs laid one after the other), which for one PLP is pinned bit-exactly to the
unmodified reference (tests/test_oracle.py); the plan compiler and the CUDA chain must agree with it bit for bit /
within the baseband tolerance, and the one-PLP form of the new entry point must equal the old one."""
import numpy as np
import pytest

import dvbt2ll_b200 as T
from dvbt2ll_b200 import configs as K
from common import cells_equal, bits_equal, mer_db, max_err_over_rms
import plan_emu as E

CASES = {
    "c1-2plp": dict(K.CONFIGS["c1"], plp_fecblocks=[3, 5], fecblocks=8),
    "c1-3plp-inband": dict(K.CONFIGS["c1"], plp_fecblocks=[2, 1, 4], fecblocks=7, inband=1, version=2, l1constellation=2, tiblocks=1),
    "2k-zigzag-2plp": dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_2K, pilotpattern=K.PILOT_PP2, guardinterval=K.GI_1_8, numdatasyms=30,
                           constellation=K.MOD_64QAM, rate=K.C3_5, l1constellation=1, plp_fecblocks=[9, 4], fecblocks=13),
    "c3-3plp": dict(K.CONFIGS["c3"], plp_fecblocks=[120, 50, 31], fecblocks=201),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_plan_matches_oracle(name):
    from oracle import t2oracle as O
    cfg = K.resolve(CASES[name])
    ch = T.Chain(cfg, max_frames=1)
    P = len(cfg["plp_fecblocks"])
    plp = ch.plan("frame.plp", np.int32)
    assert int(plp[0]) == P and int(plp[1]) == 213 + 137 * P == O.l1post_sig_bits(cfg)
    assert list(plp[2:3 + P]) == list(np.concatenate([[0], np.cumsum(cfg["plp_fecblocks"])]))
    ofm = O.FrameMapper(cfg)
    info = ch.plan("frame.info", np.int32)
    assert int(info[4]) == ofm.n_post and int(info[5]) == ofm.n_punc and int(info[6]) == ofm.dummy
    # L1-pre (carries L1_POST_SIZE and L1_POST_INFO_SIZE) and both L1-post variants, cell for cell
    pool = ch.plan("frame.pool", np.complex64)
    assert cells_equal(pool[:1840], ofm.l1pre)
    n = ofm.n_post // ofm.eta
    for v in range(cfg["t2frames"]):
        assert cells_equal(pool[1840 + v * n:1840 + (v + 1) * n], O.l1post_cells(cfg, v, ofm.n_post, ofm.n_punc)), v
    # the whole frame: per-PLP cell + time interleaving, assembly, zig-zag, frequency interleaver
    rng = np.random.default_rng(4)
    for fr in range(2):
        x = (rng.standard_normal(ofm.stream_items) + 1j * rng.standard_normal(ofm.stream_items)).astype(np.complex64)
        assert cells_equal(E.frame_emu(ch, x, fr), ofm.work(x)), (name, fr)
    # TS consumption per PLP: in-band signalling cycles follow the PLP's own FEC blocks (the oracle's BB framing is a
    # pure-Python loop: short FECFRAMEs only)
    for p, nb in enumerate(cfg["plp_fecblocks"] if not cfg["framesize"] else []):
        ob = O.BbHeaderBch(cfg["framesize"], cfg["rate"], cfg["inputmode"], cfg["inband"], nb, cfg["tsrate"])
        ts = K.make_ts(3 * nb * 2000, seed=p)
        used = 0
        for fr in range(3):
            _, u = ob.work(ts[used:], nb)
            used += u
            assert ch.plp_ts_bytes(p, 0, fr + 1) == used


def test_one_plp_through_the_multiplp_entry_is_the_reference_case():
    cfg = K.resolve("c1")
    a = T.Chain(cfg, max_frames=1)
    import ctypes as C
    p = T.ChainParams(**{n: int(cfg[n]) for n, _ in T.ChainParams._fields_})
    arr = (C.c_int * 1)(cfg["fecblocks"])
    h = T.lib().dvbt2ll_chain_create_multiplp(C.byref(p), 1, arr, 1, -1)
    assert h
    try:
        for name, dt in (("frame.code", np.int32), ("frame.pool", np.complex64), ("chain.code", np.int32)):
            n = T.lib().dvbt2ll_plan_get(h, name.encode(), None, 0)
            buf = np.empty(n, np.uint8)
            T.lib().dvbt2ll_plan_get(h, name.encode(), buf.ctypes.data, n)
            assert np.array_equal(buf, a.plan(name, np.uint8)), name
    finally:
        T.lib().dvbt2ll_destroy(h)
    with pytest.raises(ValueError):
        T.Chain(dict(cfg, plp_fecblocks=[3, 0, 5], fecblocks=8), max_frames=1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_chain_multiplp_matches_oracle(name):
    """The CUDA chain with one transport stream per PLP (TS rows = channel * num_plp + plp, two channels) against the
    numpy restatement: BCH codewords bit-exact, baseband MER >= 90 dB."""
    from oracle import t2oracle as O
    cfg = K.resolve(CASES[name])
    P = len(cfg["plp_fecblocks"])
    nch, nfr = (2, 2) if not cfg["framesize"] else (1, 1)      # the oracle's BB framing is a pure-Python loop
    ch = T.Chain(cfg, max_frames=nch * nfr)
    assert ch.num_plp == P
    width = max(ch.plp_ts_bytes(p, 0, nfr) for p in range(P))
    ts = np.zeros((nch * P, width), np.uint8)
    streams = {}
    for c in range(nch):
        for p in range(P):
            s = K.make_ts(width + 4000, seed=K.TS_SEED + 17 * c + p)
            streams[c, p] = s
            ts[c * P + p] = s[:width]
    out = ch.run_host(ts, nch, nfr).copy()
    F = cfg["fecblocks"]
    p_ = O.fec_params(cfg["framesize"], cfg["rate"])
    for c in range(nch):
        want = O.chain(cfg, [streams[c, p] for p in range(P)], nfr)
        assert [int(u) for u in want["ts_used"]] == [ch.plp_ts_bytes(p, 0, nfr) for p in range(P)]
        assert mer_db(out[c], want["samples"]) >= 90.0, (name, c)
        assert max_err_over_rms(out[c], want["samples"]) <= 1e-5
        # the BCH codewords of this channel (taps hold the last single-group run: run the channel alone)
        alone = ch.run_host(ts[c * P:(c + 1) * P], 1, nfr)[0]
        assert np.array_equal(alone.view(np.uint32), out[c].view(np.uint32))
        bch = np.unpackbits(ch.tap("bch").reshape(nfr * F, -1)[:, :p_["nbch"] // 8], axis=1)
        assert bits_equal(bch.reshape(-1), want["bch"])
        # one PLP's codewords: its blocks of every frame of the whole-frame taps
        first = np.concatenate([[0], np.cumsum(cfg["plp_fecblocks"])])
        for stage in ("bch", "fec"):
            whole = ch.tap(stage).reshape(nfr, F, -1)
            for p in range(P):
                want_p = whole[:, first[p]:first[p + 1]].reshape(-1)
                assert np.array_equal(ch.tap("%s.%d" % (stage, p)), want_p), (name, c, stage, p)
