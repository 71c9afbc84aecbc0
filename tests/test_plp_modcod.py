"""PLPs with their own FEC type, code rate, constellation and rotation (dvbt2ll_chain_create_plps, Chain(cfg["plps"])).

The checker is tests/plp_oracle.py: the numpy restatement of oracle/t2oracle.py (pinned to the unmodified reference by
tests/test_oracle.py) extended to per-PLP parameters -- per-PLP L1-post fields and PLP_START, per-PLP cell / time
interleaving, per-PLP BB framing, LDPC and mapper.  The codewords of every PLP are also anchored to a single-PLP chain
built from that PLP's parameters, whose codewords the existing suite pins to the reference."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import dvbt2ll_b200 as T
from dvbt2ll_b200 import configs as K
from common import bits_equal, cells_equal, max_err_over_rms, mer_db
import plan_emu as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S, N = K.FECFRAME_SHORT, K.FECFRAME_NORMAL


def plp(blocks, framesize, rate, constellation, rotation):
    return dict(fecblocks=blocks, framesize=framesize, rate=rate, constellation=constellation, rotation=rotation)


CASES = {
    # 256QAM for rooftop reception next to an unrotated QPSK PLP: c1's 16200 data cells exactly
    "c1-mix": dict(K.CONFIGS["c1"], plps=[plp(4, S, K.C4_5, K.MOD_256QAM, 1), plp(1, S, K.C1_2, K.MOD_QPSK, 0)]),
    # three constellation tables, room for the longer L1-post
    "c1-3mix": dict(K.CONFIGS["c1"], plps=[plp(1, S, K.C3_5, K.MOD_64QAM, 1), plp(2, S, K.C3_4, K.MOD_16QAM, 1),
                                           plp(2, S, K.C4_5, K.MOD_256QAM, 1)]),
    # two code rates, one 4-entry QPSK table: two parameter sets whose k_ofdm fill keeps the single-table form
    "c1-qpsk-rates": dict(K.CONFIGS["c1"], plps=[plp(1, S, K.C1_2, K.MOD_QPSK, 0), plp(1, S, K.C3_5, K.MOD_QPSK, 0)]),
    # mixed PLP_FEC_TYPE, one constellation table (the first PLP takes the cfg's parameters)
    "c1-fectype": dict(K.CONFIGS["c1"], plps=[dict(fecblocks=4), plp(1, N, K.C2_3, K.MOD_256QAM, 1)]),
    # N_P2 = 8 (zig-zag), in-band type B signalling, high-efficiency input mode
    "2k-zigzag-mix": dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_2K, pilotpattern=K.PILOT_PP2, guardinterval=K.GI_1_8,
                          numdatasyms=30, l1constellation=K.L1_MOD_QPSK, inband=1, version=K.VERSION_131,
                          inputmode=K.INPUTMODE_HIEFF,
                          plps=[plp(7, S, K.C3_5, K.MOD_64QAM, 1), plp(2, S, K.C1_2, K.MOD_QPSK, 0)]),
    # 32K extended: the split k_ofdm with two tables
    "c3-mix": dict(K.CONFIGS["c3"], plps=[plp(150, N, K.C2_3, K.MOD_256QAM, 1), plp(25, N, K.C1_2, K.MOD_16QAM, 1)]),
}

# the cases of tests/test_multiplp.py: PLPs of the frame's own parameters
MULTIPLP = {
    "c1-2plp": dict(K.CONFIGS["c1"], plp_fecblocks=[3, 5], fecblocks=8),
    "c1-3plp-inband": dict(K.CONFIGS["c1"], plp_fecblocks=[2, 1, 4], fecblocks=7, inband=1, version=2, l1constellation=2, tiblocks=1),
    "2k-zigzag-2plp": dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_2K, pilotpattern=K.PILOT_PP2, guardinterval=K.GI_1_8, numdatasyms=30,
                           constellation=K.MOD_64QAM, rate=K.C3_5, l1constellation=1, plp_fecblocks=[9, 4], fecblocks=13),
    "c3-3plp": dict(K.CONFIGS["c3"], plp_fecblocks=[120, 50, 31], fecblocks=201),
}


def resolve(name):
    return K.resolve(CASES[name])


def plan_bytes(h, name):
    n = T.lib().dvbt2ll_plan_get(h, name.encode(), None, 0)
    buf = np.empty(n, np.uint8)
    T.lib().dvbt2ll_plan_get(h, name.encode(), buf.ctypes.data, n)
    return buf


def create_plps(cfg, plps, max_frames=1):
    p = T.ChainParams(**{n: int(cfg[n]) for n, _ in T.ChainParams._fields_})
    arr = (T.PlpParams * max(len(plps), 1))(*[T.PlpParams(**q) for q in plps])
    return T.lib().dvbt2ll_chain_create_plps(C.byref(p), len(plps), arr, max_frames, -1)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: plan against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(CASES))
def test_plan_matches_oracle(name):
    check_plan_matches_oracle(name, resolve(name))


def check_plan_matches_oracle(name, cfg):
    """The chain's frame plan of cfg against plp_oracle: per-PLP cell counts, PLP_START and 16-byte aligned regions,
    frame counts, L1 pool of every frame index, frame mapping of two frames and per-PLP TS consumption."""
    import plp_oracle as O
    ch = T.Chain(cfg, max_frames=1)
    plps = O.plp_list(cfg)
    P = len(plps)
    assert ch.num_plp == P and ch.fecframes_per_frame == sum(q["fecblocks"] for q in plps)
    info = ch.plan("frame.plp", np.int32)
    assert int(info[0]) == P and int(info[1]) == O.l1post_sig_bits(cfg)
    cells = ch.plan("frame.plp_cells", np.int32).reshape(P, 3)
    starts = np.concatenate([[0], np.cumsum([q["fecblocks"] * q["cell_size"] for q in plps])])
    assert list(cells[:, 0]) == [q["cell_size"] for q in plps]
    assert list(cells[:, 1]) == list(starts[:P])
    if len({tuple(q[k] for k in T.PLP_KEYS) for q in plps}) > 1:
        assert all(int(o) % 8 == 0 for o in cells[:, 2])      # every PLP region of the chain's cells 16-byte aligned
    else:
        assert list(cells[:, 2]) == list(starts[:P])          # one FEC group: the PLPs' cells follow each other
    ofm = O.FrameMapper(cfg)
    fi = ch.plan("frame.info", np.int32)
    assert int(fi[1]) == ofm.stream_items and int(fi[4]) == ofm.n_post and int(fi[5]) == ofm.n_punc and int(fi[6]) == ofm.dummy
    pool = ch.plan("frame.pool", np.complex64)
    assert cells_equal(pool[:1840], ofm.l1pre)
    n = ofm.n_post // ofm.eta
    for v in range(cfg["t2frames"]):
        assert cells_equal(pool[1840 + v * n:1840 + (v + 1) * n], O.l1post_cells(cfg, v, ofm.n_post, ofm.n_punc)), v
    rng = np.random.default_rng(7)
    for fr in range(2):
        x = (rng.standard_normal(ofm.stream_items) + 1j * rng.standard_normal(ofm.stream_items)).astype(np.complex64)
        assert cells_equal(E.frame_emu(ch, x, fr), ofm.work(x)), (name, fr)
    # TS consumption per PLP (the oracle's BB framing is a pure-Python loop: the smaller PLPs only)
    for p, q in enumerate(plps):
        if q["fecblocks"] * (4 if q["framesize"] else 1) > 40:
            continue
        ob = O.BbHeaderBch(q["framesize"], q["rate"], cfg["inputmode"], cfg["inband"], q["fecblocks"], cfg["tsrate"])
        ts = K.make_ts(3 * q["fecblocks"] * 8200, seed=p)
        used = 0
        for fr in range(3):
            _, u = ob.work(ts[used:], q["fecblocks"])
            used += u
            assert ch.plp_ts_bytes(p, 0, fr + 1) == used, (name, p, fr)


def _field(bits, pos, n):
    v = 0
    for b in bits[pos:pos + n]:
        v = (v << 1) | int(b)
    return v


@pytest.mark.parametrize("name", sorted(CASES))
def test_l1post_fields_at_standard_offsets(name):
    check_l1post_fields(resolve(name))


def check_l1post_fields(cfg):
    """EN 302 755 7.2.3: configurable part 35 + 35 bits, then 89 bits per PLP (PLP_COD at +36, PLP_MOD +39,
    PLP_ROTATION +42, PLP_FEC_TYPE +43, PLP_NUM_BLOCKS_MAX +45), 32 bits; dynamic part 71 bits, then 48 bits per PLP
    (PLP_ID, PLP_START +8, PLP_NUM_BLOCKS +30)."""
    import plp_oracle as O
    plps = O.plp_list(cfg)
    P = len(plps)
    cod = {K.C1_2: 0, K.C3_5: 1, K.C2_3: 2, K.C3_4: 3, K.C4_5: 4, K.C5_6: 5, K.C1_3: 6, K.C2_5: 7}
    bits = O.l1post_sig_bits_vector(cfg, 1)
    assert len(bits) == 213 + 137 * P
    assert _field(bits, 15, 8) == P
    start = 0
    for i, q in enumerate(plps):
        c = 70 + 89 * i
        assert _field(bits, c, 8) == i
        assert _field(bits, c + 36, 3) == cod[q["rate"]]
        assert _field(bits, c + 39, 3) == q["constellation"]
        assert _field(bits, c + 42, 1) == q["rotation"]
        assert _field(bits, c + 43, 2) == q["framesize"]
        assert _field(bits, c + 45, 10) == q["fecblocks"]
        d = 70 + 89 * P + 32 + 71 + 48 * i
        assert _field(bits, d, 8) == i
        assert _field(bits, d + 8, 22) == start
        assert _field(bits, d + 30, 10) == q["fecblocks"]
        start += q["fecblocks"] * q["cell_size"]
    assert _field(bits, 70 + 89 * P + 32, 8) == 1          # FRAME_IDX


@pytest.mark.parametrize("name", sorted(MULTIPLP))
def test_frame_parameters_equal_multiplp(name):
    """Every PLP with the frame's own parameters: the tables of create_multiplp, byte for byte."""
    cfg = K.resolve(MULTIPLP[name])
    a = T.Chain(cfg, max_frames=1)
    b = T.Chain(dict(cfg, plps=[dict(fecblocks=n) for n in cfg["plp_fecblocks"]]), max_frames=1)
    for nm in ("frame.code", "frame.pool", "chain.code", "frame.plp"):
        assert np.array_equal(a.plan(nm, np.uint8), b.plan(nm, np.uint8)), nm
    assert [a.plp_ts_bytes(p, 0, 3) for p in range(a.num_plp)] == [b.plp_ts_bytes(p, 0, 3) for p in range(b.num_plp)]


@pytest.mark.parametrize("cfgname", ["c1", "c2", "c3", "c4"])
def test_one_plp_equals_chain_create(cfgname):
    cfg = K.resolve(cfgname)
    a = T.Chain(cfg, max_frames=1)
    h = create_plps(cfg, [dict(fecblocks=cfg["fecblocks"], **{k: cfg[k] for k in T.PLP_KEYS})])
    assert h, T.last_error()
    try:
        for nm in ("frame.code", "frame.pool", "chain.code"):
            assert np.array_equal(plan_bytes(h, nm), a.plan(nm, np.uint8)), nm
        assert T.lib().dvbt2ll_chain_plp_ts_bytes(h, 0, 0, 3) == a.ts_bytes(0, 3)
    finally:
        T.lib().dvbt2ll_destroy(h)


def test_rejections():
    cfg = K.resolve("c1")
    good = plp(1, S, K.C1_2, K.MOD_QPSK, 0)
    bad = [
        [dict(good, constellation=7)],                           # unknown constellation
        [good, dict(good, framesize=N, rate=K.C1_3)],            # 1/3 exists for short frames only
        [],                                                      # no PLP
        [dict(good, fecblocks=1)] * 17,                          # more than MAX_PLP
        [dict(good, fecblocks=0)],
        [plp(9, S, K.C4_5, K.MOD_256QAM, 1)],                    # over-full: 18225 cells in a frame of 16200
    ]
    for plps in bad:
        h = create_plps(cfg, plps)
        assert not h, plps
        assert T.last_error()
    # over-full is refused whatever the over-full policy says (there is no reference behaviour to reproduce)
    T.set_overfull_policy(True)
    try:
        assert not create_plps(cfg, [plp(9, S, K.C4_5, K.MOD_256QAM, 1)])
        assert "too many FEC blocks" in T.last_error()
    finally:
        T.set_overfull_policy(False)
    with pytest.raises(ValueError):
        T.Chain(dict(cfg, plps=[dict(fecblocks=3, rate=K.C1_3, framesize=N)]), max_frames=1)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _streams(ch, nch, nfr, seed=0):
    P = ch.num_plp
    width = max(ch.plp_ts_bytes(p, 0, nfr) for p in range(P))
    ts = np.zeros((nch * P, width), np.uint8)
    streams = {}
    for c in range(nch):
        for p in range(P):
            s = K.make_ts(width + 4000, seed=K.TS_SEED + seed + 17 * c + p)
            streams[c, p] = s
            ts[c * P + p] = s[:width]
    return ts, streams


def _codewords(ch, stage, p, n, nbits):
    return np.unpackbits(ch.tap("%s.%d" % (stage, p)).reshape(n, -1)[:, :nbits // 8], axis=1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_chain_matches_oracle(name):
    import plp_oracle as O
    cfg = resolve(name)
    nch, nfr = (1, 1) if any(q["framesize"] for q in O.plp_list(cfg)) else (2, 2)
    check_chain_matches_oracle(name, cfg, nch, nfr)


def check_chain_matches_oracle(name, cfg, nch, nfr):
    """Per-PLP BCH and FEC taps bit-exact, the cells of every PLP bit-exact after decoding and cell de-interleaving,
    baseband MER >= 90 dB, a channel run alone byte-equal to the same channel in the batch.  Returns the chain."""
    import plp_oracle as O
    plps = O.plp_list(cfg)
    P = len(plps)
    ch = T.Chain(cfg, max_frames=nch * nfr)
    ts, streams = _streams(ch, nch, nfr)
    out = ch.run_host(ts, nch, nfr).copy()
    pc = ch.plan("frame.plp_cells", np.int32).reshape(P, 3)
    luts = ch.plan("chain.luts", np.int32)
    shifts = ch.plan("frame.fec_shift", np.int32)
    first_block = np.concatenate([[0], np.cumsum([q["fecblocks"] for q in plps])])
    for c in range(nch):
        want = O.chain(cfg, [streams[c, p] for p in range(P)], nfr)
        assert [int(u) for u in want["ts_used"]] == [ch.plp_ts_bytes(p, 0, nfr) for p in range(P)]
        assert mer_db(out[c], want["samples"]) >= 90.0, (name, c)
        assert max_err_over_rms(out[c], want["samples"]) <= 1e-5
        alone = ch.run_host(ts[c * P:(c + 1) * P], 1, nfr)[0]       # the taps hold the last run
        assert np.array_equal(alone.view(np.uint32), out[c].view(np.uint32))
        cells16 = ch.tap("cells", np.uint16).reshape(nfr, -1)
        for p, q in enumerate(plps):
            f = O.fec_params(q["framesize"], q["rate"])
            Fp = q["fecblocks"]
            bch = _codewords(ch, "bch", p, nfr * Fp, f["nbch"])
            assert bits_equal(bch.reshape(-1), want["bch_plp"][p]), (name, c, p)
            fec = _codewords(ch, "fec", p, nfr * Fp, f["nldpc"])
            w = want["fec_plp"][p].reshape(nfr * Fp, f["nldpc"])
            par = w[:, f["nbch"]:].reshape(nfr * Fp, 360, f["q"]).transpose(0, 2, 1).reshape(nfr * Fp, -1)
            assert bits_equal(fec, np.concatenate([w[:, :f["nbch"]], par], axis=1)), (name, c, p)
            # cells: PLP p's region, decoded through its table, cell de-interleaved
            lut = O.constellation(q["constellation"], q["rotation"])
            perm, _ = O.cell_permutation(q["framesize"], q["constellation"], q["cell_size"])
            Nc = q["cell_size"]
            ref = O.interleavermod(w, q["framesize"], q["rate"], q["constellation"], q["rotation"]).reshape(nfr, Fp, Nc)
            for fr in range(nfr):
                region = cells16[fr, pc[p, 2]:pc[p, 2] + Fp * Nc].reshape(Fp, Nc).astype(np.int64)
                for r in range(Fp):
                    mem = region[r, (perm + shifts[first_block[p] + r]) % Nc]
                    im = lut[mem >> 8].real if luts[1] else lut[mem >> 8].imag
                    got = (lut[mem & 255].real + 1j * im).astype(np.complex64)
                    assert cells_equal(got, ref[fr, r]), (name, c, p, fr, r)
    return ch


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_codewords_equal_single_plp_chain(name):
    """PLP p's codewords equal those of a single-PLP chain of PLP p's parameters with fecblocks = F_p fed the same
    stream (in-band signalling off): that chain's codewords are pinned to the reference by the existing suite."""
    import plp_oracle as O
    cfg = dict(resolve(name), inband=0)
    plps = O.plp_list(cfg)
    P = len(plps)
    nfr = 1 if any(q["framesize"] for q in plps) else 2
    ch = T.Chain(cfg, max_frames=nfr)
    ts, streams = _streams(ch, 1, nfr, seed=5)
    ch.run_host(ts, 1, nfr)
    for p, q in enumerate(plps):
        one = T.Chain(dict(cfg, plps=None, fecblocks=q["fecblocks"], **{k: q[k] for k in T.PLP_KEYS}), max_frames=nfr)
        n1 = one.ts_bytes(0, nfr)
        assert n1 == ch.plp_ts_bytes(p, 0, nfr)
        one.run_host(streams[0, p][:n1][None, :], 1, nfr)
        f = O.fec_params(q["framesize"], q["rate"])
        n = nfr * q["fecblocks"]
        for stage, nbits in (("bch", f["nbch"]), ("fec", f["nldpc"])):
            # the codeword bytes of every row (the pitch pads rows to 16 bytes; the padding is not written)
            want = one.tap(stage).reshape(n, -1)[:, :nbits // 8]
            assert np.array_equal(ch.tap("%s.%d" % (stage, p)).reshape(n, -1)[:, :nbits // 8], want), (name, p, stage)
            assert np.array_equal(one.tap("%s.0" % stage).reshape(n, -1)[:, :nbits // 8], want)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c1-mix", "c3-mix"])
def test_int16_sink(name):
    cfg = resolve(name)
    ch = T.Chain(cfg, max_frames=1)
    ts, _ = _streams(ch, 1, 1, seed=9)
    ref = ch.run_host(ts, 1, 1).copy()
    ch.set_sink(1, 0.2)
    got = ch.run_host(ts, 1, 1)
    want = np.clip(np.rint(ref.view(np.float32).astype(np.float64) * 0.2 * 32767.0), -32768, 32767).reshape(1, -1, 2)
    assert got.shape == want.shape and got.dtype == np.int16
    # the kernel folds the gain into its normalisation factor: the last bit of the product may round the other way
    assert np.abs(got.astype(np.int64) - want.astype(np.int64)).max() <= 1


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(MULTIPLP))
def test_device_output_equals_multiplp(name):
    cfg = K.resolve(MULTIPLP[name])
    a = T.Chain(cfg, max_frames=2)
    b = T.Chain(dict(cfg, plps=[dict(fecblocks=n) for n in cfg["plp_fecblocks"]]), max_frames=2)
    nch = 1 if cfg["framesize"] else 2
    ts, _ = _streams(a, nch, 1, seed=3)
    x = a.run_host(ts, nch, 1).copy()
    y = b.run_host(ts, nch, 1)
    assert np.array_equal(x.view(np.uint32), y.view(np.uint32))


@pytest.mark.gpu
def test_file_modulator_plp(tmp_path):
    """t2_file_modulator --plp BLOCKS:FRAMESIZE:RATE:CONSTELLATION:ROTATION gives exactly Chain.run_host's output."""
    exe = os.path.join(ROOT, "gr-dvbt2ll_b200", "t2_file_modulator")
    if not os.path.exists(exe):
        pytest.skip("t2_file_modulator not built")
    cfg = resolve("c1-mix")
    ch = T.Chain(cfg, max_frames=3)
    nfr, P = 3, ch.num_plp
    width = max(ch.plp_ts_bytes(p, 0, nfr) for p in range(P))
    files, rows = [], []
    for p in range(P):
        ts = K.make_ts(ch.plp_ts_bytes(p, 0, nfr) - 188 * 3 - 40, seed=K.TS_SEED + p)
        path = str(tmp_path / ("plp%d.ts" % p))
        ts.tofile(path)
        files.append(path)
        rows.append(T.ts_fill(ts, 0, width)[0])
    want = ch.run_host(np.stack(rows), 1, nfr)[0]
    out = str(tmp_path / "out.cf32")
    args = []
    for q in cfg["plps"]:
        args += ["--plp", "%d:%d:%d:%d:%d" % (q["fecblocks"], q["framesize"], q["rate"], q["constellation"], q["rotation"])]
    r = subprocess.run([exe, "--config", "c1", "--batch", "2", "--out", out] + args + files, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr + r.stdout
    got = np.fromfile(out, dtype=np.complex64)
    assert got.size == want.size
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
