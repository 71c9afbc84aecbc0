"""GPU parity tests: the CUDA path, called through the C ABI (ctypes), against the compiled unmodified
reference (oracle/_ref; where it is not built, the numpy oracle behind the same API -- see the reflib fixture) and
the committed golden fixtures, on identical synthetic TS input.

Bars (BASELINE.json north_star): BBFRAME/FECFRAME bits bit-exact; cells bit-exact (the LUT reproduces the
reference's float arithmetic, so better than the 1-ulp bar); frame-mapper output bit-exact; time-domain
baseband MER >= 90 dB and max error <= 1e-5 of RMS against the oracle's double-precision IFFT.
"""
import os

import numpy as np
import pytest

import dvbt2ll_b200 as T
from dvbt2ll_b200 import configs as K
from common import bits_equal, cells_equal, mer_db, max_err_over_rms, load_golden, sha

pytestmark = pytest.mark.gpu

MER_MIN_DB = 90.0
MAX_ERR_OVER_RMS = 1e-5


def _ref_frames(reflib, cfg, ts, nframes):
    ch = reflib.Chain(cfg)
    return [ch.run_frame(ts) for _ in range(nframes)]


@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4"])
def test_blocks_match_reference(reflib, name):
    """Each drop-in block driven like the flowgraph does, two T2 frames with state carried across."""
    cfg = K.resolve(name)
    nframes = 2
    B = T.blocks_for(cfg)
    F = cfg["fecblocks"]
    n_ts = F * B["bb"].forecast(B["bb"].output_multiple)
    ts = K.make_ts(nframes * n_ts + 1000)
    refs = _ref_frames(reflib, cfg, ts, nframes)
    pos = 0
    for fr in range(nframes):
        r = refs[fr]
        bch, used = B["bb"].work(ts[pos:pos + n_ts + 400], F)
        pos += used
        assert used == r["ts_used"]
        assert bits_equal(bch, r["bch"]), "BCH codewords differ"
        fec, _ = B["ldpc"].work(bch, F)
        assert bits_equal(fec, r["fec"]), "LDPC codewords differ"
        cells, _ = B["im"].work(fec, F)
        assert cells_equal(cells, r["cells"]), "cells differ"
        mapped, _ = B["fm"].work(cells, 1)
        assert cells_equal(mapped, r["mapped"]), "frame mapper output differs"
        samples, _ = B["pg"].work(mapped, 1)
        assert samples.shape == r["samples"].shape
        assert mer_db(samples, r["samples"]) >= MER_MIN_DB
        assert max_err_over_rms(samples, r["samples"]) <= MAX_ERR_OVER_RMS
    assert B["bb"].warnings == 0


@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4"])
def test_blocks_match_golden(name):
    """Same drive, checked against the committed fixtures (generated from the reference by tools/make_golden.py)."""
    g = load_golden("chain_%s.json" % name)
    cfg = K.resolve(name)
    B = T.blocks_for(cfg)
    F = cfg["fecblocks"]
    n_ts = F * B["bb"].forecast(B["bb"].output_multiple)
    ts = K.make_ts(2 * n_ts + 1000)
    assert sha(ts[:4096]) == g["ts_head_sha256"]
    pos = 0
    for fr in range(2):
        gf = g["frames"][fr]
        bch, used = B["bb"].work(ts[pos:pos + n_ts + 400], F)
        pos += used
        assert sha(np.packbits(bch)) == gf["bch_sha256"]
        fec, _ = B["ldpc"].work(bch, F)
        assert sha(np.packbits(fec)) == gf["fec_sha256"]
        cells, _ = B["im"].work(fec, F)
        assert sha(cells) == gf["cells_sha256"]
        mapped, _ = B["fm"].work(cells, 1)
        assert sha(mapped) == gf["mapped_sha256"]
        samples, _ = B["pg"].work(mapped, 1)
        head = np.array(gf["samples_head"], dtype=np.float32).view(np.complex64)
        rms = gf["samples_rms"]
        assert np.abs(samples[:head.size] - head).max() <= MAX_ERR_OVER_RMS * rms
        assert abs(np.sqrt(np.mean(np.abs(samples.astype(np.complex128)) ** 2)) - rms) <= 1e-5 * rms


CHAIN_VARIANTS = {
    # in-band type B signalling + L1 scrambling + reserved-bias bits (v1.3.1), 16QAM L1, no time interleaver
    "c1-inband-v131": dict(K.CONFIGS["c1"], inband=1, version=2, l1scrambled=1, reservedbiasbits=1, l1constellation=2,
                           tiblocks=0, fecblocks=7),
    # MISO group 2, reserved tones, inverse-sinc equalisation, 8K
    "c2-miso-tr-eq": dict(K.CONFIGS["c2"], preamble=K.PREAMBLE_T2_MISO, misogroup=1, paprmode=2, equalization=1,
                          fecblocks=17, tiblocks=5),
    # high-efficiency input mode (sync bytes dropped, variable TS consumption per T2 frame) + in-band signalling
    "c1-hiefficiency": dict(K.CONFIGS["c1"], inputmode=1, inband=1, version=2, fecblocks=7),
    # 2K with 8 P2 symbols (zig-zag L1 mapping), QPSK L1, 64QAM data
    "2k-zigzag": dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_2K, pilotpattern=K.PILOT_PP2, guardinterval=K.GI_1_8, numdatasyms=30,
                      constellation=K.MOD_64QAM, rate=K.C3_5, fecblocks=14, l1constellation=1),
    # 1K (16 P2 symbols), BPSK L1, 16QAM rotated, one TI block
    "1k-bpsk-l1": dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_1K, pilotpattern=K.PILOT_PP4, guardinterval=K.GI_1_16, numdatasyms=40,
                       constellation=K.MOD_16QAM, rate=K.C2_3, l1constellation=K.L1_MOD_BPSK, tiblocks=1, fecblocks=9),
    # T2-Lite preamble (v1.3.1), 16K, rotated QPSK with the short 1/3 code, QPSK L1
    "16k-lite": dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_16K, pilotpattern=K.PILOT_PP3, guardinterval=K.GI_1_8, numdatasyms=12,
                     constellation=K.MOD_QPSK, rate=K.C1_3, preamble=K.PREAMBLE_T2_LITE_SISO, version=K.VERSION_131,
                     l1constellation=K.L1_MOD_QPSK, tiblocks=2, fecblocks=19),
    # 8K extended carriers, PP8, reserved tones, rotated 64QAM 3/4
    "8k-ext-pp8-tr": dict(K.CONFIGS["c2"], carriermode=K.CARRIERS_EXTENDED, pilotpattern=K.PILOT_PP8, guardinterval=K.GI_1_16,
                          numdatasyms=20, constellation=K.MOD_64QAM, rate=K.C3_4, rotation=1, paprmode=K.PAPR_TR, tiblocks=1,
                          fecblocks=13),
    # 32K with the T2-only guard interval 19/256, normal carriers, rotated 16QAM 5/6, frame-closing symbol
    "32k-t2gi": dict(K.CONFIGS["c3"], fftsize=K.FFTSIZE_32K_T2GI, guardinterval=K.GI_19_256, pilotpattern=K.PILOT_PP4,
                     numdatasyms=7, constellation=K.MOD_16QAM, rate=K.C5_6, tiblocks=1, carriermode=K.CARRIERS_NORMAL,
                     fecblocks=12),
}


@pytest.mark.parametrize("name", ["c1", "c2", "c3", "c4"] + sorted(CHAIN_VARIANTS))
def test_chain_matches_reference(reflib, name):
    """Fused device-resident chain (what bench.py times) against the reference flowgraph."""
    cfg = K.resolve(CHAIN_VARIANTS.get(name, name))
    nframes = 4 if name == "c1-hiefficiency" else 2      # frame 3 of the HEM stream consumes one byte less
    ch = T.Chain(cfg, max_frames=nframes)
    n_ts = ch.ts_bytes_per_frame
    n_all = ch.ts_bytes(0, nframes)
    ts = K.make_ts(n_all + 1000)
    refs = _ref_frames(reflib, cfg, ts, nframes)
    assert refs[0]["ts_used"] == n_ts and sum(r["ts_used"] for r in refs) == n_all
    assert reflib.Chain(cfg).fm.warnings == 0
    out = ch.run_host(ts[:n_all], 1, nframes)[0]
    S = ch.samples_per_frame
    F = cfg["fecblocks"]
    nbch = refs[0]["bch"].size // F
    nldpc = refs[0]["fec"].size // F
    bch = ch.tap("bch").reshape(nframes * F, -1)
    codes = ch.tap("cells", np.uint16)             # chain mode keeps cells as 16-bit codes, cell-interleaved
    ci_dst = ch.plan("frame.ci_dst", np.int32)
    lut = ch.plan("map.lut", np.complex64)
    single = int(ch.plan("map.im_from_re", np.int32)[0])      # 1: the high byte is w~ and Im = Re lut[w~]
    for fr in range(nframes):
        r = refs[fr]
        got = np.unpackbits(bch[fr * F:(fr + 1) * F, :nbch // 8], axis=1).reshape(-1)
        assert bits_equal(got, r["bch"])
        n = r["cells"].size
        stride = (n + 7) & ~7                          # frames are padded to a multiple of 8 cells (16 bytes)
        fc = codes[fr * stride:fr * stride + n][ci_dst]
        cells = (lut[fc & 255].real + 1j * (lut[fc >> 8].real if single else lut[fc >> 8].imag)).astype(np.complex64)
        assert cells_equal(cells, r["cells"])
        s = out[fr * S:(fr + 1) * S]
        assert mer_db(s, r["samples"]) >= MER_MIN_DB
        assert max_err_over_rms(s, r["samples"]) <= MAX_ERR_OVER_RMS


def _fuzz_configs():
    """The committed random parameter sets (tools/make_fuzz_configs.py: seed 20261018 x 16, seed 777 x 40 and the `wide`
    draw seed 4242 x 24, which adds MISO / T2-Lite preambles, MISO group, PAPR signalling modes, reserved-bias bits and
    bandwidths), or the file named by DVBT2LL_FUZZ."""
    import json
    import os
    here = os.path.join(os.path.dirname(__file__), "golden")
    paths = [os.environ["DVBT2LL_FUZZ"]] if os.environ.get("DVBT2LL_FUZZ") else [os.path.join(here, "fuzz_configs.json"),
                                                                                os.path.join(here, "fuzz_configs_r2.json"),
                                                                                os.path.join(here, "fuzz_configs_r2w.json")]
    out = []
    for p in paths:
        with open(p) as f:
            out += json.load(f)
    return out


@pytest.mark.parametrize("idx", range(int(os.environ.get("DVBT2LL_FUZZ_N", "80"))))
def test_chain_random_configs(reflib, idx):
    """80 random valid parameter sets (tools/make_fuzz_configs.py: FFT / guard interval / pilot pattern per EN 302 755,
    all constellations, rotation, both frame sizes, L1 modulations, reserved tones, in-band, both input modes, inverse
    sinc, extended carriers, v1.1.1 / v1.3.1; the last 24 also MISO / T2-Lite, PAPR modes, reserved-bias bits, bandwidths) against the reference flowgraph, two channels x three T2 frames."""
    cfg = K.resolve(_fuzz_configs()[idx])
    nch, nframes = 2, 3
    ch = T.Chain(cfg, max_frames=nch * nframes)
    n_all = ch.ts_bytes(0, nframes)
    S = ch.samples_per_frame
    ts = np.stack([K.make_ts(n_all + 400, seed=K.TS_SEED + 31 * idx + c) for c in range(nch)])
    out = ch.run_host(np.ascontiguousarray(ts[:, :n_all]), nch, nframes)
    for c in range(nch):
        refs = _ref_frames(reflib, cfg, ts[c], nframes)
        assert sum(r["ts_used"] for r in refs) == n_all
        for fr in range(nframes):
            s = out[c, fr * S:(fr + 1) * S]
            assert s.size == refs[fr]["samples"].size
            assert mer_db(s, refs[fr]["samples"]) >= MER_MIN_DB
            assert max_err_over_rms(s, refs[fr]["samples"]) <= MAX_ERR_OVER_RMS


@pytest.mark.parametrize("idx", range(0, 80, 4))
def test_blocks_random_configs(reflib, idx):
    """Every fourth of the random parameter sets through the five per-block handles (the drop-in path proper), two T2
    frames with state carried across: bits and cells bit-exact, baseband within the MER bar."""
    cfg = K.resolve(_fuzz_configs()[idx])
    nframes = 2
    B = T.blocks_for(cfg)
    F = cfg["fecblocks"]
    n_ts = B["bb"].forecast(F * B["bb"].output_multiple)
    ts = K.make_ts(nframes * n_ts + 2000, seed=K.TS_SEED + 7 * idx)
    refs = _ref_frames(reflib, cfg, ts, nframes)
    pos = 0
    for fr in range(nframes):
        r = refs[fr]
        bch, used = B["bb"].work(ts[pos:pos + n_ts + 600], F)
        pos += used
        assert used == r["ts_used"]
        assert bits_equal(bch, r["bch"]), "BCH codewords differ"
        fec, _ = B["ldpc"].work(bch, F)
        assert bits_equal(fec, r["fec"]), "LDPC codewords differ"
        cells, _ = B["im"].work(fec, F)
        assert cells_equal(cells, r["cells"]), "cells differ"
        mapped, _ = B["fm"].work(cells, 1)
        assert cells_equal(mapped, r["mapped"]), "frame mapper output differs"
        samples, _ = B["pg"].work(mapped, 1)
        assert mer_db(samples, r["samples"]) >= MER_MIN_DB
        assert max_err_over_rms(samples, r["samples"]) <= MAX_ERR_OVER_RMS


def test_chain_multichannel_and_offset(reflib):
    """c5-style batching: independent channels (seed + channel) in one launch, and a batch that starts at
    T2 frame 1 (stream history in front of the pointer) equals the tail of a batch that starts at frame 0."""
    cfg = K.resolve("c1")
    nch, nframes = 3, 3
    ch = T.Chain(cfg, max_frames=nch * nframes)
    n_ts = ch.ts_bytes_per_frame
    S = ch.samples_per_frame
    ts = np.stack([K.make_ts(nframes * n_ts, seed=K.TS_SEED + c) for c in range(nch)])
    out = ch.run_host(ts, nch, nframes)
    for c in range(nch):
        refs = _ref_frames(reflib, cfg, ts[c], nframes)
        for fr in range(nframes):
            s = out[c, fr * S:(fr + 1) * S]
            assert mer_db(s, refs[fr]["samples"]) >= MER_MIN_DB
            assert max_err_over_rms(s, refs[fr]["samples"]) <= MAX_ERR_OVER_RMS
    # offset batch: frames 1..2 of channel 0, pointer advanced by one frame (history = previous bytes)
    import ctypes as C
    sub = np.ascontiguousarray(ts[0])
    out2 = np.empty((1, 2 * S), dtype=np.complex64)
    r = T.lib().dvbt2ll_chain_run_host(ch._h, sub.ctypes.data + n_ts, sub.size, 1, 2, 1, out2.ctypes.data)
    assert r == 2, T.last_error()
    assert max_err_over_rms(out2[0], out[0, S:3 * S]) <= 1e-6


def test_chain_hiefficiency_offset_batches():
    """High-efficiency input mode: the TS bytes a T2 frame consumes depend on the stream position; batches that start
    at frames 1 and 3 (pointer advanced by dvbt2ll_chain_ts_bytes) reproduce the frames of one batch from frame 0,
    for two channels at once."""
    cfg = K.resolve(CHAIN_VARIANTS["c1-hiefficiency"])
    nch, nframes = 2, 5
    ch = T.Chain(cfg, max_frames=nch * nframes)
    S = ch.samples_per_frame
    n_all = ch.ts_bytes(0, nframes)
    assert len({ch.ts_bytes(f, 1) for f in range(nframes)}) > 1          # really position dependent
    ts = np.stack([K.make_ts(n_all, seed=K.TS_SEED + c) for c in range(nch)])
    full = ch.run_host(ts, nch, nframes)
    for first, n in ((1, 2), (3, 2), (4, 1)):
        off = ch.ts_bytes(0, first)
        sub = np.ascontiguousarray(ts[:, off:off + ch.ts_bytes(first, n)])
        out = np.empty((nch, n * S), dtype=np.complex64)
        r = T.lib().dvbt2ll_chain_run_host(ch._h, sub.ctypes.data, sub.shape[1], nch, n, first, out.ctypes.data)
        assert r == nch * n, T.last_error()
        assert np.array_equal(out, full[:, first * S:(first + n) * S])


def test_two_handles_on_two_threads():
    """Handles are independent (SURVEY 8(b) threading contract): two chains driven from two host threads at the same
    time give the same samples as when run one after the other."""
    import threading
    cfgs = [K.resolve("c1"), K.resolve(CHAIN_VARIANTS["2k-zigzag"])]
    chains = [T.Chain(c, max_frames=8) for c in cfgs]
    tss = [np.stack([K.make_ts(2 * ch.ts_bytes_per_frame, seed=K.TS_SEED + 7 * i + c) for c in range(4)]) for i, ch in enumerate(chains)]
    want = [ch.run_host(ts, 4, 2).copy() for ch, ts in zip(chains, tss)]
    got = [None, None]
    errs = []

    def work(i):
        try:
            for _ in range(5):
                got[i] = chains[i].run_host(tss[i], 4, 2).copy()
        except Exception as e:          # pragma: no cover
            errs.append(e)

    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    for i in range(2):
        assert np.array_equal(got[i], want[i])


def test_ragged_and_empty_calls():
    """noutput that is not a multiple of one frame produces floor() frames; zero output is a no-op;
    too little input is an error, not a partial frame."""
    cfg = K.resolve("c1")
    B = T.blocks_for(cfg)
    nbch = B["bb"].output_multiple
    ts = K.make_ts(3 * B["bb"].forecast(nbch) + 10)
    out = np.empty(nbch + 100, dtype=np.uint8)
    import ctypes as C
    consumed = C.c_int(0)
    L = T.lib()
    r = L.dvbt2ll_work(B["bb"]._h, ts.ctypes.data, ts.size, out.ctypes.data, nbch + 100, C.byref(consumed))
    assert r == nbch and consumed.value == B["bb"].forecast(nbch)
    r = L.dvbt2ll_work(B["bb"]._h, ts.ctypes.data, ts.size, out.ctypes.data, nbch - 1, C.byref(consumed))
    assert r == 0 and consumed.value == 0
    r = L.dvbt2ll_work(B["bb"]._h, ts.ctypes.data, 10, out.ctypes.data, nbch, C.byref(consumed))
    assert r == -3


def test_ts_sync_error_is_counted(reflib):
    """A packet whose first byte is not 0x47 only raises a warning in the reference
    (bbheaderbch_bb_impl.cc:703-705); output still follows the same rule (sync byte replaced by CRC-8)."""
    cfg = K.resolve("c1")
    bb = T.bbheaderbch_bb(cfg["framesize"], cfg["rate"], cfg["inputmode"], cfg["inband"], cfg["fecblocks"], cfg["tsrate"])
    rb = reflib.bbheaderbch(cfg["framesize"], cfg["rate"], cfg["inputmode"], cfg["inband"], cfg["fecblocks"], cfg["tsrate"])
    n = bb.forecast(bb.output_multiple)
    ts = K.make_ts(2 * n + 10)
    ts[188 * 3] = 0x00
    a, _ = bb.work(ts, 2)
    b, _ = rb.work(ts, 2)
    assert bits_equal(a, b)
    assert bb.warnings == 1 and rb.warnings == 1


@pytest.mark.parametrize("mode,inband", [(1, 0), (0, 1), (1, 1)])
def test_bbheader_hiefficiency_and_inband(reflib, mode, inband):
    """INPUTMODE_HIEFF (sync bytes dropped, CRC-8 xor MODE) and in-band type B signalling."""
    fs, rate, fecblocks, tsrate = K.FECFRAME_SHORT, K.C3_5, 3, 4000000
    bb = T.bbheaderbch_bb(fs, rate, mode, inband, fecblocks, tsrate)
    rb = reflib.bbheaderbch(fs, rate, mode, inband, fecblocks, tsrate)
    nbch = bb.output_multiple
    ts = K.make_ts(12 * (bb.forecast(nbch) + 8))
    pos_a = pos_b = 0
    for call_frames in (1, 4, 2):
        a, ua = bb.work(ts[pos_a:], call_frames)
        b, ub = rb.work(ts[pos_b:], call_frames)
        assert ua == ub
        assert bits_equal(a, b)
        pos_a += ua
        pos_b += ub


@pytest.mark.parametrize("fs,rate,con,rot", [
    (1, K.C1_2, K.MOD_QPSK, 1), (1, K.C3_5, K.MOD_16QAM, 0), (1, K.C3_4, K.MOD_64QAM, 1), (1, K.C5_6, K.MOD_256QAM, 0),
    (0, K.C1_3, K.MOD_QPSK, 0), (0, K.C2_5, K.MOD_16QAM, 1), (0, K.C1_2, K.MOD_64QAM, 0), (0, K.C5_6, K.MOD_256QAM, 1),
    (0, K.C1_3, K.MOD_256QAM, 1), (1, K.C4_5, K.MOD_16QAM, 1)])
def test_ldpc_and_mapper_modes(reflib, fs, rate, con, rot):
    """LDPC + bit interleaver/mapper over code rates, frame sizes and constellations beyond the five configs."""
    from oracle import t2oracle as O
    rng = np.random.default_rng(fs * 100 + rate * 10 + con)
    p = O.fec_params(fs, rate)
    nbch, N = p["nbch"], p["nldpc"]
    ld = T.ldpc_bb(fs, rate)
    im = T.interleavermod_bc(fs, rate, con, rot)
    rim = reflib.interleavermod(fs, rate, con, rot)
    nfr = 3
    info = rng.integers(0, 2, nfr * nbch, dtype=np.uint8)
    fec, used = ld.work(info, nfr)
    assert used == nfr * nbch
    want = O.ldpc_encode(info.reshape(nfr, nbch), fs, rate).reshape(-1)
    assert bits_equal(fec, want)
    if (fs, rate) not in reflib.REF_LDPC_BROKEN:      # the reference's dead-code encoder overruns its LUT for 3 short codes
        rbb = reflib.bbheaderbch(fs, rate, 0, 0, 1, 0)
        assert bits_equal(want, np.concatenate([rbb.ldpc(info[f * nbch:(f + 1) * nbch], N) for f in range(nfr)]))
    cells, _ = im.work(fec, nfr)
    assert cells_equal(cells, rim.work(want, nfr)[0])


def test_qpsk_mapper_every_code(reflib):
    """QPSK has three mapper paths (byte table for bits in place, transposed parity, bit by bit): every frame size /
    code rate x rotation against the reference's interleavermod, three FECFRAMEs of random bits each."""
    from oracle import t2oracle as O
    rng = np.random.default_rng(77)
    paths = set()
    for fs, rates in ((1, (K.C1_2, K.C3_5, K.C2_3, K.C3_4, K.C4_5, K.C5_6)),
                      (0, (K.C1_3, K.C2_5, K.C1_2, K.C3_5, K.C2_3, K.C3_4, K.C4_5, K.C5_6))):
        for rate in rates:
            N = O.fec_params(fs, rate)["nldpc"]
            fec = rng.integers(0, 2, 3 * N, dtype=np.uint8)
            for rot in (0, 1):
                im = T.interleavermod_bc(fs, rate, K.MOD_QPSK, rot)
                lin, par_q, _ = (int(v) for v in im.plan("map.qpsk", np.int32))
                paths.add((lin > 0, par_q > 0))
                cells, _ = im.work(fec, 3)
                assert cells_equal(cells, reflib.interleavermod(fs, rate, K.MOD_QPSK, rot).work(fec, 3)[0]), (fs, rate, rot)
    assert (True, True) in paths and (True, False) in paths      # both fast paths were exercised


def test_ldpc_parity_check_independent():
    """Known-answer independent of the reference code: every parity check of the IRA code built straight
    from the address table (check j: XOR of the info bits hitting row j, p[j] and p[j-1]) is satisfied."""
    fs, rate = 1, K.C2_3
    ld = T.ldpc_bb(fs, rate)
    rng = np.random.default_rng(7)
    nbch, N, q = 43200, 64800, 60
    info = rng.integers(0, 2, nbch, dtype=np.uint8)
    cw, _ = ld.work(info, 1)
    P = N - nbch
    row_ptr = ld.plan("ldpc.row_ptr", np.uint16).astype(int)
    ent = ld.plan("ldpc.entries", np.uint32)
    acc = np.zeros(P, dtype=np.uint8)
    for t in range(q):
        for e in range(row_ptr[t], row_ptr[t + 1]):
            g, s = int(ent[e] & 0xFFFF), int(ent[e] >> 16)
            n = np.arange(360)
            acc[q * ((n + s) % 360) + t] ^= info[360 * g + n]
    p = cw[nbch:]
    prev = np.concatenate([[0], p[:-1]]).astype(np.uint8)
    assert not np.any(acc ^ p ^ prev)


def test_fft_sizes_parseval_and_reference(reflib):
    """Every FFT size 1K..32K through block 5: against the reference, plus Parseval per symbol."""
    rng = np.random.default_rng(3)
    cases = [(K.FFTSIZE_1K, K.PILOT_PP1, K.GI_1_16, 0), (K.FFTSIZE_2K, K.PILOT_PP2, K.GI_1_8, 0),
             (K.FFTSIZE_4K, K.PILOT_PP3, K.GI_1_4, 0), (K.FFTSIZE_8K, K.PILOT_PP4, K.GI_19_128, 1),
             (K.FFTSIZE_16K, K.PILOT_PP5, K.GI_19_256, 1), (K.FFTSIZE_32K, K.PILOT_PP6, K.GI_1_32, 1),
             (K.FFTSIZE_32K, K.PILOT_PP8, K.GI_1_16, 0)]
    for fft, pp, gi, ext in cases:
        args = (ext, fft, pp, gi, 5, K.PAPR_OFF, 0, K.PREAMBLE_T2_SISO, 0, K.EQUALIZATION_ON, K.BANDWIDTH_8_0_MHZ, K.VLENGTH[fft])
        pg = T.pilotgenp1insert_cc(*args)
        rp = reflib.pilotgen(*args)
        n_in = pg.forecast(pg.output_multiple)
        assert n_in == rp.forecast(rp.output_multiple)
        x = (rng.standard_normal(2 * n_in) + 1j * rng.standard_normal(2 * n_in)).astype(np.complex64)
        y, used = pg.work(x, 2)
        want, _ = rp.work(x, 2)
        assert used == 2 * n_in
        assert mer_db(y, want) >= MER_MIN_DB, (fft, pp)
        assert max_err_over_rms(y, want) <= MAX_ERR_OVER_RMS, (fft, pp)


def test_full_size_batch_invariance():
    """BASELINE config 5 at full size (64 independent 32K / 256QAM channels in one launch), checked through
    size-independent properties: a channel's baseband does not depend on what it is batched with (bit-exact
    against single-channel runs), the result is deterministic, and every OFDM symbol satisfies Parseval
    (time-domain energy = N * normalization^2 * energy of the carriers, which for unit-power cells and the
    pilot boosts of PP7 is fixed by the frame structure -- compared channel to channel)."""
    cfg = K.resolve("c3")
    nch = 64
    ch = T.Chain(cfg, max_frames=nch)
    n_ts, S = ch.ts_bytes_per_frame, ch.samples_per_frame
    ts = np.stack([K.make_ts(n_ts, seed=K.TS_SEED + c) for c in range(nch)])
    out = ch.run_host(ts, nch, 1)
    again = ch.run_host(ts, nch, 1)
    assert np.array_equal(out.view(np.uint32), again.view(np.uint32))
    single = T.Chain(cfg, max_frames=1)
    for c in (0, 17, 63):
        alone = single.run_host(ts[c], 1, 1)[0]
        assert np.array_equal(alone.view(np.uint32), out[c].view(np.uint32)), "channel %d depends on its batch" % c
    # P1 is identical for every channel; per-symbol energies agree across channels to the statistics of 27k cells
    assert np.array_equal(out[:, :2048].view(np.uint32), np.broadcast_to(out[0, :2048], (nch, 2048)).view(np.uint32))
    N, gi, L = 32768, 256, 60
    sym = out[:, 2048:].reshape(nch, L, N + gi)
    assert np.array_equal(sym[:, :, :gi].view(np.uint32), sym[:, :, N:].view(np.uint32)), "cyclic prefix is not the symbol tail"
    e = (np.abs(sym[:, :, gi:].astype(np.complex128)) ** 2).sum(axis=2)          # [channel, symbol]
    rel = np.abs(e / e.mean(axis=0, keepdims=True) - 1.0)
    assert rel[:, 1:].max() < 0.05        # data symbols: unit-power random cells, same pilots


def test_chain_sink_gain_and_int16(reflib):
    """The flowgraph's sink side folded into the last kernel: multiply_const(0.2) and 16-bit I/Q conversion."""
    cfg = K.resolve("c4")
    ch = T.Chain(cfg, max_frames=2)
    n_ts = ch.ts_bytes_per_frame
    ts = K.make_ts(2 * n_ts)
    ref_out = ch.run_host(ts, 1, 2)[0]
    ch.set_sink(0, 0.2)
    scaled = ch.run_host(ts, 1, 2)[0]
    assert max_err_over_rms(scaled, (ref_out * np.float32(0.2)).astype(np.complex64)) <= 1e-6
    ch.set_sink(1, 0.2)
    q = ch.run_host(ts, 1, 2)[0]
    want = np.clip(np.rint(ref_out.view(np.float32).astype(np.float64) * 0.2 * 32767.0), -32768, 32767).reshape(-1, 2)
    assert q.shape == want.shape and q.dtype == np.int16
    assert np.abs(q.astype(np.int64) - want.astype(np.int64)).max() <= 1
    cfg3 = K.resolve("c3")                                   # 32K path (even/odd halves) with the int16 sink
    ch3 = T.Chain(cfg3, max_frames=1)
    ts3 = K.make_ts(ch3.ts_bytes_per_frame)
    f32 = ch3.run_host(ts3, 1, 1)[0]
    ch3.set_sink(1, 0.2)
    q3 = ch3.run_host(ts3, 1, 1)[0]
    want3 = np.clip(np.rint(f32.view(np.float32).astype(np.float64) * 0.2 * 32767.0), -32768, 32767).reshape(-1, 2)
    assert np.abs(q3.astype(np.int64) - want3.astype(np.int64)).max() <= 1


@pytest.mark.parametrize("fs,rate", [(1, r) for r in (K.C1_2, K.C3_5, K.C2_3, K.C3_4, K.C4_5, K.C5_6)] +
                         [(0, r) for r in (K.C1_3, K.C2_5, K.C1_2, K.C3_5, K.C2_3, K.C3_4, K.C4_5, K.C5_6)])
def test_bch_and_ldpc_all_codes(fs, rate):
    """All 14 T2 code configurations through BB framing + BCH + LDPC on the GPU against the oracle
    (BCH codewords divisible by g(x) and H.c = 0 are checked for the oracle itself in tests/test_oracle.py)."""
    from oracle import t2oracle as O
    p = O.fec_params(fs, rate)
    bb = T.bbheaderbch_bb(fs, rate, 0, 0, 1, 0)
    ob = O.BbHeaderBch(fs, rate, 0, 0, 1, 0)
    ld = T.ldpc_bb(fs, rate)
    nfr = 5
    ts = K.make_ts(nfr * bb.forecast(p["nbch"]) + 400, seed=fs * 100 + rate + 1)
    bch, used = bb.work(ts, nfr)
    want, used2 = ob.work(ts, nfr)
    assert used == used2 and bits_equal(bch, want)
    fec, _ = ld.work(bch, nfr)
    assert bits_equal(fec, O.ldpc_encode(want.reshape(nfr, p["nbch"]), fs, rate).reshape(-1))


def test_pilotgen_mode_sweep():
    """Block 5 over FFT sizes x pilot patterns x carrier modes x SISO/MISO x reserved tones against the oracle."""
    from oracle import t2oracle as O
    from common import pg_args
    rng = np.random.default_rng(9)
    base = dict(K.resolve("c1"))
    cases = []
    for fft, pps in ((K.FFTSIZE_1K, (0, 4)), (K.FFTSIZE_2K, (2, 6)), (K.FFTSIZE_4K, (1, 3)), (K.FFTSIZE_8K, (0, 7)),
                     (K.FFTSIZE_16K_T2GI, (5, 7)), (K.FFTSIZE_32K_T2GI, (3, 5))):
        for pp in pps:
            for ext, pre, mg, papr in ((0, 0, 0, 0), (1, 1, 1, 2), (1, 0, 0, 3)):
                cases.append(dict(base, fftsize=fft, pilotpattern=pp, carriermode=ext, preamble=pre, misogroup=mg, paprmode=papr,
                                  guardinterval=K.GI_1_16, numdatasyms=4, vlength=K.VLENGTH[fft], equalization=pp & 1))
    assert len(cases) == 36
    for cfg in cases:
        pg = T.pilotgenp1insert_cc(*pg_args(cfg))
        opg = O.PilotGen(cfg)
        n_in = pg.forecast(pg.output_multiple)
        assert n_in == opg.d["active"]
        x = (rng.standard_normal(n_in) + 1j * rng.standard_normal(n_in)).astype(np.complex64)
        y, _ = pg.work(x, 1)
        want = opg.work(x)
        assert max_err_over_rms(y, want) <= MAX_ERR_OVER_RMS, {k: cfg[k] for k in ("fftsize", "pilotpattern", "carriermode", "preamble", "paprmode")}
