"""Tone-reservation PAPR reduction on the reserved carriers (dvbt2ll_chain_set_papr_tr, k_papr_tr).

The checker is tests/papr_oracle.py: a float64 restatement of the iteration, with the reserved carriers taken from the
reference-pinned oracle's carrier map.  The stage's input x is the same chain's output with the stage off, which the
existing suite pins to the reference."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import dvbt2ll_b200 as T
from dvbt2ll_b200 import configs as K
from oracle import t2oracle as O
import papr_oracle as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TR = K.PAPR_TR

LITE = dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_16K, pilotpattern=K.PILOT_PP3, guardinterval=K.GI_1_8, numdatasyms=12,
            constellation=K.MOD_QPSK, rate=K.C1_3, preamble=K.PREAMBLE_T2_LITE_SISO, version=K.VERSION_131,
            l1constellation=K.L1_MOD_QPSK, tiblocks=2, fecblocks=19)

# plan cases: every FFT size, normal and extended carriers, MISO group 2, T2-Lite, frame-closing symbols
PLAN_CASES = {
    "1k": dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_1K, pilotpattern=K.PILOT_PP4, guardinterval=K.GI_1_16, numdatasyms=40,
               constellation=K.MOD_16QAM, rate=K.C2_3, tiblocks=1, fecblocks=1),
    "2k": dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_2K, pilotpattern=K.PILOT_PP2, guardinterval=K.GI_1_8, numdatasyms=30,
               fecblocks=1),
    "4k-fc": dict(K.CONFIGS["c1"], fecblocks=1),
    "8k": dict(K.CONFIGS["c2"], fecblocks=1),
    "8k-ext": dict(K.CONFIGS["c2"], carriermode=K.CARRIERS_EXTENDED, pilotpattern=K.PILOT_PP8, guardinterval=K.GI_1_16,
                   numdatasyms=20, fecblocks=1),
    "8k-miso-tx2": dict(K.CONFIGS["c2"], preamble=K.PREAMBLE_T2_MISO, misogroup=1, equalization=1, fecblocks=1),
    "16k": dict(K.CONFIGS["c4"], fecblocks=1),
    "16k-ext-lite": dict(LITE, carriermode=K.CARRIERS_EXTENDED, fecblocks=1),
    "32k-ext": dict(K.CONFIGS["c3"], fecblocks=1),
    "32k-normal-fc": dict(K.CONFIGS["c3"], fftsize=K.FFTSIZE_32K_T2GI, guardinterval=K.GI_19_256, pilotpattern=K.PILOT_PP4,
                          numdatasyms=7, carriermode=K.CARRIERS_NORMAL, fecblocks=1),
}


def tr_cfg(cfg, **kw):
    return K.resolve(dict(cfg, paprmode=TR, **kw))


def tr_tables(ch, N):
    sset = ch.plan("ofdm.tr_set", np.int32)
    bins = ch.plan("ofdm.tr_bins", np.int32)
    ker = ch.plan("ofdm.tr_kernel", np.complex64).reshape(-1, N)
    return sset, bins.reshape(ker.shape[0], -1), ker


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_plan_cases_cover_frame_closing_symbols():
    assert sum(O.PilotGen(tr_cfg(c)).d["n_fc"] > 0 for c in PLAN_CASES.values()) >= 2


@pytest.mark.parametrize("name", sorted(PLAN_CASES))
def test_tables_match_oracle(name):
    cfg = tr_cfg(PLAN_CASES[name])
    pg = O.PilotGen(cfg)
    N, L = pg.d["N"], pg.d["L"]
    ch = T.Chain(cfg, max_frames=1)
    ch.set_papr_tr(4, 2.0, 1.0)
    sset, bins, ker = tr_tables(ch, N)
    assert sset.size == L and ker.shape[0] == bins.shape[0] <= pg.d["dy"] + 1
    for l in range(L):
        assert np.array_equal(bins[sset[l]], P.reserved_bins(cfg, l, pg)), l
    S = bins.shape[1]
    for s in range(ker.shape[0]):
        want = P.tr_kernel(bins[s], N)
        assert ker[s, 0] == 1.0
        assert np.abs(ker[s] - want).max() <= 2e-7
        spec = np.fft.fft(ker[s].astype(np.complex128))
        ideal = np.zeros(N, np.complex128)
        ideal[bins[s]] = N / S
        assert np.abs(spec - ideal).max() <= 1e-6 * N / S


def test_oracle_invariants():
    """Only the reserved bins change, |R_b| <= tone_max, and the stop reason agrees with the trace."""
    rng = np.random.default_rng(5)
    N, S, g = 2048, 18, 0.05
    bins = np.sort(rng.choice(N, S, replace=False))
    for it, V, A in ((10, 2.0, 10.0), (10, 2.0, 0.3), (3, 1.5, 10.0), (10, 100.0, 1.0)):
        x = (rng.standard_normal(N) + 1j * rng.standard_normal(N)) / np.sqrt(2)
        X0 = np.fft.fft(x)
        r = P.tr_reduce(x, bins, it, V, A, g)
        X1 = np.fft.fft(r["out"])
        keep = np.ones(N, bool)
        keep[bins] = False
        assert np.abs(X1[keep] - X0[keep]).max() <= 1e-9 * np.abs(X0).max()
        R = (X1[bins] - X0[bins]) / (g * N)
        assert np.allclose(R, r["R"], atol=1e-12)
        assert np.abs(R).max() <= A * (1 + 1e-12)
        peak = np.abs(r["out"]).max()
        if r["reason"] == P.STOP_CLIP:
            assert peak <= V * (1 + 1e-12)
        if r["reason"] == P.STOP_LIMIT:
            assert r["applied"] == it
        else:
            assert r["applied"] < it
        if V >= 100:
            assert r["reason"] == P.STOP_CLIP and r["applied"] == 0


def test_rejections():
    for papr in (K.PAPR_OFF, K.PAPR_ACE):
        ch = T.Chain(K.resolve(dict(K.CONFIGS["c1"], paprmode=papr)), max_frames=1)
        with pytest.raises(ValueError):
            ch.set_papr_tr(4, 2.0, 1.0)
        with pytest.raises(KeyError):
            ch.plan("ofdm.tr_set", np.int32)
    ch = T.Chain(tr_cfg(K.CONFIGS["c1"], fecblocks=7), max_frames=1)
    for it, v, a in ((-1, 2.0, 1.0), (65, 2.0, 1.0), (4, 0.0, 1.0), (4, -1.0, 1.0), (4, float("nan"), 1.0),
                     (4, float("inf"), 1.0), (4, 2.0, 0.0), (4, 2.0, float("nan")), (4, 2.0, float("inf"))):
        with pytest.raises(ValueError):
            ch.set_papr_tr(it, v, a)
    ch.set_papr_tr(64, 2.0, 1.0)
    ch.set_papr_tr(0, 2.0, 1.0)
    ch = T.Chain(K.resolve(dict(K.CONFIGS["c1"], paprmode=K.PAPR_BOTH, fecblocks=7)), max_frames=1)
    ch.set_papr_tr(1, 2.0, 1.0)


def test_papr_tr_fit_counts():
    """The reserved carriers take cells: c1, c3 and c4 fit 7, 200 and 119 FEC blocks with TR, c2 its own 19."""
    for name, blocks in (("c1", 7), ("c2", 19), ("c3", 200), ("c4", 119)):
        T.Chain(tr_cfg(K.CONFIGS[name], fecblocks=blocks), max_frames=1)
    for name in ("c1", "c3", "c4"):
        with pytest.raises(ValueError):
            T.Chain(tr_cfg(K.CONFIGS[name]), max_frames=1)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
GPU_CASES = {
    "c1-tr": tr_cfg(K.CONFIGS["c1"], fecblocks=7),
    "c2-tr": tr_cfg(K.CONFIGS["c2"]),
    "c3-tr": tr_cfg(K.CONFIGS["c3"], fecblocks=200),
    "c4-tr": tr_cfg(K.CONFIGS["c4"], fecblocks=119),
    # the existing MISO / equalisation variant with its frame filled: symbols that carry only dummy cells and pilots have a
    # real spectrum, so their peaks come in exactly tied mirror pairs, which float32 and float64 may order differently
    "c2-miso-tr-eq": tr_cfg(K.CONFIGS["c2"], preamble=K.PREAMBLE_T2_MISO, misogroup=1, equalization=1, fecblocks=19, tiblocks=5),
    "16k-lite-tr": tr_cfg(LITE),
    "c3-mix-tr": tr_cfg(K.CONFIGS["c3"], plps=[dict(fecblocks=150, framesize=K.FECFRAME_NORMAL, rate=K.C2_3,
                                                    constellation=K.MOD_256QAM, rotation=1),
                                               dict(fecblocks=25, framesize=K.FECFRAME_NORMAL, rate=K.C1_2,
                                                    constellation=K.MOD_16QAM, rotation=1)]),
}
NCH, NFR, ITER, CLIP_DB, TONE_MAX = 2, 2, 10, 7.0, 3.0


def _ts(ch, nch, nfr):
    rows = []
    for c in range(nch):
        for p in range(ch.num_plp):
            rows.append(K.make_ts(ch.ts_bytes(0, nfr) + 2000, seed=K.TS_SEED + 17 * c + p))
    n = max(r.size for r in rows)
    return np.stack([np.pad(r, (0, n - r.size)) for r in rows])


def _symbols(y, pg, nfr):
    """[frames][L][gi + N] view of one channel's samples (P1 dropped)."""
    d = pg.d
    spf = 2048 + d["L"] * (d["N"] + d["gi"])
    y = y.reshape(nfr, spf)
    return y[:, 2048:].reshape(nfr, d["L"], d["N"] + d["gi"])


def _run(cfg, vclip=None, iters=ITER, tone_max=TONE_MAX, sink=None, nch=NCH, nfr=NFR, zero_after=False):
    ch = T.Chain(cfg, max_frames=nch * nfr)
    if sink:
        ch.set_sink(*sink)
    if vclip is not None:
        ch.set_papr_tr(iters, vclip, tone_max)
        if zero_after:
            ch.set_papr_tr(0, vclip, tone_max)
    out = ch.run_host(_ts(ch, nch, nfr), nch, nfr)
    return ch, out


def _vclip(x_off, pg, db=CLIP_DB):
    sym = _symbols(x_off.reshape(-1), pg, x_off.size // (2048 + pg.d["L"] * (pg.d["N"] + pg.d["gi"])))
    rms = np.sqrt(np.mean(np.abs(sym.astype(np.complex128)) ** 2))
    return float(rms * 10 ** (db / 20))


def _kernels(ch, pg):
    sset, bins, _ = tr_tables(ch, pg.d["N"])
    return sset, bins, [P.tr_kernel(b, pg.d["N"]) for b in bins]


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GPU_CASES))
def test_chain_papr_tr_matches_oracle(name):
    cfg = GPU_CASES[name]
    pg = O.PilotGen(cfg)
    N, L, gi, g = pg.d["N"], pg.d["L"], pg.d["gi"], float(pg.norm)
    nfr = max(NFR, -(-200 // (NCH * L)))       # at least 200 symbols, so that the 1 % bound on ambiguous ones can be met
    _, x_off = _run(cfg, nfr=nfr)
    V = _vclip(x_off, pg)
    ch, y = _run(cfg, V, nfr=nfr)
    stats = ch.tap("papr", np.int16).reshape(NCH, nfr, L)
    sset, bins, kers = _kernels(ch, pg)
    n_amb = n_sym = n_iter = 0
    for c in range(NCH):
        xs, ys = _symbols(x_off[c], pg, nfr), _symbols(y[c], pg, nfr)
        # P1 untouched (in place: byte-equal)
        spf = 2048 + L * (N + gi)
        for f in range(nfr):
            assert np.array_equal(y[c][f * spf: f * spf + 2048].view(np.uint32), x_off[c][f * spf: f * spf + 2048].view(np.uint32))
        for f in range(nfr):
            for l in range(L):
                x, out = xs[f, l, gi:], ys[f, l]
                s = sset[l]
                st = int(stats[c, f, l])
                n_sym += 1
                n_iter += st & 0xFF
                # cyclic prefix bit-equal to the useful tail
                assert np.array_equal(out[:gi].view(np.uint32), out[N:].view(np.uint32))
                if st & 0xFF == 0:
                    assert np.array_equal(out.view(np.uint32), xs[f, l].view(np.uint32))
                # invariants: only the reserved bins change, and they stay within tone_max
                X0 = np.fft.fft(x.astype(np.complex128)) / (g * N)
                X1 = np.fft.fft(out[gi:].astype(np.complex128)) / (g * N)
                keep = np.ones(N, bool)
                keep[bins[s]] = False
                dpow = np.mean(np.abs(X0[keep][np.abs(X0[keep]) > 0]) ** 2)
                err = np.mean(np.abs(X1[keep] - X0[keep]) ** 2)
                assert 10 * np.log10(dpow / max(err, 1e-300)) >= 90, (c, f, l)
                assert np.abs(X1[bins[s]]).max() <= TONE_MAX * (1 + 1e-5), (c, f, l)
                r = P.tr_reduce(x, bins[s], ITER, V, TONE_MAX, g, kernel=kers[s])
                if r["ambiguous"]:
                    n_amb += 1
                    continue
                assert (st & 0xFF, st >> 8) == (r["applied"], r["reason"]), (c, f, l)
                want = r["out"]
                mer = 10 * np.log10(np.mean(np.abs(want) ** 2) / max(np.mean(np.abs(out[gi:] - want) ** 2), 1e-300))
                assert mer >= 90, (c, f, l, mer)
    print("%s: %d symbols, %d ambiguous, mean updates %.2f, vclip %.4f" % (name, n_sym, n_amb, n_iter / n_sym, V))
    assert n_amb <= 0.01 * n_sym
    assert n_iter >= n_sym       # the clip is low enough that symbols iterate


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["16k-lite-tr", "c1-tr", "c3-tr", "c4-tr"])
def test_chain_papr_tr_reduces_papr(name):
    """Over the batch, at a clip 9 dB above the RMS: the largest per-symbol PAPR and the samples above vclip decrease."""
    cfg = GPU_CASES[name]
    pg = O.PilotGen(cfg)
    N, gi = pg.d["N"], pg.d["gi"]
    _, x_off = _run(cfg)
    V = _vclip(x_off, pg, 9.0)
    _, y = _run(cfg, V, tone_max=6.0)

    def papr(z):
        s = np.abs(np.concatenate([_symbols(z[c], pg, NFR)[..., gi:] for c in range(NCH)]).reshape(-1, N)) ** 2
        return (s.max(axis=1) / s.mean(axis=1)).max(), int((s > V * V).sum())
    p0, n0 = papr(x_off)
    p1, n1 = papr(y)
    print("%s: max PAPR %.2f -> %.2f dB, samples above vclip %d -> %d" % (name, 10 * np.log10(p0), 10 * np.log10(p1), n0, n1))
    assert p1 < p0 and n1 < n0, (p0, p1, n0, n1)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c1-tr", "c3-tr"])
def test_chain_papr_tr_off_means_off(name):
    cfg = GPU_CASES[name]
    _, x_off = _run(cfg)
    _, z = _run(cfg, 1.0, zero_after=True)
    assert np.array_equal(z.view(np.uint32), x_off.view(np.uint32))
    ch = T.Chain(cfg, max_frames=1)
    ch.run_host(_ts(ch, 1, 1), 1, 1)
    with pytest.raises(RuntimeError):
        ch.tap("papr", np.int16)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c1-tr", "c3-tr", "c4-tr"])
def test_chain_papr_tr_sink(name):
    """int16 sink and gain != 1: k_ofdm at gain 1 into the scratch, then the stated conversion of the complex64 output."""
    cfg = GPU_CASES[name]
    pg = O.PilotGen(cfg)
    _, x_off = _run(cfg)
    V = _vclip(x_off, pg)
    _, y = _run(cfg, V)
    gain = np.float32(0.2)
    _, z16 = _run(cfg, V, sink=(1, float(gain)))
    v = y.view(np.float32).reshape(NCH, -1, 2)
    want = np.clip(np.rint((gain * v) * np.float32(32767)), -32768, 32767).astype(np.int16)
    assert np.array_equal(z16, want)
    _, zg = _run(cfg, V, sink=(0, 0.5))
    assert np.array_equal(zg.view(np.uint32), (np.float32(0.5) * y).view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c1-tr", "c3-tr"])
def test_chain_papr_tr_batch_invariance(name):
    cfg = GPU_CASES[name]
    pg = O.PilotGen(cfg)
    _, x_off = _run(cfg, nch=1, nfr=4)
    V = _vclip(x_off, pg)
    ch = T.Chain(cfg, max_frames=4)
    ch.set_papr_tr(ITER, V, TONE_MAX)
    ts = _ts(ch, 1, 4)[0]
    full = ch.run_host(ts[None, :], 1, 4)
    stats4 = ch.tap("papr", np.int16)
    spf = ch.samples_per_frame
    for f in range(4):
        start, hist = ch.ts_bytes(0, f), ch.history_bytes(f)
        row = ts[start - hist: start + ch.ts_bytes(f, 1)]
        one = ch.run_host(row[None, :], 1, 1, first_frame=f)
        assert np.array_equal(one.view(np.uint32), full[:, f * spf:(f + 1) * spf].view(np.uint32)), f
        assert np.array_equal(ch.tap("papr", np.int16), stats4[f * pg.d["L"]:(f + 1) * pg.d["L"]])
    d_ts = T.DeviceBuffer(ts.size, data=ts)
    d_out = T.DeviceBuffer(4 * spf * 8)
    ch.run_device(d_ts.ptr, ts.size, 1, 4, 0, d_out.ptr, None)
    T.device_synchronize()
    dev = d_out.to_host(np.complex64)
    assert np.array_equal(dev.view(np.uint32), full.reshape(-1).view(np.uint32))


@pytest.mark.gpu
def test_file_modulator_papr_tr():
    """t2_file_modulator --config c2 --papr-tr gives the Python chain's bytes for the same TS."""
    app = os.path.join(ROOT, "gr-dvbt2ll_b200", "t2_file_modulator")
    cfg = GPU_CASES["c2-tr"]
    nfr = 2
    ch = T.Chain(cfg, max_frames=nfr)
    ch.set_papr_tr(ITER, 2.5, TONE_MAX)
    # whole packets covering both frames: the app completes a trailing partial packet with null packets
    ts = K.make_ts(-(-ch.ts_bytes(0, nfr) // 188) * 188)
    want = ch.run_host(ts[None, :], 1, nfr)
    with tempfile.TemporaryDirectory() as d:
        tsf, outf = os.path.join(d, "in.ts"), os.path.join(d, "out.cf32")
        ts.tofile(tsf)
        subprocess.check_call([app, "--config", "c2", "--papr-tr", "%d:2.5:%r" % (ITER, TONE_MAX), "--frames", str(nfr),
                               "--batch", "2", "--out", outf, tsf])
        got = np.fromfile(outf, np.complex64)
    assert np.array_equal(got.view(np.uint32), want.reshape(-1).view(np.uint32))
