"""MISO processing for transmitter group 2 (EN 302 755 9.1, modified Alamouti): dvbt2ll_chain_set_miso and the dual
calls dvbt2ll_chain_run_{host,device}_miso.

The checker is tests/miso_oracle.py: the reference-pinned oracle's frame-mapper output, paired per OFDM symbol and fed to
the oracle's group-2 pilot generator.  Group 1 is the existing output, which the rest of the suite pins to the
reference."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import dvbt2ll_b200 as T
from dvbt2ll_b200 import configs as K
from oracle import t2oracle as O
import miso_oracle as M
from common import cells_equal, max_err_over_rms, mer_db

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAX_ERR_OVER_RMS = 1e-5

LITE = dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_16K, pilotpattern=K.PILOT_PP3, guardinterval=K.GI_1_8, numdatasyms=12,
            constellation=K.MOD_QPSK, rate=K.C1_3, version=K.VERSION_131, l1constellation=K.L1_MOD_QPSK, tiblocks=2,
            fecblocks=10)


def miso(cfg, **kw):
    c = dict(cfg, preamble=K.PREAMBLE_T2_MISO)
    c.update(kw)
    return K.resolve(c)


MIX_PLPS = [dict(fecblocks=2, framesize=K.FECFRAME_SHORT, rate=K.C3_5, constellation=K.MOD_16QAM, rotation=1),
            dict(fecblocks=3, framesize=K.FECFRAME_SHORT, rate=K.C1_2, constellation=K.MOD_QPSK, rotation=0)]

# 1K (16 P2 symbols), 2K (8 P2 symbols), 4K with a frame-closing symbol, 8K with TR and inverse sinc, 16K T2-Lite,
# 32K extended carriers, a two-table create_plps chain
CASES = {
    "1k": miso(K.CONFIGS["c1"], fftsize=K.FFTSIZE_1K, pilotpattern=K.PILOT_PP4, guardinterval=K.GI_1_16, numdatasyms=40,
               constellation=K.MOD_16QAM, rate=K.C2_3, tiblocks=1, fecblocks=2),
    "2k": miso(K.CONFIGS["c1"], fftsize=K.FFTSIZE_2K, pilotpattern=K.PILOT_PP2, guardinterval=K.GI_1_8, numdatasyms=30,
               fecblocks=4),
    "4k-fc": miso(K.CONFIGS["c1"], fecblocks=6),
    "8k-tr-eq": miso(K.CONFIGS["c2"], paprmode=K.PAPR_TR, equalization=1, numdatasyms=20, fecblocks=3, tiblocks=1),
    "16k-lite": miso(LITE, preamble=K.PREAMBLE_T2_LITE_MISO),
    "32k-ext": miso(K.CONFIGS["c3"], numdatasyms=8, fecblocks=12),
    "4k-mix": miso(K.CONFIGS["c1"], numdatasyms=14, plps=MIX_PLPS),
}
# every constellation, rotated
for _con, _name in ((K.MOD_QPSK, "qpsk"), (K.MOD_16QAM, "16qam"), (K.MOD_64QAM, "64qam"), (K.MOD_256QAM, "256qam")):
    CASES["8k-" + _name] = miso(K.CONFIGS["c2"], constellation=_con, rotation=1, framesize=K.FECFRAME_SHORT, rate=K.C3_4,
                                numdatasyms=10, fecblocks=6, tiblocks=1)
PLAN_CASES = ["1k", "2k", "4k-fc", "8k-tr-eq", "16k-lite", "32k-ext", "4k-mix"]


def tx(cfg, group):
    return dict(cfg, misogroup=group)


def plan(ch, name, dtype=np.int32):
    return ch.plan(name, dtype)


def _symbols(ch, cfg):
    """Per symbol l: the carrier of each of its cells, in the order the frequency interleaver emits them."""
    pg = O.PilotGen(cfg)
    L, cps = pg.d["L"], pg.d["c_ps"]
    code = plan(ch, "ofdm.code").reshape(L, cps)
    start = plan(ch, "ofdm.sym_data_start")
    for l in range(L):
        k = np.flatnonzero(code[l] >= 0)
        order = k[np.argsort(code[l, k])]          # carrier of cell i
        assert np.array_equal(code[l, order], np.arange(start[l], start[l + 1]))
        yield l, order


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_checker_alamouti_round_trip():
    """The checker's own group-1 / group-2 baseband, Alamouti-combined, gives back the frame-mapper cells."""
    cfg = CASES["1k"]
    ch = T.Chain(cfg, max_frames=1)
    ts = K.make_ts(ch.ts_bytes(0, 2) + 1000)
    want = O.chain(cfg, ts, 2)
    y1, y2 = M.miso_samples(cfg, want["mapped"], 2)
    assert np.array_equal(y1, want["samples"])
    assert mer_db(M.alamouti_combine(cfg, y1, y2, 2), want["mapped"]) >= 90.0


@pytest.mark.parametrize("name", PLAN_CASES)
def test_group2_tables(name):
    """Group 2's carrier codes are group 1's with each symbol's consecutive cells swapped; its pilots, nulls and
    reserved carriers are a TX2 chain's; its pool holds the transformed L1 / dummy cells."""
    cfg = CASES[name]
    pg = O.PilotGen(cfg)
    L, cps = pg.d["L"], pg.d["c_ps"]
    c1, c2 = T.Chain(tx(cfg, 0), max_frames=1), T.Chain(tx(cfg, 1), max_frames=1)
    with pytest.raises(KeyError):
        plan(c2, "chain.miso_code")
    c2.set_miso(1)
    code1 = plan(c1, "chain.code").reshape(L, cps)
    code_tx2 = plan(c2, "chain.code").reshape(L, cps)
    code2 = plan(c2, "chain.miso_code").reshape(L, cps)
    pool1 = plan(c1, "chain.pool", np.complex64)
    pool2 = plan(c2, "chain.miso_pool", np.complex64)
    assert np.array_equal(plan(c1, "ofdm.code") >= 0, plan(c2, "ofdm.code") >= 0)
    assert np.array_equal(plan(c2, "chain.pool", np.complex64), pool1)
    want_pool = pool1.copy()
    seen = np.zeros(pool1.size, np.int8)
    n_pool = 0
    for l, order in _symbols(c2, cfg):
        assert order.size % 2 == 0, l
        data = np.zeros(cps, bool)
        data[order] = True
        assert np.array_equal(code2[l, ~data], code_tx2[l, ~data]), l
        src = code1[l, order.reshape(-1, 2)[:, ::-1].reshape(-1)]      # cell i takes cell i ^ 1
        assert np.array_equal(code2[l, order], src), l
        for i, v in enumerate(src):
            if v >= 0:
                continue
            p = ~v
            z = pool1[p]
            if z == 0:
                continue
            want_pool[p] = (-z.real + 1j * z.imag) if i % 2 == 0 else np.conj(z)
            seen[p] += 1
            n_pool += 1
    assert n_pool > 0 and seen.max() == 1          # L1 (and dummy) cells, each at one position
    info = plan(c1, "frame.info")
    base = pool1.size - plan(c1, "frame.pool", np.complex64).size
    l1b, l1n, l1v = base + info[7], info[8], info[9]
    for v in range(1, l1v):                          # the other L1-post variants take variant 0's transform
        post = slice(l1b, l1b + l1n)
        sel = np.arange(l1b + v * l1n, l1b + (v + 1) * l1n)
        z = pool1[sel]
        neg_re = want_pool[post].real != pool1[post].real
        neg_im = want_pool[post].imag != pool1[post].imag
        want_pool[sel] = np.where(neg_re, -z.real, z.real) + 1j * np.where(neg_im, -z.imag, z.imag)
    assert cells_equal(pool2, want_pool.astype(np.complex64))
    # group 1 of the same frame: a TX1 chain's tables
    c2.set_miso(0)
    assert np.array_equal(plan(c2, "chain.code").reshape(L, cps), code_tx2)


def test_even_cell_counts_sweep():
    """Every P2, data and frame-closing symbol of every MISO plan the library accepts has an even cell count (1K-32K,
    normal and extended carriers, PP1-PP8, TR on and off, T2 and T2-Lite MISO).  The counts come from the oracle's
    carrier map, and the library's plan agrees with them."""
    accepted = 0
    for fft in (K.FFTSIZE_1K, K.FFTSIZE_2K, K.FFTSIZE_4K, K.FFTSIZE_8K, K.FFTSIZE_16K, K.FFTSIZE_32K):
        for pp in range(8):
            for carriers in (K.CARRIERS_NORMAL, K.CARRIERS_EXTENDED):
                for papr in (K.PAPR_OFF, K.PAPR_TR):
                    for pre in (K.PREAMBLE_T2_MISO, K.PREAMBLE_T2_LITE_MISO):
                        for gi, nsym in ((K.GI_1_8, 9), (K.GI_1_16, 20)):
                            try:
                                b = T.pilotgenp1insert_cc(carriers, fft, pp, gi, nsym, papr, K.VERSION_131, pre, 1, 0,
                                                          K.BANDWIDTH_8_0_MHZ, K.VLENGTH[fft])
                            except Exception:
                                continue
                            accepted += 1
                            where = (fft, pp, carriers, papr, pre, gi, nsym)
                            cfg = K.resolve(dict(K.CONFIGS["c1"], carriermode=carriers, fftsize=fft, pilotpattern=pp,
                                                 guardinterval=gi, numdatasyms=nsym, paprmode=papr, preamble=pre,
                                                 version=K.VERSION_131, misogroup=1))
                            counts = np.array(M.symbol_cells(cfg))
                            assert np.all(counts % 2 == 0), where
                            assert np.array_equal(np.diff(b.plan("ofdm.sym_data_start", np.int32)), counts), where
    assert accepted >= 200, accepted


def test_oracle_counts_match_plan():
    for name in PLAN_CASES:
        cfg = CASES[name]
        ch = T.Chain(cfg, max_frames=1)
        assert np.array_equal(np.diff(plan(ch, "ofdm.sym_data_start")), M.symbol_cells(cfg)), name


def test_rejections():
    for pre in (K.PREAMBLE_T2_SISO, K.PREAMBLE_T2_LITE_SISO):
        cfg = K.resolve(dict(LITE if pre == K.PREAMBLE_T2_LITE_SISO else K.CONFIGS["c1"], preamble=pre))
        ch = T.Chain(cfg, max_frames=1)
        with pytest.raises(ValueError):
            ch.set_miso(1)
        with pytest.raises(ValueError):
            ch.set_miso(0)
        ts = K.make_ts(ch.ts_bytes(0, 1))
        with pytest.raises(RuntimeError):
            ch.run_host_miso(ts[None, :], 1, 1)
    # tone reservation on: refused by the dual call, allowed with set_miso
    ch = T.Chain(tx(CASES["8k-tr-eq"], 1), max_frames=1)
    ch.set_papr_tr(4, 2.0, 1.0)
    ch.set_miso(1)
    ts = K.make_ts(ch.ts_bytes(0, 1))
    with pytest.raises(RuntimeError):
        ch.run_host_miso(ts[None, :], 1, 1)
    # a NULL output
    ch = T.Chain(CASES["4k-fc"], max_frames=1)
    out = np.empty(ch.samples_per_frame, np.complex64)
    for a, b in ((out.ctypes.data, None), (None, out.ctypes.data)):
        assert T.lib().dvbt2ll_chain_run_host_miso(ch._h, ts.ctypes.data, ts.size, 1, 1, 0, a, b) < 0
        assert T.lib().dvbt2ll_chain_run_device_miso(ch._h, ts.ctypes.data, ts.size, 1, 1, 0, a, b, None) < 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
NCH, NFR = 2, 2


def _streams(ch, nch, nfr):
    """TS rows (channel * num_plp + plp) and each row's stream, for run_host."""
    P = ch.num_plp
    width = max(ch.plp_ts_bytes(p, 0, nfr) for p in range(P))
    streams = [K.make_ts(width + 4000, seed=K.TS_SEED + 17 * c + p) for c in range(nch) for p in range(P)]
    return np.stack([s[:width] for s in streams]), streams


def _checker(cfg, streams, c, nfr):
    """(group 1, group 2) checker baseband of channel c."""
    if "plps" in cfg:
        import plp_oracle
        P = len(cfg["plps"])
        mapped = plp_oracle.chain(cfg, streams[c * P:(c + 1) * P], nfr)["mapped"]
    else:
        mapped = O.chain(cfg, streams[c], nfr)["mapped"]
    return M.miso_samples(cfg, mapped, nfr)


def _run(cfg, nch=NCH, nfr=NFR, sink=None, on=True):
    ch = T.Chain(cfg, max_frames=nch * nfr)
    if sink:
        ch.set_sink(*sink)
    if on is not None:
        ch.set_miso(1 if on else 0)
    ts, streams = _streams(ch, nch, nfr)
    return ch, ts, streams, ch.run_host(ts, nch, nfr)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_group2_matches_checker(name):
    cfg = tx(CASES[name], 1)
    _, _, streams, out = _run(cfg)
    for c in range(NCH):
        _, want = _checker(cfg, streams, c, NFR)
        assert mer_db(out[c], want) >= 90.0, (name, c)
        assert max_err_over_rms(out[c], want) <= MAX_ERR_OVER_RMS, (name, c)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["4k-fc", "32k-ext", "4k-mix"])
def test_group2_int16_sink(name):
    cfg = tx(CASES[name], 1)
    gain = np.float32(0.2)
    _, _, streams, out = _run(cfg, sink=(1, float(gain)))
    for c in range(NCH):
        _, want = _checker(cfg, streams, c, NFR)
        w = np.stack([want.real, want.imag], axis=-1).astype(np.float64) * float(gain) * 32767
        ref = np.clip(np.rint(w), -32768, 32767)
        assert np.abs(out[c].astype(np.int64) - ref).max() <= 1, (name, c)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["1k", "4k-fc", "32k-ext"])
def test_set_miso_off_gives_todays_bytes(name):
    cfg = tx(CASES[name], 1)
    ch, ts, _, _ = _run(cfg, on=None)
    plain = ch.run_host(ts, NCH, NFR).copy()
    ch.set_miso(1)
    on = ch.run_host(ts, NCH, NFR).copy()
    ch.set_miso(0)
    off = ch.run_host(ts, NCH, NFR)
    assert np.array_equal(off.view(np.uint32), plain.view(np.uint32))
    assert not np.array_equal(on.view(np.uint32), plain.view(np.uint32))
    # group 1 with processing on is group 1
    c1 = T.Chain(tx(cfg, 0), max_frames=NCH * NFR)
    a = c1.run_host(ts, NCH, NFR).copy()
    c1.set_miso(1)
    assert np.array_equal(c1.run_host(ts, NCH, NFR).view(np.uint32), a.view(np.uint32))


def _bytes(x):
    return np.ascontiguousarray(x).view(np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("name,sink", [("1k", None), ("4k-fc", (1, 0.2)), ("32k-ext", None), ("4k-mix", None),
                                       ("8k-64qam", (1, 0.5))])
@pytest.mark.parametrize("group", [0, 1])
def test_dual_call(name, sink, group):
    """out1 equals a TX1 chain, out2 a TX2 chain with set_miso(1), whatever misogroup the dual chain has; host equals
    device; one batch equals the same frames split over calls (first_frame > 0, history bytes)."""
    cfg = CASES[name]
    nfr = 3
    _, ts, streams, want1 = _run(tx(cfg, 0), nch=1, nfr=nfr, sink=sink, on=None)
    _, _, _, want2 = _run(tx(cfg, 1), nch=1, nfr=nfr, sink=sink)
    ch = T.Chain(tx(cfg, group), max_frames=nfr)
    if sink:
        ch.set_sink(*sink)
    out1, out2 = ch.run_host_miso(ts, 1, nfr)
    assert np.array_equal(_bytes(out1), _bytes(want1))
    assert np.array_equal(_bytes(out2), _bytes(want2))
    # device form
    P, spf = ch.num_plp, ch.samples_per_frame
    ssz = 4 if sink and sink[0] else 8
    d_ts = T.DeviceBuffer(ts.size, data=np.ascontiguousarray(ts))
    d1, d2 = T.DeviceBuffer(nfr * spf * ssz), T.DeviceBuffer(nfr * spf * ssz)
    ch.run_device_miso(d_ts.ptr, ts.shape[1], 1, nfr, 0, d1.ptr, d2.ptr, None)
    T.device_synchronize()
    assert np.array_equal(d1.to_host(np.uint8), _bytes(want1).reshape(-1))
    assert np.array_equal(d2.to_host(np.uint8), _bytes(want2).reshape(-1))
    # frame by frame, with the stream history in front
    for f in range(nfr):
        hist = ch.history_bytes(f)
        rows = []
        for p in range(P):
            start = ch.plp_ts_bytes(p, 0, f)
            rows.append(streams[p][start - hist: start + ch.plp_ts_bytes(p, f, 1)])
        n = max(r.size for r in rows)
        rows = np.stack([np.pad(r, (0, n - r.size)) for r in rows])
        a, b = ch.run_host_miso(rows, 1, 1, first_frame=f)
        per = _bytes(want1).size // nfr
        assert np.array_equal(_bytes(a).reshape(-1), _bytes(want1).reshape(-1)[f * per:(f + 1) * per]), f
        assert np.array_equal(_bytes(b).reshape(-1), _bytes(want2).reshape(-1)[f * per:(f + 1) * per]), f


@pytest.mark.gpu
def test_dual_call_many_channels():
    """Several channels: run_host's channel groups on two streams, two copies back per group."""
    cfg = CASES["2k"]
    nch = 16
    _, ts, _, want1 = _run(tx(cfg, 0), nch=nch, nfr=1, on=None)
    _, _, _, want2 = _run(tx(cfg, 1), nch=nch, nfr=1)
    ch = T.Chain(tx(cfg, 0), max_frames=nch)
    out1, out2 = ch.run_host_miso(ts, nch, 1)
    assert np.array_equal(out1.view(np.uint32), want1.view(np.uint32))
    assert np.array_equal(out2.view(np.uint32), want2.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["1k", "32k-ext"])
def test_alamouti_receiver_recovers_group1(name):
    """A receiver combining the GPU's two outputs over random flat channels recovers group 1's own data cells."""
    cfg = CASES[name]
    ch = T.Chain(cfg, max_frames=NFR)
    ts, _ = _streams(ch, 1, NFR)
    out1, out2 = ch.run_host_miso(ts, 1, NFR)
    cells = np.concatenate([np.concatenate(s) for s in M.data_carriers(cfg, out1[0], NFR)])
    got = M.alamouti_combine(cfg, out1[0], out2[0], NFR, seed=3)
    assert mer_db(got, cells) >= 90.0


@pytest.mark.gpu
def test_file_modulator_miso_both():
    """t2_file_modulator --miso both --out2 writes the dual call's two outputs."""
    app = os.path.join(ROOT, "gr-dvbt2ll_b200", "t2_file_modulator")
    cfg = miso(K.CONFIGS["c2"])
    nfr = 2
    ch = T.Chain(cfg, max_frames=nfr)
    # whole packets covering both frames: the app completes a trailing partial packet with null packets
    ts = K.make_ts(-(-ch.ts_bytes(0, nfr) // 188) * 188)
    want1, want2 = ch.run_host_miso(ts[None, :], 1, nfr)
    with tempfile.TemporaryDirectory() as d:
        tsf, o1, o2 = os.path.join(d, "in.ts"), os.path.join(d, "tx1.cf32"), os.path.join(d, "tx2.cf32")
        ts.tofile(tsf)
        subprocess.check_call([app, "--config", "c2", "--miso", "both", "--frames", str(nfr), "--batch", "2",
                               "--out", o1, "--out2", o2, tsf])
        got1, got2 = np.fromfile(o1, np.complex64), np.fromfile(o2, np.complex64)
        subprocess.check_call([app, "--config", "c2", "--miso", "2", "--frames", str(nfr), "--batch", "2", "--out", o2, tsf])
        got2s = np.fromfile(o2, np.complex64)
    assert np.array_equal(got1.view(np.uint32), want1.reshape(-1).view(np.uint32))
    assert np.array_equal(got2.view(np.uint32), want2.reshape(-1).view(np.uint32))
    assert np.array_equal(got2s.view(np.uint32), want2.reshape(-1).view(np.uint32))
