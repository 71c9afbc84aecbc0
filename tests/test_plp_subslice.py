"""PLP types, groups and sub-slicing (dvbt2ll_chain_create_plp_layout, Chain(cfg) with "type" / "group" in cfg["plps"]
and cfg["subslices"]).

The checker is tests/plp_layout_oracle.py, tests/plp_oracle.py with common, type-1 and type-2 PLPs placed by EN 302 755
8.3.6.3 and the layout fields in L1-post.  The FEC side is the type-1 twin's: the same PLPs as type-1 PLPs go through
test_plp_modcod.check_chain_matches_oracle, and the type-2 chain's codeword and cell taps equal the twin's.  Besides, a
receiver walk that reads nothing but the decoded L1-post fields and the plan's frame collects each PLP's cells at
PLP_START + s * SUB_SLICE_INTERVAL and compares them with the same PLP's cells in the type-1 frame.  The layout only
moves cells inside the frame builder's gather, so the mapper's cells of a type-2 chain equal those of its type-1 twin.

Cases: the 16-PLP 8K and 32K extended-carrier frames of tests/test_chain_modes.py with every PLP type 2 and 135
sub-slices (L_i = 15 .. 240 cells, all eight constellation tables, the 2-CTA 32K split); a 2K frame (N_P2 = 8, zig-zag)
with a common PLP, two type-1 PLPs and two type-2 PLPs of different ModCod whose sub-slices cross the data-symbol
boundaries, in-band type B signalling and high-efficiency input; c3's frame with a common PLP ahead of the two c3-mix
PLPs as type 2 with 135 sub-slices."""
import os
import subprocess

import numpy as np
import pytest

import dvbt2ll_b200 as T
from dvbt2ll_b200 import configs as K
from common import cells_equal, max_err_over_rms, mer_db
import miso_oracle as MO
import plan_emu as E
import plp_layout_oracle as LO
import plp_oracle as PO
import test_chain_modes as CM
import test_miso as MI
import test_papr_tr as TP
import test_plp_modcod as PM

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S, N = K.FECFRAME_SHORT, K.FECFRAME_NORMAL
NCH, NFR = 2, 2
LAYOUT_KEYS = ("type", "group")


def plp(blocks, framesize, rate, constellation, rotation, **kw):
    return dict(fecblocks=blocks, framesize=framesize, rate=rate, constellation=constellation, rotation=rotation, **kw)


def typed(cfg, types, subslices, groups=None):
    """cfg with PLP_TYPE types[i] (and PLP_GROUP_ID groups[i]) for its PLPs and `subslices` sub-slices per frame."""
    groups = groups or [1] * len(types)
    return dict(cfg, plps=[dict(q, type=t, group=g) for q, t, g in zip(cfg["plps"], types, groups)], subslices=subslices)


def type1_twin(cfg):
    """The same PLPs as type-1 data PLPs of group 1 through dvbt2ll_chain_create_plps."""
    twin = dict(cfg, plps=[{k: v for k, v in q.items() if k not in LAYOUT_KEYS} for q in cfg["plps"]])
    twin.pop("subslices", None)
    return twin


C3_MIX = [plp(150, N, K.C2_3, K.MOD_256QAM, 1), plp(25, N, K.C1_2, K.MOD_16QAM, 1)]
CASES = {
    "8k-ext": typed(CM.MODE_CHAINS["8k-ext"], [2] * 16, 135),
    "32k-ext": typed(CM.MODE_CHAINS["32k-ext"], [2] * 16, 135),
    # common PLP of group 2 serving the type-1 PLP 1; type-2 sub-slices of 45 and 60 cells
    "2k-zigzag": K.resolve(dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_2K, pilotpattern=K.PILOT_PP2, guardinterval=K.GI_1_8,
                                numdatasyms=30, l1constellation=K.L1_MOD_QPSK, inband=1, version=K.VERSION_131,
                                inputmode=K.INPUTMODE_HIEFF, subslices=135,
                                plps=[plp(1, S, K.C1_2, K.MOD_QPSK, 0, type=0, group=2),
                                      plp(2, S, K.C3_5, K.MOD_64QAM, 1, type=1, group=2),
                                      plp(1, S, K.C2_3, K.MOD_16QAM, 1, type=1),
                                      plp(3, S, K.C4_5, K.MOD_256QAM, 1, type=2),
                                      plp(1, S, K.C1_2, K.MOD_QPSK, 0, type=2)])),
    # c3-mix as type 2 (D = 1,215,000 and 405,000 cells) behind a common PLP of 4050 cells
    "c3": K.resolve(dict(K.CONFIGS["c3"], subslices=135,
                         plps=[plp(1, S, K.C1_2, K.MOD_16QAM, 1, type=0)] + [dict(q, type=2) for q in C3_MIX])),
}
# the MISO frame (transmitter group 2) and the tone-reservation frame.  The 16 PLPs still fit beside the reserved
# carriers, and every symbol keeps data cells: a symbol of dummy cells only has a real spectrum, whose mirror-pair peaks
# tie exactly and leave the peak-cancellation order ambiguous between float32 and float64.
MISO_CASE = K.resolve(dict(CASES["8k-ext"], preamble=K.PREAMBLE_T2_MISO, misogroup=1))
TR_CASE = TP.tr_cfg(CASES["32k-ext"])


def _field(bits, pos, n):
    v = 0
    for b in bits[pos:pos + n]:
        v = (v << 1) | int(b)
    return v


def decode_l1post(cfg, cells, n_post, ksig):
    """The K_sig signalling bits carried by one variant's L1-post cells: hard decisions on the L1 constellation, the
    16/64QAM demux and column interleaver undone, the systematic bits in front of the punctured parity, descrambled."""
    O = PO
    l1mod = cfg["l1constellation"]
    if l1mod == 0:
        tx = (cells.real < 0).astype(np.uint8)
    else:
        eta = [1, 2, 4, 6][l1mod]
        lut = O.constellation(l1mod - 1, 0)
        words = np.abs(cells[:, None] - lut[None, :]).argmin(axis=1)
        if l1mod == 1:
            tx = np.stack([words >> 1, words & 1], axis=1).reshape(-1).astype(np.uint8)
        else:
            ncol, rows = 2 * eta, n_post // (2 * eta)
            pack = (words[0::2] << eta) | words[1::2]
            il = np.zeros((rows, ncol), np.uint8)
            mux = O.TAB["l1_mux16" if eta == 4 else "l1_mux64"]
            for e in range(ncol):
                il[:, int(mux[e])] = (pack >> (ncol - 1 - e)) & 1
            tx = il.T.reshape(-1)
    sig = tx[:ksig].copy()
    if cfg["version"] == K.VERSION_131 and cfg["l1scrambled"]:
        sig ^= O.bb_prbs(ksig)
    assert list(sig[-32:]) == list(O.crc32_bits(list(sig[:-32])))
    return sig


def l1post_fields(cfg, bits, P):
    """EN 302 755 7.2.3: SUB_SLICES_PER_FRAME at bit 0; per PLP (configurable part, 89 bits from bit 70) PLP_ID,
    PLP_TYPE +8, PLP_GROUP_ID +28; dynamic part (from 70 + 89 P + 32) FRAME_IDX, SUB_SLICE_INTERVAL +8, TYPE_2_START +30,
    then per PLP (48 bits from +71) PLP_ID, PLP_START +8, PLP_NUM_BLOCKS +30."""
    d = 70 + 89 * P + 32
    f = dict(subslices=_field(bits, 0, 15), num_plp=_field(bits, 15, 8), frame_idx=_field(bits, d, 8),
             interval=_field(bits, d + 8, 22), type2_start=_field(bits, d + 30, 22), plp_id=[], type=[], group=[],
             start=[], blocks=[])
    for i in range(P):
        c, e = 70 + 89 * i, d + 71 + 48 * i
        f["plp_id"].append(_field(bits, c, 8))
        f["type"].append(_field(bits, c + 8, 3))
        f["group"].append(_field(bits, c + 28, 8))
        assert _field(bits, e, 8) == i
        f["start"].append(_field(bits, e + 8, 22))
        f["blocks"].append(_field(bits, e + 30, 10))
    return f


def plan_l1post(ch, cfg, variant):
    """The decoded L1-post fields of one variant in the chain's frame pool."""
    fi = ch.plan("frame.info", np.int32)
    pool = ch.plan("frame.pool", np.complex64)
    base, n = int(fi[7]), int(fi[8])
    ksig = int(ch.plan("frame.plp", np.int32)[1])
    bits = decode_l1post(cfg, pool[base + variant * n:base + (variant + 1) * n], int(fi[4]), ksig)
    return l1post_fields(cfg, bits, ch.num_plp)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(CASES))
def test_plan_matches_oracle(name):
    """The plan against plp_layout_oracle: layout, frame counts, L1-pre, every L1-post variant, the frame mapping of two
    frames and each PLP's TS consumption."""
    O = LO
    cfg = CASES[name]
    ch = T.Chain(cfg, max_frames=1)
    plps = O.plp_list(cfg)
    P = len(plps)
    lay = O.layout(cfg)
    got = ch.plp_layout
    assert got["type"] == [q["type"] for q in plps] and got["group"] == [q["group"] for q in plps]
    assert got["start"] == lay["start"] and got["slice_cells"] == lay["slice"]
    assert (got["subslices"], got["subslice_interval"], got["type2_start"]) == (lay["subslices"], lay["interval"],
                                                                                 lay["type2_start"])
    cells = ch.plan("frame.plp_cells", np.int32).reshape(P, 3)
    assert list(cells[:, 0]) == [q["cell_size"] for q in plps]
    assert int(ch.plan("frame.plp", np.int32)[1]) == PO.l1post_sig_bits(cfg)
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
    # TS consumption per PLP: the layout does not change it
    twin = T.Chain(type1_twin(cfg), max_frames=1)
    for p in range(P):
        assert [ch.plp_ts_bytes(p, 0, k) for k in (1, 2, 3)] == [twin.plp_ts_bytes(p, 0, k) for k in (1, 2, 3)]
    for p, q in enumerate(plps):
        if q["fecblocks"] * (4 if q["framesize"] else 1) > 40:
            continue
        ob = PO.BbHeaderBch(q["framesize"], q["rate"], cfg["inputmode"], cfg["inband"], q["fecblocks"], cfg["tsrate"])
        ts = K.make_ts(3 * q["fecblocks"] * 8200, seed=p)
        used = 0
        for fr in range(3):
            _, u = ob.work(ts[used:], q["fecblocks"])
            used += u
            assert ch.plp_ts_bytes(p, 0, fr + 1) == used, (name, p, fr)


@pytest.mark.parametrize("name", sorted(PM.CASES))
def test_layout_oracle_equals_plp_oracle_for_type1(name):
    """Without types, groups or sub-slices plp_layout_oracle is plp_oracle: the same L1-post bits and the same frame."""
    cfg = PM.resolve(name)
    for v in range(cfg["t2frames"]):
        assert LO.l1post_sig_bits_vector(cfg, v) == PO.l1post_sig_bits_vector(cfg, v)
    a, b = LO.FrameMapper(cfg), PO.FrameMapper(cfg)
    x = (np.arange(a.stream_items) + 1j).astype(np.complex64)
    for fr in range(2):
        assert np.array_equal(a.work(x).view(np.uint64), b.work(x).view(np.uint64)), (name, fr)


@pytest.mark.parametrize("name", sorted(CASES))
def test_l1post_fields_at_standard_offsets(name):
    """Every variant of the plan's L1-post cells, decoded: the layout fields at their EN 302 755 7.2.3 offsets, and the
    whole signalling equal to the oracle's."""
    O = LO
    cfg = CASES[name]
    ch = T.Chain(cfg, max_frames=1)
    plps = O.plp_list(cfg)
    P = len(plps)
    N_ = cfg["subslices"]
    D = [q["fecblocks"] * q["cell_size"] for q in plps]
    L = [d // N_ if q["type"] == 2 else d for q, d in zip(plps, D)]
    t2 = [i for i, q in enumerate(plps) if q["type"] == 2]
    t2s = sum(D[:t2[0]])
    for v in range(cfg["t2frames"]):
        f = plan_l1post(ch, cfg, v)
        assert f["frame_idx"] == v and f["num_plp"] == P and f["plp_id"] == list(range(P))
        assert f["subslices"] == N_
        assert f["type"] == [q["type"] for q in plps]
        assert f["group"] == [q["group"] for q in plps]
        assert f["blocks"] == [q["fecblocks"] for q in plps]
        assert f["interval"] == sum(L[i] for i in t2)
        assert f["type2_start"] == t2s
        for i in range(P):
            want = sum(D[:i]) if plps[i]["type"] != 2 else t2s + sum(L[j] for j in t2 if j < i)
            assert f["start"][i] == want, (name, i)
        # the oracle's field vector carries the same bits
        fi = ch.plan("frame.info", np.int32)
        n = int(fi[8])
        bits = decode_l1post(cfg, ch.plan("frame.pool", np.complex64)[int(fi[7]) + v * n:int(fi[7]) + (v + 1) * n],
                             int(fi[4]), PO.l1post_sig_bits(cfg))
        assert list(bits) == O.l1post_sig_bits_vector(cfg, v)


def data_addresses(ch):
    """Frame positions (before the frequency interleaver) of data-cell addresses 0, 1, ...: every position that does not
    carry L1 signalling, in frame order.  The P2 symbols open with their L1-pre and L1-post cells (EN 302 755 8.3.6.2:
    spread over the N_P2 symbols when there are several)."""
    d = ch.plan("ofdm.dims", np.int32)
    fi = ch.plan("frame.info", np.int32)
    fft_index = {1024: 0, 2048: 1, 4096: 2, 8192: 3, 16384: 4, 32768: 5}[int(d[0])]
    NP = (16, 8, 4, 2, 1, 1)[fft_index]
    framed = ch.plan("frame.framed", np.int32)
    l1 = np.zeros(framed.size, bool)
    l1post = int(fi[8])
    CP = int(ch.plan("ofdm.sym_data_start", np.int32)[1])
    for n in range(NP):
        l1[n * CP:n * CP + (1840 + l1post) // NP] = True
    return np.flatnonzero(~l1)


@pytest.mark.parametrize("name", sorted(CASES))
def test_receiver_walk(name):
    """Index-coded cells through the plan's frame (frame.framed by way of frame_emu); with nothing but the decoded L1-post
    fields, each PLP's cells are collected as a receiver does -- PLP_START + s * SUB_SLICE_INTERVAL, L_i = D_i / N cells
    per sub-slice for type 2, one block for common and type-1 PLPs.  Each PLP gets exactly the cells it carries in the
    type-1 frame of the same PLPs, in order; every data cell is used once; dummy cells, then unmodulated cells, follow."""
    cfg = CASES[name]
    ch = T.Chain(cfg, max_frames=1)
    twin = T.Chain(type1_twin(cfg), max_frames=1)
    fi = ch.plan("frame.info", np.int32)
    items = int(fi[1])
    x = (np.arange(items) + 1j * 7.0).astype(np.complex64)        # data cell k of the mapper -> k + 7j
    for fr in range(2):
        f = plan_l1post(ch, cfg, fr)
        frame = {}
        for c, key in ((ch, "typed"), (twin, "type1")):
            out = E.frame_emu(c, x, fr)
            framed = np.empty_like(out)
            framed[c.plan("frame.fi_src", np.int32)] = out
            frame[key] = framed[data_addresses(c)]
        got, ref = frame["typed"], frame["type1"]
        N_, used = f["subslices"], np.zeros(got.size, int)
        cell_size = [int(n) for n in ch.plan("frame.plp_cells", np.int32).reshape(-1, 3)[:, 0]]
        ref_start = 0
        for i in range(ch.num_plp):
            D = f["blocks"][i] * cell_size[i]
            if f["type"][i] == 2:
                L = D // N_
                addr = np.concatenate([f["start"][i] + s * f["interval"] + np.arange(L) for s in range(N_)])
            else:
                addr = f["start"][i] + np.arange(D)
            used[addr] += 1
            assert np.array_equal(got[addr].view(np.uint64), ref[ref_start:ref_start + D].view(np.uint64)), (name, fr, i)
            assert np.all(got[addr].imag == 7.0)
            ref_start += D
        assert ref_start == items
        assert np.all(used[:items] == 1) and not used[items:].any()
        # dummy cells (the plan's pool) and the unmodulated cells of the frame-closing symbol behind the last data cell
        pool = ch.plan("frame.pool", np.complex64)
        dummy = int(fi[6])
        assert cells_equal(got[items:items + dummy], pool[int(fi[10]):int(fi[10]) + dummy])
        assert not np.any(got[items + dummy:])


@pytest.mark.parametrize("name", sorted(CASES))
def test_type1_layout_equals_create_plps(name):
    """Every PLP type 1 in group 1 with one sub-slice, through dvbt2ll_chain_create_plp_layout: the tables of
    dvbt2ll_chain_create_plps, byte for byte."""
    twin = type1_twin(CASES[name])
    a = T.Chain(twin, max_frames=1)
    b = T.Chain(dict(twin, plps=[dict(q, type=1, group=1) for q in twin["plps"]], subslices=1), max_frames=1)
    for nm in ("chain.code", "chain.run_desc", "chain.pool", "frame.framed", "frame.pool", "frame.plp_cells"):
        assert np.array_equal(a.plan(nm, np.uint8), b.plan(nm, np.uint8)), nm


@pytest.mark.parametrize("name", sorted(CASES))
def test_one_subslice_equals_type1_data(name):
    """Every PLP type 2 with one sub-slice: the frame of the type-1 PLPs; only the L1-post cells (PLP_TYPE) differ."""
    twin = type1_twin(CASES[name])
    a = T.Chain(twin, max_frames=1)
    b = T.Chain(typed(twin, [2] * len(twin["plps"]), 1), max_frames=1)
    assert np.array_equal(a.plan("frame.framed", np.int32), b.plan("frame.framed", np.int32))
    assert np.array_equal(a.plan("chain.code", np.int32), b.plan("chain.code", np.int32))
    fi = a.plan("frame.info", np.int32)
    l1 = slice(int(fi[7]), int(fi[7]) + int(fi[8]) * int(fi[9]))
    pa, pb = a.plan("frame.pool", np.complex64), b.plan("frame.pool", np.complex64)
    assert not np.array_equal(pa[l1], pb[l1])
    pa[l1] = pb[l1] = 0
    assert np.array_equal(pa.view(np.uint64), pb.view(np.uint64))


REFUSALS = {
    "type-outside-0-2": ([1, 3], [1, 1], 1, "PLP 1"),
    "out-of-mapping-order": ([2, 1], [1, 1], 135, "PLP 1"),
    "subslices-below-1": ([1, 2], [1, 1], 0, "sub-slices"),
    "subslices-above-32767": ([1, 2], [1, 1], 32768, "sub-slices"),
    "subslices-without-type2": ([1, 1], [1, 1], 135, "type-2"),
    "subslices-not-dividing": ([1, 2], [1, 1], 7, "PLP 1"),
    "group-outside-0-255": ([1, 2], [1, 256], 1, "PLP 1"),
    "two-common-plps-in-a-group": ([0, 0, 1], [3, 3, 3], 1, "PLP 0"),
    "common-plp-without-data-plp": ([0, 1], [4, 1], 1, "PLP 0"),
}


@pytest.mark.parametrize("name", sorted(REFUSALS))
def test_refusals(name):
    """Each invalid layout refused at create, the message naming the PLP (or the sub-slice count)."""
    types, groups, n, msg = REFUSALS[name]
    base = [plp(1, S, K.C1_2, K.MOD_QPSK, 0), plp(2, S, K.C2_3, K.MOD_16QAM, 1), plp(1, S, K.C3_5, K.MOD_64QAM, 1)]
    cfg = K.resolve(dict(K.CONFIGS["c1"], fftsize=K.FFTSIZE_2K, pilotpattern=K.PILOT_PP2, guardinterval=K.GI_1_8,
                         numdatasyms=30, l1constellation=K.L1_MOD_QPSK, plps=base[:len(types)]))
    with pytest.raises(ValueError) as e:
        T.Chain(typed(cfg, types, n, groups), max_frames=1)
    assert msg in str(e.value), str(e.value)
    # the same PLPs as type-1 PLPs of group 1 fit the frame
    T.Chain(typed(cfg, [1] * len(types), 1), max_frames=1)


@pytest.mark.parametrize("name", sorted(CASES))
def test_staging_figures(name):
    """k_ofdm's staging of each case beside its type-1 twin: bulk copies per symbol (chain.run_cnt) and bytes staged per
    symbol (chain.stage_bytes).  Every case is accepted at create."""
    cfg = CASES[name]
    ch, twin = T.Chain(cfg, max_frames=1), T.Chain(type1_twin(cfg), max_frames=1)
    fig = {}
    for key, c in (("type2", ch), ("type1", twin)):
        rc, sb = c.plan("chain.run_cnt", np.int32), c.plan("chain.stage_bytes", np.int32)
        fig[key] = (int(rc.max()), int(rc.sum()), int(sb.max()))
    print("%s: max runs / runs per frame / max staging bytes: type 2 %s, type 1 %s" % (name, fig["type2"], fig["type1"]))
    assert fig["type2"][0] >= 1


def test_layout_keys_select_the_layout_entry_point():
    """Without "type", "group" and "subslices" a cfg builds exactly as before; "subslices" needs cfg["plps"]."""
    cfg = PM.resolve("c1-mix")
    assert T.plp_layout(cfg) is None
    assert T.plp_layout(dict(cfg, subslices=1)).num_subslices == 1
    with pytest.raises(ValueError):
        T.plp_layout(dict(K.resolve("c1"), subslices=2))
    lay = T.Chain(cfg, max_frames=1).plp_layout
    assert lay["type"] == [1, 1] and lay["group"] == [1, 1] and lay["subslices"] == 1
    assert lay["subslice_interval"] == 0 and lay["type2_start"] == 0 and lay["start"] == [0, 8100]


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_chain_matches_oracle(name):
    """2 channels x 2 T2 frames (both L1-post variants).  The type-1 twin against plp_oracle
    (test_plp_modcod.check_chain_matches_oracle: bch.<p> / fec.<p> bit-exact, each PLP's cells); the type-2 chain's
    bch.<p>, fec.<p> and cells taps byte-equal to the twin's for the same streams (the stages before the frame builder do
    not see the layout); its baseband against plp_layout_oracle at MER >= 90 dB and max error / RMS <= 1e-5; a channel
    alone byte-equal to the batch."""
    cfg = CASES[name]
    twin = PM.check_chain_matches_oracle(name, type1_twin(cfg), NCH, NFR)
    ch = T.Chain(cfg, max_frames=NCH * NFR)
    P = ch.num_plp
    ts, streams = PM._streams(ch, NCH, NFR)
    out = ch.run_host(ts, NCH, NFR).copy()
    twin.run_host(ts, NCH, NFR)
    for stage in ["cells"] + ["%s.%d" % (k, p) for k in ("bch", "fec") for p in range(P)]:
        assert np.array_equal(ch.tap(stage), twin.tap(stage)), (name, stage)
    for c in range(NCH):
        want = LO.chain(cfg, [streams[c, p] for p in range(P)], NFR)
        assert [int(u) for u in want["ts_used"]] == [ch.plp_ts_bytes(p, 0, NFR) for p in range(P)]
        assert mer_db(out[c], want["samples"]) >= 90.0, (name, c)
        assert max_err_over_rms(out[c], want["samples"]) <= 1e-5, (name, c)
        alone = ch.run_host(ts[c * P:(c + 1) * P], 1, NFR)[0]
        assert np.array_equal(alone.view(np.uint32), out[c].view(np.uint32)), (name, c)
    print("%s: LUT copies %d (type-1 twin %d)" % (name, int(ch.plan("chain.luts", np.int32)[2]),
                                                  int(twin.plan("chain.luts", np.int32)[2])))


@pytest.mark.gpu
def test_int16_sink():
    ch = T.Chain(CASES["32k-ext"], max_frames=NCH * NFR)
    ts, _ = PM._streams(ch, NCH, NFR, seed=9)
    ref = ch.run_host(ts, NCH, NFR).copy()
    ch.set_sink(1, 0.2)
    got = ch.run_host(ts, NCH, NFR)
    want = np.clip(np.rint(ref.view(np.float32).astype(np.float64) * 0.2 * 32767.0), -32768, 32767).reshape(NCH, -1, 2)
    assert got.shape == want.shape and got.dtype == np.int16
    # the kernel folds the gain into its normalisation factor: the last bit of the product may round the other way
    assert np.abs(got.astype(np.int64) - want.astype(np.int64)).max() <= 1


@pytest.mark.gpu
def test_tone_reservation(monkeypatch):
    """Tone reservation on the sub-sliced 32K extended frame, checked as tests/test_papr_tr.py checks its cases."""
    monkeypatch.setitem(TP.GPU_CASES, "32k-ext-type2-tr", TR_CASE)
    TP.test_chain_papr_tr_matches_oracle("32k-ext-type2-tr")


@pytest.mark.gpu
def test_miso_dual_call():
    """The sub-sliced 8K extended frame as a MISO frame: group 1 of the dual call byte-equal to a TX1 chain, group 2
    against tests/miso_oracle.py over plp_layout_oracle's frame at MER >= 90 dB."""
    cfg = MISO_CASE
    _, ts, streams, want1 = MI._run(MI.tx(cfg, 0), nch=1, nfr=NFR, on=None)
    ch = T.Chain(cfg, max_frames=NFR)
    out1, out2 = ch.run_host_miso(ts, 1, NFR)
    assert np.array_equal(out1.view(np.uint32), want1.view(np.uint32))
    mapped = LO.chain(cfg, streams[:ch.num_plp], NFR)["mapped"]
    _, want2 = MO.miso_samples(cfg, mapped, NFR)
    assert mer_db(out2[0], want2) >= 90.0
    assert max_err_over_rms(out2[0], want2) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_launches_equal_type1_twin(name):
    """The layout changes tables only: a run makes as many kernel launches as the type-1 twin's (one BB / BCH per PLP,
    one LDPC and one mapper per FEC group, one k_ofdm)."""
    counts = []
    for cfg in (CASES[name], type1_twin(CASES[name])):
        ch = T.Chain(cfg, max_frames=1)
        width = max(ch.plp_ts_bytes(p, 0, 1) for p in range(ch.num_plp))
        ts = np.stack([K.make_ts(width, seed=K.TS_SEED + p) for p in range(ch.num_plp)])
        ch.run_host(ts, 1, 1)
        l0 = T.kernel_launches()
        ch.run_host(ts, 1, 1)
        counts.append(T.kernel_launches() - l0)
    P = len(CASES[name]["plps"])
    assert counts[0] == counts[1] == P + 2 * P + 1, counts


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [1, 2])
def test_file_modulator(tmp_path, batch):
    """t2_file_modulator --plp ... --plp-types 2,2 --subslices 135 gives exactly Chain.run_host's output, frame by frame
    and in batches."""
    exe = os.path.join(ROOT, "gr-dvbt2ll_b200", "t2_file_modulator")
    if not os.path.exists(exe):
        pytest.skip("t2_file_modulator not built")
    cfg = typed(PM.resolve("c1-mix"), [2, 2], 135, groups=[1, 3])
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
    args += ["--plp-types", "2,2", "--plp-groups", "1,3", "--subslices", "135"]
    r = subprocess.run([exe, "--config", "c1", "--batch", str(batch), "--out", out] + args + files, capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stderr + r.stdout
    got = np.fromfile(out, dtype=np.complex64)
    assert got.size == want.size
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
