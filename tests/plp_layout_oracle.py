"""TEST INFRASTRUCTURE ONLY -- tests/plp_oracle.py extended to PLP types, groups and sub-slicing (EN 302 755 8.3.6.3):
cfg["plps"] entries may name a PLP_TYPE "type" (0 common, 1 data type 1, 2 data type 2; default 1) and a PLP_GROUP_ID
"group" (default 1), and the config the SUB_SLICES_PER_FRAME "subslices" of its type-2 PLPs (default 1).

PLPs are listed common, type 1, type 2.  Common and type-1 PLPs take one block of cells each from data-cell address 0;
TYPE_2_START is their cell sum (0 without type-2 PLPs).  Type-2 PLP i with D_i cells per frame has sub-slices of
L_i = D_i / N cells, SUB_SLICE_INTERVAL = sum of L_i, and cell k of its time-interleaver output goes to
PLP_START_i + (k div L_i) SUB_SLICE_INTERVAL + k mod L_i, PLP_START_i = TYPE_2_START + sum of L_j over the type-2 PLPs
before it.  BB framing, FEC, the mapper, the cell and time interleavers and the pilot generator are tests/plp_oracle.py's
and oracle/t2oracle.py's; this module changes where the frame builder places the cells and what L1-post says."""
import numpy as np

from oracle import t2oracle as _O
from oracle.t2oracle import TAB, VERSION_131, PilotGen, bb_prbs, constellation, crc32_bits
import plp_oracle as PO

_bits, _l1_fec = _O._bits, _O._l1_fec


def plp_list(c):
    """plp_oracle.plp_list with each PLP's "type" and "group" (default 1)."""
    out = PO.plp_list(c)
    for p in out:
        p.setdefault("type", 1)
        p.setdefault("group", 1)
    return out


def layout(c):
    """The data-cell layout of the PLPs: dict of per-PLP "start" (PLP_START) and "slice" (L_i: cells per sub-slice, a
    common or type-1 PLP's cells per frame), "subslices" (N), "interval" (SUB_SLICE_INTERVAL) and "type2_start"
    (TYPE_2_START; both 0 without type-2 PLPs)."""
    plps = plp_list(c)
    N = c.get("subslices", 1)
    D = [p["fecblocks"] * p["cell_size"] for p in plps]
    slc = [d // N if p["type"] == 2 else d for p, d in zip(plps, D)]
    t2 = [i for i, p in enumerate(plps) if p["type"] == 2]
    type2_start = sum(D[:t2[0]]) if t2 else 0
    start = [sum(D[:i]) if p["type"] != 2 else type2_start + sum(slc[j] for j in t2 if j < i) for i, p in enumerate(plps)]
    return dict(start=start, slice=slc, subslices=N, interval=sum(slc[j] for j in t2), type2_start=type2_start)


def _put(b, pos, v, n):
    b[pos:pos + n] = _bits(v, n)


def l1post_sig_bits_vector(c, frame_idx):
    """plp_oracle's K_sig L1-post bits with the layout fields written at their EN 302 755 7.2.3 offsets -- configurable
    part: SUB_SLICES_PER_FRAME at bit 0, per PLP (89 bits from bit 70) PLP_TYPE at +8 and PLP_GROUP_ID at +28; dynamic
    part (from 70 + 89 P + 32): SUB_SLICE_INTERVAL at +8, TYPE_2_START at +30, per PLP (48 bits from +71) PLP_START at +8
    -- and the CRC-32 recomputed."""
    plps = plp_list(c)
    P, lay = len(plps), layout(c)
    b = list(PO.l1post_sig_bits_vector(c, frame_idx)[:-32])
    _put(b, 0, lay["subslices"], 15)
    for i, p in enumerate(plps):
        _put(b, 70 + 89 * i + 8, p["type"], 3)
        _put(b, 70 + 89 * i + 28, p["group"], 8)
    d = 70 + 89 * P + 32
    _put(b, d + 8, lay["interval"], 22)
    _put(b, d + 30, lay["type2_start"], 22)
    for i in range(P):
        _put(b, d + 71 + 48 * i + 8, lay["start"][i], 22)
    return b + crc32_bits(b)


def l1post_cells(c, frame_idx, n_post, n_punc):
    """plp_oracle.l1post_cells (add_l1post :1536-1910: BCH + LDPC with shortening and puncturing, L1 mapping) over this
    module's signalling bits."""
    v131 = c["version"] == VERSION_131
    sig = np.array(l1post_sig_bits_vector(c, frame_idx), dtype=np.uint8)
    if v131 and c["l1scrambled"]:
        sig ^= bb_prbs(sig.size)
    l1mod = c["l1constellation"]
    suffix = {0: "bqpsk", 1: "bqpsk", 2: "16qam", 3: "64qam"}[l1mod]
    pad, punct = TAB["post_padding_" + suffix], TAB["post_puncture_" + suffix]
    ksig = sig.size
    is_pad = np.zeros(7032, dtype=bool)
    if ksig <= 360:
        m, last = 19, 360 - ksig
    else:
        m = (7032 - ksig) // 360
        last = 7032 - ksig - 360 * m
    for n in range(m):
        g = int(pad[n])
        is_pad[g * 360: g * 360 + (192 if g == 19 else 360)] = True
    g = int(pad[m])
    end = g * 360 + (192 if g == 19 else 360)
    is_pad[end - last:end] = True
    k = np.zeros(7032, dtype=np.uint8)
    k[~is_pad] = sig
    cw = _l1_fec(list(k), 7200, "ldpc_tab_1_2S_L1", 25)
    keep = np.ones(16200, dtype=bool)
    full = n_punc // 360
    for cidx in range(full):
        keep[7200 + np.arange(360) * 25 + int(punct[cidx])] = False
    keep[7200 + np.arange(n_punc - full * 360) * 25 + int(punct[full])] = False
    tx = np.concatenate([cw[:7032][~is_pad], cw[7032:7200], cw[7200:][keep[7200:]]])
    assert tx.size == n_post
    if l1mod == 0:
        return (1.0 - 2.0 * tx).astype(np.complex64)
    eta = [1, 2, 4, 6][l1mod]
    lut = constellation(l1mod - 1, 0)
    if l1mod == 1:
        return lut[(tx[0::2].astype(int) << 1) | tx[1::2]]
    ncol = 2 * eta
    rows = n_post // ncol
    il = tx.reshape(ncol, rows).T
    mux = TAB["l1_mux16" if eta == 4 else "l1_mux64"]
    pack = np.zeros(rows, dtype=np.int64)
    for e in range(ncol):
        pack = (pack << 1) | il[:, int(mux[e])]
    return lut[np.stack([pack >> eta, pack & ((1 << eta) - 1)], axis=1).reshape(-1)]


class FrameMapper(PO.FrameMapper):
    """plp_oracle's frame mapper with the data cells at their layout addresses and this module's L1-post."""

    def __init__(self, c):
        PO.FrameMapper.__init__(self, c)
        self.plps = [dict(q, type=p["type"]) for q, p in zip(self.plps, plp_list(c))]

    def work(self, cells):
        c, d = self.c, self.d
        T = c["tiblocks"]
        blocks = []                                                      # TI blocks (size, PLP), PLP after PLP
        for p in self.plps:
            Fp = p["fecblocks"]
            if T == 0:
                sizes = [1] * Fp
            else:
                small, big = Fp // T, -(-Fp // T)
                nbig = Fp % T
                sizes = [small] * (T - nbig) + [big] * nbig
            blocks += [(k, p) for k in sizes]
        ti = np.empty(self.stream_items, dtype=np.complex64)
        base = 0
        for k, p in blocks:                                              # cell interleaver :1973-1998
            Nc = p["cell_size"]
            n = 0
            for r in range(k):
                shift = Nc
                while shift >= Nc:
                    t, sh = n, 0
                    for _ in range(p["deg"]):
                        sh |= t & 1
                        sh <<= 1
                        t >>= 1
                    shift = sh
                    n += 1
                ti[base + (p["perm"] + shift) % Nc] = cells[base: base + Nc]
                base += Nc
        if T:                                                            # time interleaver :1999-2028
            out, o = np.empty_like(ti), 0
            for k, p in blocks:
                rows = p["cell_size"] // 5
                cols = 5 * k
                out[o:o + rows * cols] = ti[o:o + rows * cols].reshape(cols, rows).T.reshape(-1)
                o += rows * cols
            ti = out
        lay, data, o = layout(c), np.empty_like(ti), 0                   # PLP_START and sub-slices (8.3.6.3)
        for i, p in enumerate(self.plps):
            D = p["fecblocks"] * p["cell_size"]
            L = lay["slice"][i]
            step = lay["interval"] if p["type"] == 2 else L
            for s in range(D // L):
                data[lay["start"][i] + s * step: lay["start"][i] + s * step + L] = ti[o + s * L: o + (s + 1) * L]
            o += D
        l1post = l1post_cells(c, self.t2_frame_num, self.n_post, self.n_punc)
        self.t2_frame_num = (self.t2_frame_num + 1) % c["t2frames"]
        linear = np.concatenate([self.l1pre, l1post, data, self.dummy_cells,
                                 np.zeros(d["n_fc"] - d["c_fc"], dtype=np.complex64)])
        NP, CP = d["n_p2"], d["c_p2"]
        if NP == 1:
            framed = linear
        else:                                                            # zig-zag :2047-2103
            framed = np.empty_like(linear)
            pre, post = 1840 // NP, l1post.size // NP
            rest = CP - pre - post
            read = 1840 + l1post.size
            for n in range(NP):
                framed[n * CP: n * CP + pre] = linear[n: 1840: NP][:pre]
                framed[n * CP + pre: n * CP + pre + post] = linear[1840 + n: 1840 + l1post.size: NP][:post]
                framed[n * CP + pre + post: (n + 1) * CP] = linear[read: read + rest]
                read += rest
            framed[NP * CP:] = linear[read:]
        out, off, sym = np.empty_like(framed), 0, 0                      # frequency interleaver :2104-2142
        for kind, count, n in (("p2", NP, CP), ("data", d["n_data_syms"], d["c_data"]), ("fc", 1 if d["n_fc"] else 0, d["n_fc"])):
            for _ in range(count):
                out[off: off + n] = framed[off + self.H[kind, sym & 1]]
                off += n
                sym += 1
        return out


def chain(c, ts, nframes):
    """plp_oracle.chain (per PLP BB framing + BCH, LDPC, mapper) with the frame built by this module's FrameMapper:
    "mapped" and "samples" follow the layout, every other entry is plp_oracle's."""
    out = PO.chain(c, ts, nframes)
    fm, pg = FrameMapper(c), PilotGen(c)
    mapped = [fm.work(f) for f in out["cells"].reshape(nframes, -1)]
    out["mapped"] = np.concatenate(mapped)
    out["samples"] = np.concatenate([pg.work(m) for m in mapped])
    return out
