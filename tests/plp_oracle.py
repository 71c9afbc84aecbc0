"""TEST INFRASTRUCTURE ONLY -- the numpy restatement (oracle/t2oracle.py) extended to PLPs that each have their own FEC
type, code rate, constellation and rotation: a config with "plps" (a list of dicts with fecblocks and optional framesize,
rate, constellation, rotation; missing keys take the config's values).

Restated from EN 302 755's field list, not from the reference (which is single-PLP): per PLP its own BB framing + BCH,
LDPC, bit interleaver + mapper and cell interleaver (cells per FECFRAME, permutation, shift), time-interleaver rows
N_c / 5 per TI block, L1-post PLP_COD / PLP_MOD / PLP_ROTATION / PLP_FEC_TYPE and PLP_START advancing by each PLP's
cells.  Everything else is oracle/t2oracle.py itself, which stays pinned to the unmodified reference."""
import numpy as np

from oracle.t2oracle import (C1_2, C1_3, C2_3, C2_5, C3_4, C3_5, C4_5, C5_6, TAB, VERSION_111, VERSION_131, BbHeaderBch,
                             PilotGen, bb_prbs, cell_permutation, constellation, crc32_bits, fec_params, interleavermod,
                             ldpc_encode)
from oracle import t2oracle as _O

_bits, _l1_fec = _O._bits, _O._l1_fec
_PLP_KEYS = ("framesize", "rate", "constellation", "rotation")
_PLP_COD = {C1_3: 6, C2_5: 7, C1_2: 0, C3_5: 1, C2_3: 2, C3_4: 3, C4_5: 4, C5_6: 5}


def plp_list(c):
    """Every PLP as a dict of fecblocks, framesize, rate, constellation, rotation, cell_size: cfg["plps"] entries with
    their missing keys taken from the cfg, else the cfg's own parameters for every PLP of oracle.t2oracle.plp_blocks(c)."""
    if c.get("plps"):
        out = [dict({k: c[k] for k in _PLP_KEYS}, **p) for p in c["plps"]]
    else:
        out = [dict({k: c[k] for k in _PLP_KEYS}, fecblocks=nb) for nb in _O.plp_blocks(c)]
    for p in out:
        p["cell_size"] = (64800 if p["framesize"] else 16200) // (2 * (p["constellation"] + 1))
    return out


def l1post_sig_bits(c):
    """K_sig of L1-post: 213 + 137 NUM_PLP bits."""
    return 213 + 137 * len(plp_list(c))


def l1post_sig_bits_vector(c, frame_idx):
    """The K_sig L1-post signalling bits of T2 frame index frame_idx before scrambling and FEC (EN 302 755 7.2.3:
    configurable part from bit 0, dynamic part, CRC-32), as a list of 0/1."""
    v131 = c["version"] == VERSION_131
    bias = bool(c["reservedbiasbits"]) and v131
    plps = plp_list(c)
    r1 = 0x7FF if bias else 0
    ff = 0xFF if bias else 0
    b = _bits(1, 15) + _bits(len(plps), 8) + _bits(0, 4) + _bits(0, 8) + _bits(0, 3) + _bits(729833333, 32)
    for pid, p in enumerate(plps):                    # configurable part, one entry per PLP (:1582-1672 for the single one)
        b += (_bits(pid, 8) + _bits(1, 3) + _bits(3, 5) + [0] + _bits(0, 3) + _bits(0, 8) + _bits(1, 8) +
              _bits(_PLP_COD[p["rate"]], 3) + _bits(p["constellation"], 3) + [p["rotation"]] + _bits(p["framesize"], 2) +
              _bits(p["fecblocks"], 10) + _bits(1, 8) +
              _bits(c["tiblocks"], 8) + [0, 0] + [1 if (c["inband"] and v131) else 0] + _bits(r1, 11) +
              _bits(0 if c["version"] == VERSION_111 else c["inputmode"] + 1, 2) + [0, 0])
    b += _bits(0, 2) + _bits(0x3FFFFFFF if bias else 0, 30)
    b += _bits(frame_idx, 8) + _bits(0, 22) + _bits(0, 22) + _bits(0, 8) + _bits(0, 3) + _bits(ff, 8)
    start = 0
    for pid, p in enumerate(plps):                    # dynamic part: PLP_ID, PLP_START (cell address), PLP_NUM_BLOCKS, reserved
        b += _bits(pid, 8) + _bits(start, 22) + _bits(p["fecblocks"], 10) + _bits(ff, 8)
        start += p["fecblocks"] * p["cell_size"]
    b += _bits(ff, 8)
    return b + crc32_bits(b)



def l1post_cells(c, frame_idx, n_post, n_punc):
    """add_l1post :1536-1910.  plp_id_dynamic is never initialised by the reference (:240 sets plp_id twice);
    it is 0 on a fresh heap and pinned to 0 in oracle/ref_driver.cc."""
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
    il = tx.reshape(ncol, rows).T                       # :1832-1852 column write, row read, no twist
    mux = TAB["l1_mux16" if eta == 4 else "l1_mux64"]
    pack = np.zeros(rows, dtype=np.int64)
    for e in range(ncol):                               # :1879-1907 the map is the SOURCE index here
        pack = (pack << 1) | il[:, int(mux[e])]
    return lut[np.stack([pack >> eta, pack & ((1 << eta) - 1)], axis=1).reshape(-1)]


# --------------------------------------------------------------------------------------------------


def _frame_cfg(c):
    """The config as oracle/t2oracle.py sees it: PLP 0's parameters and the PLP count (what L1-pre, N_post / N_punc and
    the frequency interleaver depend on)."""
    plps = plp_list(c)
    return dict(c, plp_fecblocks=[p["fecblocks"] for p in plps], fecblocks=sum(p["fecblocks"] for p in plps),
                **{k: plps[0][k] for k in _PLP_KEYS})


class FrameMapper(_O.FrameMapper):
    """oracle/t2oracle.py's frame mapper with every PLP's own cell interleaver and time-interleaver rows."""

    def __init__(self, c):
        _O.FrameMapper.__init__(self, _frame_cfg(c))
        self.c = c
        self.plps = plp_list(c)
        for p in self.plps:                                             # cell interleaver of every PLP
            p["perm"], p["deg"] = cell_permutation(p["framesize"], p["constellation"], p["cell_size"])
        self.stream_items = sum(p["fecblocks"] * p["cell_size"] for p in self.plps)
        d = self.d
        self.dummy = self.mapped_items - self.stream_items - 1840 - self.n_post // self.eta - (d["n_fc"] - d["c_fc"])
        self.dummy_cells = (1.0 - 2.0 * bb_prbs(max(self.dummy, 0))).astype(np.complex64)

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
        l1post = l1post_cells(c, self.t2_frame_num, self.n_post, self.n_punc)
        self.t2_frame_num = (self.t2_frame_num + 1) % c["t2frames"]
        linear = np.concatenate([self.l1pre, l1post, ti, self.dummy_cells,
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
    """oracle/t2oracle.py's chain() for nframes T2 frames of one channel, `ts` one transport stream per PLP: per PLP BB
    framing + BCH, LDPC and bit interleaver + mapper.  "bch_plp" / "fec_plp" [PLP] hold each PLP's codewords of all frames."""
    plps = plp_list(c)
    tss = list(ts)
    bbs = [BbHeaderBch(p["framesize"], p["rate"], c["inputmode"], c["inband"], p["fecblocks"], c["tsrate"]) for p in plps]
    fm, pg = FrameMapper(c), PilotGen(c)
    res = dict(cells=[], mapped=[], samples=[])
    bch_plp, fec_plp = [[] for _ in plps], [[] for _ in plps]
    pos = [0] * len(plps)
    for _ in range(nframes):
        cells = []
        for i, p in enumerate(plps):
            bch, used = bbs[i].work(tss[i][pos[i]:], p["fecblocks"])
            pos[i] += used
            fec = ldpc_encode(bch.reshape(p["fecblocks"], -1), p["framesize"], p["rate"])
            cells.append(interleavermod(fec, p["framesize"], p["rate"], p["constellation"], p["rotation"]).reshape(-1))
            bch_plp[i].append(bch)
            fec_plp[i].append(fec.reshape(-1))
        cells = np.concatenate(cells)
        mapped = fm.work(cells)
        samples = pg.work(mapped)
        for k, v in (("cells", cells), ("mapped", mapped), ("samples", samples)):
            res[k].append(v)
    out = {k: np.concatenate(v) for k, v in res.items()}
    out["bch_plp"] = [np.concatenate(v) for v in bch_plp]
    out["fec_plp"] = [np.concatenate(v) for v in fec_plp]
    out["bch"] = np.concatenate([np.concatenate(v) for v in bch_plp])
    out["fec"] = np.concatenate([np.concatenate(v) for v in fec_plp])
    out["ts_used"] = pos
    return out
