"""MISO processing (EN 302 755 9.1, modified Alamouti) restated on top of the reference-pinned oracle/t2oracle.py.

The reference sends group 1's cells from both transmitter groups; group 2 here sends, per OFDM symbol with cells g_i in
the order the frequency interleaver emits them (L1, dummy and unmodulated cells included), e_2i = -conj(g_2i+1) and
e_2i+1 = conj(g_2i).  Each group keeps its own pilots.  No reference output exists for this; alamouti_combine() is a
receiver that shows the two outputs form a decodable pair."""
import numpy as np

from oracle import t2oracle as O


def symbol_cells(cfg):
    """Data cells per OFDM symbol (the count of DATA carriers; the same for both groups)."""
    pg = O.PilotGen(cfg)
    return [int((pg.carrier_map(l) == O.DATA).sum()) for l in range(pg.d["L"])]


def alamouti(g, counts):
    """Group 2's cells of one T2 frame from group 1's (frame-mapper output g)."""
    e, pos = np.empty_like(g), 0
    for n in counts:
        s = g[pos:pos + n]
        e[pos:pos + n:2] = -np.conj(s[1::2])
        e[pos + 1:pos + n:2] = np.conj(s[0::2])
        pos += n
    return e


def miso_samples(cfg, mapped, nframes):
    """(group 1, group 2 with MISO processing) baseband of frames whose frame-mapper output is `mapped`."""
    counts = symbol_cells(cfg)
    frames = mapped.reshape(nframes, sum(counts))
    g1, g2 = O.PilotGen(dict(cfg, misogroup=0)), O.PilotGen(dict(cfg, misogroup=1))
    return (np.concatenate([g1.work(f) for f in frames]),
            np.concatenate([g2.work(alamouti(f, counts)) for f in frames]))


def data_carriers(cfg, y, nframes):
    """Per (frame, symbol): the data-carrier values of baseband y (GI dropped, FFT, divided by N * norm)."""
    pg = O.PilotGen(cfg)
    N, L, gi, cps = pg.d["N"], pg.d["L"], pg.d["gi"], pg.d["c_ps"]
    syms = y.reshape(nframes, -1)[:, 2048:].reshape(nframes, L, N + gi)[..., gi:].astype(np.complex128)
    spec = np.fft.fftshift(np.fft.fft(syms, axis=-1), axes=-1) / (N * np.float64(pg.norm))
    X = spec[..., pg.left:pg.left + cps]
    return [[X[f, l][pg.carrier_map(l) == O.DATA] for l in range(L)] for f in range(nframes)]


def alamouti_combine(cfg, y1, y2, nframes, seed=0):
    """Receiver: r = h1 X1 + h2 X2 on the data carriers, random complex h1, h2 per symbol, then
    g_2i = (conj(h1) r_2i + h2 conj(r_2i+1)) / (|h1|^2 + |h2|^2), g_2i+1 = (conj(h1) r_2i+1 - h2 conj(r_2i)) / (...).
    Returns the recovered cells of all frames, in frame-mapper order."""
    rng = np.random.default_rng(seed)
    x1, x2 = data_carriers(cfg, y1, nframes), data_carriers(cfg, y2, nframes)
    out = []
    for f in range(nframes):
        for a, b in zip(x1[f], x2[f]):
            h1, h2 = rng.standard_normal(2) @ [1, 1j], rng.standard_normal(2) @ [1, 1j]
            r = h1 * a + h2 * b
            g = np.empty_like(r)
            p = abs(h1) ** 2 + abs(h2) ** 2
            g[0::2] = (np.conj(h1) * r[0::2] + h2 * np.conj(r[1::2])) / p
            g[1::2] = (np.conj(h1) * r[1::2] - h2 * np.conj(r[0::2])) / p
            out.append(g)
    return np.concatenate(out)
