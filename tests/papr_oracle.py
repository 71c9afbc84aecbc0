"""Tone-reservation PAPR reduction (EN 302 755 9.6.2, peak-cancellation form) restated in float64 numpy: the checker of
the chain's k_papr_tr stage (dvbt2ll_chain_set_papr_tr).  The reserved carriers come from the reference-pinned
oracle's carrier map (oracle/t2oracle.py PilotGen.carrier_map)."""
import numpy as np

from oracle import t2oracle as O

STOP_CLIP, STOP_TONE, STOP_LIMIT = 1, 2, 3
AMBIGUOUS_REL = 1e-5


def reserved_bins(cfg, l, pg=None):
    """FFT bins of symbol l's reserved carriers (P2PAPR / TRPAPR), in carrier order: bin (k + left_nulls + N/2) mod N."""
    pg = pg or O.PilotGen(cfg)
    m = pg.carrier_map(l)
    k = np.nonzero((m == O.P2PAPR) | (m == O.TRPAPR))[0]
    N = pg.d["N"]
    return ((k + pg.left + N // 2) % N).astype(np.int64)


def tr_kernel(bins, N):
    """p_n = (1/|S|) sum_{b in S} exp(+j 2 pi b n / N), complex128."""
    n = np.arange(N, dtype=np.int64)
    acc = np.zeros(N, dtype=np.complex128)
    for b in bins:
        acc += np.exp(2j * np.pi * ((int(b) * n) % N) / N)
    return acc / len(bins)


def tr_reduce(x, bins, iterations, vclip, tone_max, g, kernel=None):
    """Peak cancellation of one symbol's useful samples x.  Returns dict(out, applied, reason, ambiguous, R):
    `ambiguous` is raised when a decision of the trace was within 1e-5 relative (the two largest |c|, y against vclip,
    the largest |R_b + dR_b| against tone_max), where float32 arithmetic may decide the other way."""
    c = np.asarray(x, dtype=np.complex128).copy()
    N, S = c.size, len(bins)
    bins = np.asarray(bins, dtype=np.int64)
    p = tr_kernel(bins, N) if kernel is None else kernel
    R = np.zeros(S, dtype=np.complex128)
    V, A = float(vclip), float(tone_max)
    ambiguous, applied, reason = False, 0, STOP_LIMIT
    for _ in range(iterations):
        a = np.abs(c)
        m = int(np.argmax(a))
        y = a[m]
        top2 = np.partition(a, -2)[-2:]
        if top2[1] - top2[0] <= AMBIGUOUS_REL * top2[1]:
            ambiguous = True
        if abs(y - V) <= AMBIGUOUS_REL * V:
            ambiguous = True
        if y <= V:
            reason = STOP_CLIP
            break
        beta = (y - V) * c[m] / y
        dR = -beta * np.exp(-2j * np.pi * ((bins * m) % N) / N) / (g * S)
        mx = np.abs(R + dR).max()
        if abs(mx - A) <= AMBIGUOUS_REL * A:
            ambiguous = True
        if mx > A:
            reason = STOP_TONE
            break
        R = R + dR
        c = c - beta * np.roll(p, m)      # p[(n - m) mod N]
        applied += 1
    return dict(out=c, applied=applied, reason=reason, ambiguous=ambiguous, R=R)
