"""Kernel launches per chain run: every PLP gets its own BB / BCH launch, and each FEC group (all PLPs when they share
one parameter set, else each PLP) one LDPC and one mapper launch; then one k_ofdm per output and k_papr_tr when tone
reservation is on.  A chain whose PLPs share their parameters must not fall back to a launch per PLP: its outputs would
not change, only its speed."""
import numpy as np
import pytest

import dvbt2ll_b200 as T
from dvbt2ll_b200 import configs as K
import test_miso
import test_papr_tr
import test_plp_modcod


def _ts(ch):
    """One T2 frame of TS for one channel: a row per PLP."""
    width = max(ch.plp_ts_bytes(p, 0, 1) for p in range(ch.num_plp))
    return np.stack([K.make_ts(width, seed=K.TS_SEED + p) for p in range(ch.num_plp)])


# (name, cfg, launches): P BB + groups x (LDPC + mapper) + k_ofdm
CASES = [
    ("c1", K.resolve("c1"), 1 + 2 + 1),
    ("c2", K.resolve("c2"), 1 + 2 + 1),
    ("c3", K.resolve("c3"), 1 + 2 + 1),
    ("c4", K.resolve("c4"), 1 + 2 + 1),
    ("c1-3plp-inband", K.resolve(test_plp_modcod.MULTIPLP["c1-3plp-inband"]), 3 + 2 + 1),
    ("c1-mix", test_plp_modcod.resolve("c1-mix"), 2 + 2 * 2 + 1),
    ("c1-qpsk-rates", test_plp_modcod.resolve("c1-qpsk-rates"), 2 + 2 * 2 + 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfg,launches", CASES, ids=[c[0] for c in CASES])
def test_launches_per_run(name, cfg, launches):
    ch = T.Chain(cfg, max_frames=1)
    ts = _ts(ch)
    ch.run_host(ts, 1, 1)                 # device set-up outside the count
    l0 = T.kernel_launches()
    ch.run_host(ts, 1, 1)
    assert T.kernel_launches() - l0 == launches, name


@pytest.mark.gpu
def test_launches_with_tone_reservation():
    ch = T.Chain(test_papr_tr.GPU_CASES["c3-tr"], max_frames=1)
    ch.set_papr_tr(4, 2.0, 1.0)
    ts = _ts(ch)
    ch.run_host(ts, 1, 1)
    l0 = T.kernel_launches()
    ch.run_host(ts, 1, 1)
    assert T.kernel_launches() - l0 == 1 + 2 + 1 + 1


@pytest.mark.gpu
def test_launches_of_the_miso_dual_call():
    ch = T.Chain(test_miso.CASES["4k-fc"], max_frames=1)
    ts = _ts(ch)
    ch.run_host_miso(ts, 1, 1)
    l0 = T.kernel_launches()
    ch.run_host_miso(ts, 1, 1)
    assert T.kernel_launches() - l0 == 1 + 2 + 2
