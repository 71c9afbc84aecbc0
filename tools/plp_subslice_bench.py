"""Time a chain whose PLPs are type-2 data PLPs with sub-slicing against the same PLPs as type-1 data PLPs.

c3-mix-t1: c3's 32K extended frame with a normal 256QAM 2/3 rotated PLP x 150 and a normal 16QAM 1/2 rotated PLP x 25,
both type 1 (one block of cells each); c3-mix-t2: the same PLPs as type 2 with 135 sub-slices per frame (D = 1,215,000
and 405,000 cells: sub-slices of 9000 and 3000 cells, SUB_SLICE_INTERVAL 12000).  The kernels and their launches are
the same; only the frame builder's gather, and with it k_ofdm's staging (bulk copies per symbol, staging bytes, the
constellation-table copies that fit beside them in shared memory), differs.  Both chains run 64 channels x 1 T2 frame per
step from device-resident TS and output (no host copies), alternating in one process: warm-up, then ROUNDS rounds of
STEPS steps each.  Prints one JSON line per chain: ms per step from a host clock around the steps and a device
synchronise, the chain's own per-stage CUDA events (bb_bch, ldpc, map, ofdm, total), the largest number of bulk copies of
one symbol, the largest staging bytes of one symbol, the constellation-table copies k_ofdm kept in shared memory, and the
card name and power limit the numbers were taken on.

usage: python tools/plp_subslice_bench.py [--channels 64] [--steps 20] [--rounds 4] [--warmup 5]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gr-dvbt2ll_b200", "python")):
    if p not in sys.path:
        sys.path.insert(0, p)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import dvbt2ll_b200 as T  # noqa: E402
from dvbt2ll_b200 import configs as K  # noqa: E402
import plp_modcod_bench as B  # noqa: E402

C3_MIX = B.CONFIGS["c3-mix"]
CONFIGS = {
    "c3-mix-t1": C3_MIX,
    "c3-mix-t2": dict(C3_MIX, plps=[dict(q, type=2) for q in C3_MIX["plps"]], subslices=135),
}
B.CONFIGS.update(CONFIGS)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=64)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not T.device_available():
        raise SystemExit("plp_subslice_bench: no CUDA device")
    gpu = B.card()
    runs = [B.Run(n, args.channels) for n in ("c3-mix-t1", "c3-mix-t2")]
    for r in runs:
        for _ in range(args.warmup):
            r.step()
    T.device_synchronize()
    stages = {r.name: [] for r in runs}
    for k in range(args.rounds):
        for r in (runs if k % 2 == 0 else runs[::-1]):
            stages[r.name].append(r.timed(args.steps))
    for r in runs:
        st = {key: round(float(np.median([s[key] for s in stages[r.name]])), 4) for key in stages[r.name][0]}
        luts = r.ch.plan("chain.luts", np.int32)
        print(json.dumps(dict(
            config=r.name, channels=args.channels, frames=1, steps=args.steps, rounds=args.rounds,
            ms_per_step_median=round(float(np.median(r.ms)), 4), ms_per_step_all=[round(x, 4) for x in r.ms],
            stage_ms_median=st, max_runs=int(r.ch.plan("chain.run_cnt", np.int32).max()),
            max_stage_bytes=int(r.ch.plan("chain.stage_bytes", np.int32).max()), lut_copies=int(luts[2]),
            card=gpu)))


if __name__ == "__main__":
    main()
