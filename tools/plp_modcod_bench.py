"""Time a chain whose PLPs have their own constellations against the single-ModCod chain of the same frame.

c3-mix: c3's 32K extended frame with a normal 256QAM 2/3 rotated PLP x 150 and a normal 16QAM 1/2 rotated PLP x 25, so
k_ofdm runs its two-table form; c3: the same frame with one PLP.  Both chains run 64 channels x 1 T2 frame per step from
device-resident TS and output (no host copies), alternating in one process: warm-up, then ROUNDS rounds of STEPS steps
each.  Prints one JSON line per chain: Msamples/s from a host clock around the steps and a device synchronise, the
chain's own per-stage CUDA events (bb_bch, ldpc, map, ofdm, total), the constellation-table copies k_ofdm kept in shared
memory, and the card name and power limit the numbers were taken on.

usage: python tools/plp_modcod_bench.py [--channels 64] [--steps 20] [--rounds 4] [--warmup 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "gr-dvbt2ll_b200", "python")):
    if p not in sys.path:
        sys.path.insert(0, p)

import dvbt2ll_b200 as T  # noqa: E402
from dvbt2ll_b200 import configs as K  # noqa: E402

CONFIGS = {
    "c3-mix": dict(K.CONFIGS["c3"], plps=[
        dict(fecblocks=150, framesize=K.FECFRAME_NORMAL, rate=K.C2_3, constellation=K.MOD_256QAM, rotation=1),
        dict(fecblocks=25, framesize=K.FECFRAME_NORMAL, rate=K.C1_2, constellation=K.MOD_16QAM, rotation=1)]),
    "c3": K.CONFIGS["c3"],
}


def card():
    """Name, power limit and maximum SM clock of device 0 (read-only query)."""
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip()
    except Exception as e:          # the numbers are still printed; the card line says why it is missing
        return "unknown (%s)" % e


class Run(object):
    def __init__(self, name, nch):
        self.name = name
        self.ch = T.Chain(CONFIGS[name], max_frames=nch, device=0)
        self.nch, P = nch, self.ch.num_plp
        self.pitch = (max(self.ch.plp_ts_bytes(p, 0, 1) for p in range(P)) + 255) & ~255
        ts = np.zeros((nch * P, self.pitch), np.uint8)
        for r in range(nch * P):
            ts[r, :self.pitch] = K.make_ts(self.pitch, seed=K.TS_SEED + r)
        self.d_ts = T.DeviceBuffer(ts.nbytes, data=ts)
        self.d_out = T.DeviceBuffer(nch * self.ch.samples_per_frame * 8)
        self.samples = nch * self.ch.samples_per_frame
        self.ms = []

    def step(self):
        self.ch.run_device(self.d_ts.ptr, self.pitch, self.nch, 1, 0, self.d_out.ptr, None)

    def timed(self, steps):
        T.device_synchronize()
        self.ch.enable_timing(True)
        t0 = time.perf_counter()
        for _ in range(steps):
            self.step()
        T.device_synchronize()
        self.ms.append((time.perf_counter() - t0) * 1e3 / steps)
        stage = self.ch.stage_ms()
        self.ch.enable_timing(False)
        return stage


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=64)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not T.device_available():
        raise SystemExit("plp_modcod_bench: no CUDA device")
    gpu = card()
    runs = [Run(n, args.channels) for n in ("c3-mix", "c3")]
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
            msamples_per_s=round(r.samples / (float(np.median(r.ms)) * 1e-3) / 1e6, 1),
            stage_ms_median=st, lut_tables=int(luts[0]), lut_single=int(luts[1]), lut_copies=int(luts[2]),
            card=gpu)))


if __name__ == "__main__":
    main()
