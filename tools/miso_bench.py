"""Cost of MISO processing (dvbt2ll_chain_set_miso) and what the dual call (dvbt2ll_chain_run_device_miso) saves.

Configs: c3 and c4 with preamble = T2_MISO (c3 then fits 201 FEC blocks, c4 its own 120).  Per config three chains run
64 channels x 1 T2 frame per step from device-resident TS and output, alternating in one process: (a) misogroup TX1,
(b) misogroup TX2 with MISO processing, (c) the dual call, both groups from one BB/BCH, LDPC and mapper pass.  Warm-up,
then ROUNDS rounds of STEPS steps (the order reversed every other round), medians.

One JSON line per (config, variant): step ms (host clock around the steps and a device synchronise) and the chain's
stage ms; then one summary line per config: (b - a) in "ofdm" (the cost of the sign flip and the paired look-up), and
(c) against (a) + (b) (what the shared front end saves).  The card name, power limit and maximum SM clock are read in
the same run.

usage: python tools/miso_bench.py [--channels 64] [--steps 20] [--rounds 4] [--warmup 5]
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
    "c3-miso": dict(K.CONFIGS["c3"], preamble=K.PREAMBLE_T2_MISO, fecblocks=201),
    "c4-miso": dict(K.CONFIGS["c4"], preamble=K.PREAMBLE_T2_MISO),
}
VARIANTS = ("tx1", "tx2-miso", "dual")


def card():
    """Name, power limit and maximum SM clock of device 0 (read-only query)."""
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip()
    except Exception as e:          # the numbers are still printed; the card line says why it is missing
        return "unknown (%s)" % e


class Run(object):
    def __init__(self, cfg, variant, nch, d_ts, pitch):
        self.variant, self.nch, self.d_ts, self.pitch = variant, nch, d_ts, pitch
        self.ch = T.Chain(dict(cfg, misogroup=1 if variant == "tx2-miso" else 0), max_frames=nch, device=0)
        if variant == "tx2-miso":
            self.ch.set_miso(1)
        spf = self.ch.samples_per_frame
        self.d_out = [T.DeviceBuffer(nch * spf * 8) for _ in range(2 if variant == "dual" else 1)]
        self.ms, self.stage = [], []

    def step(self):
        if self.variant == "dual":
            self.ch.run_device_miso(self.d_ts.ptr, self.pitch, self.nch, 1, 0, self.d_out[0].ptr, self.d_out[1].ptr, None)
        else:
            self.ch.run_device(self.d_ts.ptr, self.pitch, self.nch, 1, 0, self.d_out[0].ptr, None)

    def timed(self, steps):
        T.device_synchronize()
        self.ch.enable_timing(True)
        t0 = time.perf_counter()
        for _ in range(steps):
            self.step()
        T.device_synchronize()
        self.ms.append((time.perf_counter() - t0) * 1e3 / steps)
        self.stage.append(self.ch.stage_ms())
        self.ch.enable_timing(False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=64)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not T.device_available():
        raise SystemExit("miso_bench: no CUDA device")
    gpu = card()
    for name, c in CONFIGS.items():
        cfg = K.resolve(c)
        probe = T.Chain(cfg, max_frames=1)
        pitch = (probe.ts_bytes(0, 1) + 255) & ~255
        ts = np.stack([K.make_ts(pitch, seed=K.TS_SEED + r) for r in range(args.channels)])
        d_ts = T.DeviceBuffer(ts.nbytes, data=ts)
        runs = {v: Run(cfg, v, args.channels, d_ts, pitch) for v in VARIANTS}
        for r in runs.values():
            for _ in range(args.warmup):
                r.step()
        for k in range(args.rounds):
            for v in (VARIANTS if k % 2 == 0 else VARIANTS[::-1]):
                runs[v].timed(args.steps)
        med = {}
        for v, r in runs.items():
            med[v] = dict(step=float(np.median(r.ms)),
                          **{s: float(np.median([x[s] for x in r.stage])) for s in r.stage[0]})
            print(json.dumps(dict(config=name, variant=v, channels=args.channels, frames=1, steps=args.steps,
                                  rounds=args.rounds, ms_per_step_median=round(med[v]["step"], 4),
                                  ms_per_step_all=[round(x, 4) for x in r.ms],
                                  stage_ms_median={s: round(x, 4) for s, x in med[v].items() if s != "step"}, card=gpu)),
                  flush=True)
        a, b, d = med["tx1"], med["tx2-miso"], med["dual"]
        print(json.dumps(dict(config=name, summary=True,
                              miso_ofdm_cost_ms=round(b["ofdm"] - a["ofdm"], 4),
                              miso_ofdm_cost_rel=round((b["ofdm"] - a["ofdm"]) / a["ofdm"], 4),
                              dual_step_ms=round(d["step"], 4), two_chains_step_ms=round(a["step"] + b["step"], 4),
                              dual_saves_ms=round(a["step"] + b["step"] - d["step"], 4),
                              front_end_ms=round(a["bb_bch"] + a["ldpc"] + a["map"], 4), card=gpu)), flush=True)
        del runs
        T.device_synchronize()


if __name__ == "__main__":
    main()
