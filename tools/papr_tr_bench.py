"""Cost and effect of tone-reservation PAPR reduction (dvbt2ll_chain_set_papr_tr) on the chain.

Configs: c3, c4 and c2 with paprmode = TR, at the FEC block counts that fit the frame once the reserved carriers are
taken out (200, 119 and c2's own 19).  Per config one chain runs 64 channels x 1 T2 frame per step from device-resident
TS and output; the variants -- stage off, then iterations = 10 with vclip 10, 9 and 8 dB above the RMS of the stage-off
output -- alternate in one process (set_papr_tr between steps): warm-up, then ROUNDS rounds of STEPS steps, medians.
The clip level sets how many symbols iterate, and so the time, which is why it is swept.

One JSON line per (config, variant): step ms (host clock around the steps and a device synchronise), the chain's
"ofdm" stage (k_ofdm + k_papr_tr) and its growth over the stage-off variant (the TR cost), the mean updates per symbol
(from the "papr" tap), the achieved L2 bytes/s of the kernel-table reads (updates x N x 8 bytes over the TR cost), the
PAPR at CCDF 1e-3 and 1e-4 over the useful samples of the first channels (stage off against on), tone_max, and the
card name, power limit and maximum SM clock read in the same run.

usage: python tools/papr_tr_bench.py [--channels 64] [--steps 20] [--rounds 4] [--warmup 5] [--tone-max 4.0]
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
    "c3-tr": dict(K.CONFIGS["c3"], paprmode=K.PAPR_TR, fecblocks=200),
    "c4-tr": dict(K.CONFIGS["c4"], paprmode=K.PAPR_TR, fecblocks=119),
    "c2-tr": dict(K.CONFIGS["c2"], paprmode=K.PAPR_TR),
}
ITERATIONS = 10
CLIP_DB = (10.0, 9.0, 8.0)
PAPR_CHANNELS = 4      # channels copied back for the PAPR statistics


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
        self.name, self.nch = name, nch
        self.cfg = K.resolve(CONFIGS[name])
        self.ch = T.Chain(self.cfg, max_frames=nch, device=0)
        self.spf = self.ch.samples_per_frame
        self.pitch = (self.ch.ts_bytes(0, 1) + 255) & ~255
        ts = np.stack([K.make_ts(self.pitch, seed=K.TS_SEED + r) for r in range(nch)])
        self.d_ts = T.DeviceBuffer(ts.nbytes, data=ts)
        self.d_out = T.DeviceBuffer(nch * self.spf * 8)
        self.N = self.cfg["vlength"]
        self.ms, self.stage = {}, {}

    def step(self):
        self.ch.run_device(self.d_ts.ptr, self.pitch, self.nch, 1, 0, self.d_out.ptr, None)

    def useful(self):
        """|x|^2 of the OFDM symbols (P1 dropped) of the first PAPR_CHANNELS channels."""
        n = min(PAPR_CHANNELS, self.nch)
        y = T.copy_to_host(np.empty(n * self.spf, np.complex64), self.d_out.ptr).reshape(n, self.spf)[:, 2048:]
        return np.abs(y.astype(np.complex128)) ** 2

    def timed(self, key, steps):
        T.device_synchronize()
        self.ch.enable_timing(True)
        t0 = time.perf_counter()
        for _ in range(steps):
            self.step()
        T.device_synchronize()
        self.ms.setdefault(key, []).append((time.perf_counter() - t0) * 1e3 / steps)
        self.stage.setdefault(key, []).append(self.ch.stage_ms())
        self.ch.enable_timing(False)


def ccdf_db(p2, probs=(1e-3, 1e-4)):
    """PAPR (dB over the mean power) exceeded by a fraction `prob` of the samples."""
    r = p2 / p2.mean()
    return [round(float(10 * np.log10(np.quantile(r, 1.0 - q))), 3) for q in probs]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=64)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--tone-max", type=float, default=4.0)
    args = ap.parse_args()
    if not T.device_available():
        raise SystemExit("papr_tr_bench: no CUDA device")
    gpu = card()
    for name in CONFIGS:
        r = Run(name, args.channels)
        r.step()
        T.device_synchronize()
        off = r.useful()
        rms = float(np.sqrt(off.mean()))
        variants = [("off", None)] + [("tr%gdB" % db, rms * 10 ** (db / 20)) for db in CLIP_DB]

        def setv(v):
            r.ch.set_papr_tr(ITERATIONS if v is not None else 0, v if v is not None else 1.0, args.tone_max)
        for key, v in variants:
            setv(v)
            for _ in range(args.warmup):
                r.step()
        for k in range(args.rounds):
            for key, v in (variants if k % 2 == 0 else variants[::-1]):
                setv(v)
                r.timed(key, args.steps)
        med = {key: {s: float(np.median([x[s] for x in r.stage[key]])) for s in r.stage[key][0]} for key, _ in variants}
        for key, v in variants:
            setv(v)
            r.step()
            T.device_synchronize()
            line = dict(config=name, variant=key, channels=args.channels, frames=1, steps=args.steps, rounds=args.rounds,
                        ms_per_step_median=round(float(np.median(r.ms[key])), 4),
                        ms_per_step_all=[round(x, 4) for x in r.ms[key]],
                        stage_ms_median={s: round(x, 4) for s, x in med[key].items()},
                        papr_db_ccdf_1e3_1e4_off=ccdf_db(off), card=gpu)
            if v is not None:
                st = r.ch.tap("papr", np.int16)
                upd = (st & 0xFF).astype(np.int64)
                tr_ms = med[key]["ofdm"] - med["off"]["ofdm"]
                table_bytes = float(upd.sum()) * r.N * 8
                line.update(iterations=ITERATIONS, vclip_db_over_rms=float(key[2:-2]), vclip=round(v, 5),
                            rms_off=round(rms, 5), tone_max=args.tone_max, tr_ms=round(tr_ms, 4),
                            mean_updates_per_symbol=round(float(upd.mean()), 3),
                            stop_reasons={n: int(((st >> 8) == c).sum()) for n, c in (("clip", 1), ("tone", 2), ("limit", 3))},
                            table_l2_gbytes_per_s=round(table_bytes / (tr_ms * 1e-3) / 1e9, 1) if tr_ms > 0 else None,
                            papr_db_ccdf_1e3_1e4_on=ccdf_db(r.useful()))
            print(json.dumps(line), flush=True)
        del r
        T.device_synchronize()


if __name__ == "__main__":
    main()
