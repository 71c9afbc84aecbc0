#!/usr/bin/env python
"""bench.py -- DVB-T2 modulator hot path on B200: T2 baseband MS/s (x real-time) and FECFRAMEs/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the fused chain (TS bytes -> complex baseband) over one batch of synthetic transport
streams: BASELINE.json config 5 = 64 independent 32K / 256QAM-rotated / CR 2/3 channels (config 3), one T2
frame per channel per step, the 64 channels sharded over the N GPUs of the job (64 / N channels each: STRONG
scaling, "config 5 as stated") with seeds 0x12345678 + global channel index.  There is no data-path
collective; at N > 1 every step ends with the ordered reassembly of all ranks' frames on GPU 0 through the
library's own entry points (dvbt2ll_gather_*: one NVLink peer copy per rank on a side stream, double-buffered,
overlapping the rank's next step) and that reassembly is INSIDE the timed value.

value      = whole-job output Msamples/s, TS resident in HBM, at N > 1 including the ordered reassembly on GPU 0
             (CUDA events on the launching streams, max over ranks)
e2e        = same metric through dvbt2ll_chain_run_host(): pinned HOST TS in, HOST samples out, copies timed
roofline   = the dominant kernel (k_ofdm: carrier fill + IFFT + GI) against the measured HBM copy peak
cpu_baseline / --impl reference = the UNMODIFIED reference flowgraph (oracle/_ref, GNU Radio shim) on host cores

PyTorch is only plumbing here (device buffers, streams/events, torch.distributed); the hot path is
libdvbt2ll_cuda.so called through its C ABI.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gr-dvbt2ll_b200", "python"))

import numpy as np  # noqa: E402

METRIC = "t2_baseband_msps"
UNIT = "Msamples/s"
NVLINK_PEER_GBS = 770.0     # measured peer copy per direction per GPU on this pool (B200_PROFILING.md); nominal 900


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", help="per-channel configuration (c1..c4)")
    ap.add_argument("--channels", type=int, default=64, help="independent channels of the whole job per step")
    ap.add_argument("--frames", type=int, default=1, help="T2 frames per channel per step")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-frames", type=int, default=24, help="T2 frames timed for cpu_baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip per_config / dropin_e2e (N = 1 extras)")
    ap.add_argument("--no-parity", action="store_true", help="skip the untimed per-rank parity check")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed sample of the last step's baseband "
                                                          "(what the caller of the timed path receives) as DIR/*.npy")
    ap.add_argument("--deadline", type=int, default=-1, help="seconds after which a run without a result reports where it stopped and exits "
                                                             "(default: 420 for N > 1, 1500 for N = 1; 0 = never)")
    return ap.parse_args()


def workload_name(args):
    if args.config == "c3":
        return ("c5: %d x c3 channels (32K ext, 256QAM rot, CR 2/3, GI 1/128, PP7, 202 FECFRAMEs/T2 frame), %d T2 frame/channel/step, "
                "channels sharded over the GPUs" % (args.channels, args.frames))
    return "%d x %s channels, %d T2 frame/channel/step, channels sharded over the GPUs" % (args.channels, args.config, args.frames)


def config_dict(args, S, F):
    """The `config` object: identical keys and values on the repo arm and the reference arm."""
    frames = args.channels * args.frames
    return {"workload": workload_name(args), "per_channel_config": args.config, "channels": args.channels,
            "t2_frames_per_channel_per_step": args.frames, "t2_frames_per_step": frames,
            "fecframes_per_step": frames * F, "samples_per_step": frames * S}


# --------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU reference arm: unmodified reference flowgraph (oracle/_ref) on host cores
# --------------------------------------------------------------------------------------------------
def _ref_worker(job):
    cfg, seeds, nframes = job
    from oracle import ref
    from dvbt2ll_b200 import configs as K
    ref.lib().ref_set_quiet(1)
    ref.lib().ref_set_fft_fast(1)      # float Stockham FFT stand-in for FFTW (oracle/shim/gnuradio/fft/fft.h)
    ref.lib().ref_fft_seconds(1)
    timers = {}
    n, busy = 0, 0.0
    for seed in seeds:                 # one channel per seed, nframes consecutive T2 frames of it
        ch = ref.Chain(cfg)
        ts = K.make_ts((nframes + 1) * ch.ts_bytes_per_t2_frame() + 1000, seed=seed)
        t0 = time.perf_counter()
        for _ in range(nframes):
            n += ch.run_frame(ts, timers=timers)["samples"].size
        busy += time.perf_counter() - t0
    timers["fft"] = ref.lib().ref_fft_seconds(1)
    return n, busy, timers


def cpu_reference_run(cfg, channels, nframes, procs):
    """Times `channels` independent channels x `nframes` T2 frames of the reference chain on `procs` host
    processes (channels dealt round-robin). Returns dict or None."""
    from oracle import ref
    if not ref.available():
        return None
    from dvbt2ll_b200 import configs as K
    procs = max(1, min(procs, channels))
    jobs = [(cfg, [K.TS_SEED + c for c in range(p, channels, procs)], nframes) for p in range(procs)]
    t0 = time.perf_counter()
    if procs == 1:
        res = [_ref_worker(jobs[0])]
    else:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(procs) as pool:
            res = pool.map(_ref_worker, jobs)
    wall = time.perf_counter() - t0
    samples = sum(r[0] for r in res)
    busy = max(r[1] for r in res)
    stage = {}
    for r in res:
        for k, v in r[2].items():
            stage[k] = stage.get(k, 0.0) + v
    return {"samples": samples, "seconds": busy, "wall": wall, "frames": channels * nframes, "procs": procs,
            "stage_seconds": {k: round(v, 4) for k, v in stage.items()}}


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown CPU"


def run_reference_arm(args):
    from dvbt2ll_b200 import configs as K
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = K.resolve(args.config)
    procs = max(1, min(len(os.sched_getaffinity(0)), 64, args.channels))
    warm = max(0, min(args.warmup, 1))
    for _ in range(warm):
        cpu_reference_run(cfg, min(procs, args.channels), 1, procs)
    tot_s, tot_t = 0, 0.0
    stage = {}
    r = None
    for _ in range(args.steps):
        r = cpu_reference_run(cfg, args.channels, args.frames, procs)     # the whole step: every channel, 64 / P per process
        if r is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libdvbt2ll_ref.so not built"}))
            return
        tot_s += r["samples"]; tot_t += r["seconds"]
        for k, v in r["stage_seconds"].items():
            stage[k] = stage.get(k, 0.0) + v
    value = tot_s / tot_t / 1e6
    F = cfg["fecblocks"]
    S = r["samples"] // r["frames"]
    stage_sum = sum(v for k, v in stage.items() if k != "fft")
    fft_share = stage.get("fft", 0.0) / stage_sum if stage_sum > 0 else None
    sample = ("%d channels x %d T2 frame(s) of %s per step (the whole step) x %d steps, %d worker processes (%d channel(s) each) on %s; "
              "unmodified reference sources + GNU Radio shim, single-precision radix-4 FFT stand-in for FFTW; stage CPU-seconds %s" % (
                  args.channels, args.frames, args.config, args.steps, r["procs"], (args.channels + r["procs"] - 1) // r["procs"], cpu_model(),
                  json.dumps({k: round(v, 2) for k, v in stage.items()})))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": warm, "ms_per_step": 1e3 * tot_t / max(1, args.steps), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u8/f32", "data": "synthetic",
        "config": config_dict(args, S, F),
        "x_realtime": value / K.REALTIME_MSPS, "fecframes_per_s": value * 1e6 / S * F,
        "fft_share_of_cpu_time": fft_share,
        "value_without_fft": (value / (1.0 - fft_share)) if fft_share is not None and fft_share < 1 else None,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": r["procs"], "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
DUMP_SAMPLES = 1 << 21      # 16 MB of float32 I/Q + 16 MB of float64 indices


def dump_outputs(path, out):
    """Write the timed path's output `out` (complex64 [channels, samples per channel]) for output-by-output comparison
    of two builds: baseband.npy = float32 [n, 2] (I, Q) at the flat indices in baseband_index.npy (float64), a sample
    drawn with a fixed seed (the whole array when it is small enough)."""
    flat = out.reshape(-1)
    if flat.size <= DUMP_SAMPLES:
        idx = np.arange(flat.size)
    else:
        idx = np.sort(np.random.default_rng(20261020).choice(flat.size, DUMP_SAMPLES, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "baseband.npy"), flat[idx].view(np.float32).reshape(-1, 2))
    np.save(os.path.join(path, "baseband_index.npy"), idx.astype(np.float64))


def mer_db(got, want):
    err = np.sum(np.abs(got.astype(np.complex128) - want) ** 2)
    sig = np.sum(np.abs(want.astype(np.complex128)) ** 2)
    return float(10 * np.log10(sig / max(err, 1e-300)))


def reference_frame(cfg, ts_row):
    """First T2 frame of one channel through the checker (oracle/_ref when built, else the numpy oracle)."""
    from oracle import ref
    if ref.available():
        ref.lib().ref_set_quiet(1)
        ref.lib().ref_set_fft_fast(0)
        return ref.Chain(cfg).run_frame(np.concatenate([ts_row, np.zeros(2048, np.uint8)]))["samples"], "oracle/_ref"
    from oracle import t2oracle
    return t2oracle.chain(cfg, ts_row, 1)["samples"], "oracle/t2oracle.py"


def stage_roofline(chain, cfg, frames, stage_ms, peak, peak_src):
    """Dominant-kernel roofline of a chain configuration from the per-stage CUDA-event times."""
    S, F = chain.samples_per_frame, chain.fecframes_per_frame
    nldpc = 64800 if cfg["framesize"] else 16200
    cell_size = nldpc // (2 * (cfg["constellation"] + 1))
    dims = chain.plan("ofdm.dims", np.int32)
    active_items = int(dims[15])
    ofdm_bytes = frames * 8 * (active_items + S)              # SURVEY 8(d): 8*mapped_items + 8*samples per T2 frame
    map_bytes = frames * F * (nldpc // 8 + 2 * cell_size)     # chain mode: packed codewords in, 16-bit cell codes out
    ach = ofdm_bytes / (stage_ms["ofdm"] * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": "k_ofdm (cell staging + carrier fill + IFFT + scale + guard interval + P1)",
            "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": ofdm_bytes, "kernel_ms": stage_ms["ofdm"], "stage_ms": stage_ms,
            "fec_frontend_ms": sum(v for k, v in stage_ms.items() if k in ("bb_bch", "ldpc", "map", "ldpc_map")),
            "map_kernel_gbs": (map_bytes / (stage_ms["map"] * 1e-3) / 1e9) if "map" in stage_ms else None}


def time_chain(torch, chain, stream, d_ts, pitch, nch, nfr, d_out, steps, min_warm_s=0.2):
    """Warm up, then time `steps` device-resident runs with CUDA events on the launching stream. Returns (ms/step, stage_ms)."""
    sp = stream.cuda_stream
    chain.enable_timing(False)
    t_w, n_w = time.perf_counter(), 0
    while n_w < 3 or time.perf_counter() - t_w < min_warm_s:
        chain.run_device(d_ts.data_ptr(), pitch, nch, nfr, 0, d_out.data_ptr(), sp)
        n_w += 1
        if n_w % 8 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    chain.enable_timing(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        chain.run_device(d_ts.data_ptr(), pitch, nch, nfr, 0, d_out.data_ptr(), sp)
    e1.record(stream)
    torch.cuda.synchronize()
    st = chain.stage_ms()
    chain.enable_timing(False)
    return e0.elapsed_time(e1) / steps, st, n_w


def per_config_extras(torch, T, K, dev, stream, peak, peak_src, steps):
    """c1, c2, c4 (BASELINE.json configs[0], [1], [3]) on one GPU, 64 channels each: device MS/s, x real time, FECFRAMEs/s,
    per-stage ms, dominant-kernel roofline, and the unmodified reference on one host core beside it."""
    out = {}
    for name, nch, nfr in (("c1", 64, 8), ("c2", 64, 1), ("c4", 64, 1)):
        cfg = K.resolve(name)
        chain = T.Chain(cfg, max_frames=nch * nfr, device=dev.index)
        n_ts, S, F = chain.ts_bytes_per_frame, chain.samples_per_frame, chain.fecframes_per_frame
        pitch = (nfr * n_ts + 255) // 256 * 256
        ts = np.zeros((nch, pitch), np.uint8)
        for c in range(nch):
            ts[c, :nfr * n_ts] = K.make_ts(nfr * n_ts, seed=K.TS_SEED + c)
        d_ts = torch.from_numpy(ts).to(dev)
        d_out = torch.empty((nch, nfr * S), dtype=torch.complex64, device=dev)
        ms, st, _ = time_chain(torch, chain, stream, d_ts, pitch, nch, nfr, d_out, steps)
        frames = nch * nfr
        v = frames * S / (ms * 1e-3) / 1e6
        ent = {"workload": "%d x %s channels x %d T2 frame(s) per step" % (nch, name, nfr), "value": v, "unit": UNIT,
               "ms_per_step": ms, "x_realtime": v / K.REALTIME_MSPS, "fecframes_per_s": frames * F / (ms * 1e-3),
               "launches_per_step": 4, "roofline": stage_roofline(chain, cfg, frames, st, peak, peak_src)}
        # launch-bound small frames: the same step replayed from a CUDA graph (one graph launch instead of four kernel launches)
        try:
            sp = stream.cuda_stream
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                chain.run_device(d_ts.data_ptr(), pitch, nch, nfr, 0, d_out.data_ptr(), sp)
            for _ in range(3):
                g.replay()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                g.replay()
            e1.record(stream)
            torch.cuda.synchronize()
            gms = e0.elapsed_time(e1) / steps
            ent["cuda_graph"] = {"ms_per_step": gms, "value": frames * S / (gms * 1e-3) / 1e6, "speedup_vs_stream_launches": ms / gms}
            del g
        except Exception as e:      # pragma: no cover
            ent["cuda_graph"] = {"error": str(e)[:200]}
            torch.cuda.synchronize()
        # the reference on ONE host core, bounded to a few seconds
        nf_cpu = {"c1": 40, "c2": 6, "c4": 4}[name]
        r = cpu_reference_run(cfg, 1, nf_cpu, 1)
        if r is not None:
            cv = r["samples"] / r["seconds"] / 1e6
            ent["cpu_reference_1core"] = {"value": cv, "unit": UNIT, "sample": "%d consecutive T2 frames of one channel" % nf_cpu,
                                          "stage_seconds": r["stage_seconds"]}
            ent["gpu_over_1core"] = v / cv
        out[name] = ent
        del chain, d_ts, d_out
    return out


def per_block_device_extras(torch, T, K, dev, stream, peak, peak_src, cfg_name, nframes, steps):
    """The five drop-in blocks' own kernels, device-resident (dvbt2ll_work_device: the items already in HBM in the
    reference's item types -- one byte per bit between the bit blocks, complex64 cells after the mapper), nframes T2 frames
    per call, each block fed by the previous block's output.  Per block: ms per call, the bytes of its input and output
    items over that time, and for the cell-domain stages SURVEY 8(d)'s algorithmic bytes against the measured HBM copy rate."""
    cfg = K.resolve(cfg_name)
    b = T.blocks_for(cfg)
    F = cfg["fecblocks"]
    nfec = nframes * F
    nldpc = 64800 if cfg["framesize"] else 16200
    sp = stream.cuda_stream
    om = {k: v.output_multiple for k, v in b.items()}
    n_out = {"bb": nfec * om["bb"], "ldpc": nfec * om["ldpc"], "im": nfec * om["im"], "fm": nframes * om["fm"], "pg": nframes * om["pg"]}
    n_in = {"bb": None, "ldpc": n_out["bb"], "im": n_out["ldpc"], "fm": n_out["im"], "pg": n_out["fm"]}
    item_in = {"bb": 1, "ldpc": 1, "im": 1, "fm": 8, "pg": 8}
    item_out = {"bb": 1, "ldpc": 1, "im": 8, "fm": 8, "pg": 8}
    # TS for the BB block: one stream; the block carries its packet phase from call to call, so every call is handed the
    # (periodic) stream at the phase it expects: base + consumed % 188, with >= 187 bytes of history in front
    need = b["bb"].forecast(n_out["bb"]) + 2 * 188
    period = K.make_ts(188 * 64)
    reps = (need + 188 + period.size - 1) // period.size + 1
    d_ts = torch.zeros(256 + reps * period.size, dtype=torch.uint8, device=dev)
    d_ts[256:] = torch.from_numpy(period).to(dev).repeat(reps)
    n_in["bb"] = need
    bufs = {"ts": d_ts[256:]}
    for k in ("bb", "ldpc", "im", "fm", "pg"):
        bufs[k] = torch.empty(n_out[k] * item_out[k] + 64, dtype=torch.uint8, device=dev)
    src = {"bb": "ts", "ldpc": "bb", "im": "ldpc", "fm": "im", "pg": "fm"}
    if n_in["fm"] < b["fm"].forecast(n_out["fm"]) or n_in["pg"] < b["pg"].forecast(n_out["pg"]):
        raise RuntimeError("block item counts do not chain")
    out = {"workload": "%d %s T2 frames (%d FECFRAMEs) per call, items resident in HBM, dvbt2ll_work_device" % (nframes, cfg_name, nfec),
           "peak": peak, "peak_source": peak_src, "blocks": {}}
    mapped, stream_items, samples = om["fm"], b["fm"].forecast(om["fm"]), om["pg"]
    alg = {"im": ("mapper: Nldpc/8 packed bits in + 8 B per cell out, per FECFRAME", nfec * (nldpc // 8 + 8 * om["im"])),
           "fm": ("frame mapper (cell + time interleaver, L1, frame, frequency interleaver): 8 B x (stream items + mapped items)", nframes * 8 * (stream_items + mapped)),
           "pg": ("pilots + IFFT + guard interval + P1: 8 B x (mapped items + samples)", nframes * 8 * (b["pg"].forecast(samples) + samples))}
    names = {"bb": "bbheaderbch_bb", "ldpc": "ldpc_bb", "im": "interleavermod_bc", "fm": "framemapperfint_cc", "pg": "pilotgenp1insert_cc"}
    for k in ("bb", "ldpc", "im", "fm", "pg"):
        blk, din, dout = b[k], bufs[src[k]], bufs[k]
        consumed_total = [0]
        def call():
            ofs = consumed_total[0] % 188 if k == "bb" else 0
            r, used = blk.work_device(din.data_ptr() + ofs, n_in[k], dout.data_ptr(), n_out[k], sp)
            consumed_total[0] += used
            if r != n_out[k]:
                raise RuntimeError("%s produced %d of %d items" % (k, r, n_out[k]))
            return used
        used = 0
        for _ in range(3):
            used = call()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            call()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        api_bytes = used * item_in[k] + n_out[k] * item_out[k]
        ent = {"ms_per_call": ms, "item_bytes_in_out": int(api_bytes), "item_gbs": api_bytes / (ms * 1e-3) / 1e9,
               "item_frac_of_peak": api_bytes / (ms * 1e-3) / 1e9 / peak}
        if k in alg:
            ent["algorithmic"] = {"what": alg[k][0], "bytes": int(alg[k][1]), "gbs": alg[k][1] / (ms * 1e-3) / 1e9,
                                  "frac_of_peak": alg[k][1] / (ms * 1e-3) / 1e9 / peak}
        out["blocks"][names[k]] = ent
    del bufs, d_ts, b
    return out


def dropin_extras(torch, T, K, cfg_name, frames_timed):
    """The reference-facing per-block path: one T2 frame per round through the five dvbt2ll_work() handles
    (bbheaderbch -> ldpc -> interleavermod -> framemapper -> pilotgen) on PAGEABLE host buffers -- what a GNU Radio
    scheduler hands to general_work() -- then with the buffers registered on first sight, then with the device-resident
    hand-off between adjacent handles, then with the host copies of the linked edges left out as well."""
    cfg = K.resolve(cfg_name)
    res = {}
    for mode in ("pageable", "host_register", "host_register+link", "host_register+link_lazy_host"):
        b = T.blocks_for(cfg)
        order = [b["bb"], b["ldpc"], b["im"], b["fm"], b["pg"]]
        F = cfg["fecblocks"]
        if mode != "pageable":
            for blk in order:
                blk.set_host_register(True)
        if "link" in mode:
            for i in range(4):
                order[i].link_to(order[i + 1], lazy_host=mode.endswith("lazy_host"))
        nframes = [F, F, F, 1, 1]
        bufs = [np.empty(n * blk.output_multiple, dtype=blk.out_dtype) for blk, n in zip(order, nframes)]
        need0 = b["bb"].forecast(F * b["bb"].output_multiple) + 1024
        ts_all = K.make_ts((frames_timed + 3) * need0, seed=K.TS_SEED)
        ts_buf = np.empty(need0, np.uint8)          # the scheduler's input buffer: fixed address, refilled every round
        pos = 0

        def one_frame():
            nonlocal pos
            ts_buf[:] = ts_all[pos:pos + need0]
            _, used = order[0].work_into(ts_buf, bufs[0], nframes[0])
            pos += used
            for i in range(1, 5):
                order[i].work_into(bufs[i - 1], bufs[i], nframes[i])

        one_frame()
        one_frame()
        t0 = time.perf_counter()
        for _ in range(frames_timed):
            one_frame()
        dt = (time.perf_counter() - t0) / frames_timed
        S = bufs[4].size
        res[mode] = {"value": S / dt / 1e6, "unit": UNIT, "ms_per_t2_frame": dt * 1e3,
                     "link_hits": sum(blk.link_hits for blk in order[1:])}
        nbytes = [ts_buf.nbytes] + [x.nbytes for x in bufs]
        res["h2d_bytes_per_frame"] = int(sum(nbytes[:5]))
        res["d2h_bytes_per_frame"] = int(sum(nbytes[1:]))
        del order, b            # handles first (they unregister), buffers after
        del bufs, ts_buf
    # the same five handles the way GNU Radio's thread-per-block scheduler drives them: one thread per block, every edge a
    # ring of three T2-frame slots at fixed addresses, a block works as soon as it has a frame of input and a free slot
    import threading
    for mode in ("host_register+link", "host_register+link_lazy_host"):
        b = T.blocks_for(cfg)
        order = [b["bb"], b["ldpc"], b["im"], b["fm"], b["pg"]]
        F = cfg["fecblocks"]
        for blk in order:
            blk.set_host_register(True)
        for i in range(4):
            order[i].link_to(order[i + 1], lazy_host=mode.endswith("lazy_host"))
        nframes = [F, F, F, 1, 1]
        SLOTS = 3
        rings = [[np.empty(n * blk.output_multiple, dtype=blk.out_dtype) for _ in range(SLOTS)] for blk, n in zip(order, nframes)]
        need0 = b["bb"].forecast(F * b["bb"].output_multiple) + 1024
        n_run = frames_timed + 2
        ts_all = K.make_ts((n_run + 1) * need0, seed=K.TS_SEED)
        ts_buf = np.empty(need0, np.uint8)
        cv = threading.Condition()
        produced = [0] * 5
        consumed = [0] * 5          # consumed[i]: frames of edge i taken by its reader (edge 4's reader is the sink below)
        errors = []

        def block_thread(i):
            pos = 0
            try:
                for f in range(n_run):
                    with cv:
                        cv.wait_for(lambda: (i == 0 or produced[i - 1] > f) and produced[i] - consumed[i] < SLOTS)
                    if i == 0:
                        ts_buf[:] = ts_all[pos:pos + need0]
                        _, used = order[0].work_into(ts_buf, rings[0][f % SLOTS], nframes[0])
                        pos += used
                    else:
                        order[i].work_into(rings[i - 1][f % SLOTS], rings[i][f % SLOTS], nframes[i])
                    with cv:
                        produced[i] += 1
                        if i > 0:
                            consumed[i - 1] += 1
                        cv.notify_all()
            except Exception as e:          # surface in the main thread
                errors.append(e)
                with cv:
                    produced[i] = 1 << 30
                    cv.notify_all()
        threads = [threading.Thread(target=block_thread, args=(i,)) for i in range(5)]
        for t in threads:
            t.start()
        t_first = None
        for f in range(n_run):              # the sink
            with cv:
                cv.wait_for(lambda: produced[4] > f)
                consumed[4] += 1
                cv.notify_all()
            if f == 1:
                t_first = time.perf_counter()
        dt = (time.perf_counter() - t_first) / (n_run - 2)
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        S = rings[4][0].size
        res[mode + ", thread per block"] = {"value": S / dt / 1e6, "unit": UNIT, "ms_per_t2_frame": dt * 1e3,
                                            "link_hits": sum(blk.link_hits for blk in order[1:]),
                                            "late_host_writes": sum(blk.link_late_writes for blk in order[:4])}
        del order, b
        del rings, ts_buf
    res["api"] = "five dvbt2ll_work() handles, 1 T2 frame (%d FECFRAMEs) per round, %s" % (cfg["fecblocks"], cfg_name)
    return res


STAGE = {"name": "start"}


def stage(name):
    """Where the run is (reported by the watchdog if the run stops making progress)."""
    STAGE["name"] = name


def start_watchdog(seconds, rank, world):
    """A multi-rank run that stops making progress (a lost peer, a device-side wait that is never satisfied) must not hang the
    caller silently: after `seconds` rank 0 prints a line that says where the run was, and every rank exits."""
    if seconds <= 0:
        return

    def fire():
        time.sleep(seconds)
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": 0.0, "unit": UNIT, "n_gpus": world, "higher_is_better": True,
                              "error": "bench.py: no result after %d s; the run was in stage '%s' -- value 0 = not measured" % (seconds, STAGE["name"])}))
            sys.stdout.flush()
        os._exit(4)
    threading.Thread(target=fire, daemon=True).start()


def run_ours(args):
    import torch
    import torch.distributed as dist
    import dvbt2ll_b200 as T
    from dvbt2ll_b200 import configs as K
    from dvbt2ll_b200 import shard

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    start_watchdog(args.deadline if args.deadline >= 0 else (420 if world > 1 else 1500), rank, world)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        stage("process group init")
        dist.init_process_group("nccl", device_id=dev)
    stage("plan + synthetic TS")

    cfg = K.resolve(args.config)
    nfr = args.frames
    my_ch = shard.channels_for_rank(args.channels, world, rank)          # config 5 as stated: 64 / N channels per GPU
    nch = len(my_ch)
    counts = [len(shard.channels_for_rank(args.channels, world, r)) for r in range(world)]
    frames = nch * nfr
    weak_nch = args.channels                                             # extra: the same 64 channels on EVERY GPU
    chain = T.Chain(cfg, max_frames=max(frames, weak_nch * nfr if world > 1 else 0, 1), device=local)
    n_ts, S, F = chain.ts_bytes_per_frame, chain.samples_per_frame, chain.fecframes_per_frame
    pitch = (nfr * n_ts + 255) // 256 * 256

    # synthetic TS: one independent stream per channel (seed + global channel index), pinned on the host
    ts_host = torch.empty((max(nch, 1), pitch), dtype=torch.uint8).pin_memory()
    ts_np = ts_host.numpy()
    for i, c in enumerate(my_ch):
        ts_np[i, :nfr * n_ts] = K.make_ts(nfr * n_ts, seed=K.TS_SEED + c)
    d_ts = ts_host.to(dev)
    d_out = torch.empty((max(nch, 1), nfr * S), dtype=torch.complex64, device=dev)
    # a dedicated (non-default) stream: its handle is what the C ABI launches on and what the CUDA events time
    stream = torch.cuda.Stream(device=dev)
    consumer = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    assert sp != 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    stage("parity check against the checker")
    # ---- untimed: every rank checks one of its OWN channels (its last) against the checker
    parity = {"ok": None}
    if not args.no_parity and nch > 0:
        chain.run_device(d_ts.data_ptr(), pitch, nch, nfr, 0, d_out.data_ptr(), sp)
        torch.cuda.synchronize()
        got = d_out[nch - 1, :S].cpu().numpy()
        want, src = reference_frame(cfg, ts_np[nch - 1, :nfr * n_ts])
        m = mer_db(got, want)
        parity = {"ok": bool(m >= 90.0), "mer_db": m, "channel": my_ch[-1], "checker": src}
        if not parity["ok"]:
            raise SystemExit("bench.py: rank %d channel %d differs from %s (MER %.1f dB)" % (rank, my_ch[-1], src, m))
    parity_ok_ranks = 1 if parity["ok"] else 0
    if world > 1:
        t = torch.tensor([parity_ok_ranks], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        parity_ok_ranks = int(t.item())

    # ---- ordered reassembly on GPU 0 (N > 1): the library's gather, connected once
    G = None
    part_bytes = nfr * S * 8
    offs, sizes, slot_bytes = shard.slot_layout(counts, part_bytes)
    if world > 1:
        stage("reassembly: connect")
        G = T.Gather(rank, world, 0, local, slot_bytes, sizes[rank], n_slots=2)
        blobs = [None] * world
        dist.all_gather_object(blobs, G.export())
        G.connect(blobs)
        barrier()

    cp = consumer.cuda_stream
    step_no = [0]

    def gather_step(ssz=8):
        """One step with the reassembly: produce in place (root) or locally, push, root waits and releases."""
        k = step_no[0]
        step_no[0] += 1
        off, nb = offs[rank] * ssz // 8, sizes[rank] * ssz // 8
        p = G.acquire(k, off, sp)
        chain.run_device(d_ts.data_ptr(), pitch, nch, nfr, 0, p, sp)
        G.push(k, off, nb, sp)
        if rank == 0:
            slot = G.wait(k, cp)
            G.release(k, cp)
            return slot
        return None

    def plain_step():
        chain.run_device(d_ts.data_ptr(), pitch, nch, nfr, 0, d_out.data_ptr(), sp)

    def timed(step_fn, steps, end_stream):
        """barrier, K steps, end event on `end_stream` (where the rank's last piece of work completes), max over ranks"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            step_fn()
        e1.record(stream if end_stream is None else end_stream)
        barrier()
        return allmax(e0.elapsed_time(e1)) / steps

    # clocks are sampled from before the warm-up until after the timed region (nvidia-smi needs ~0.1 s to
    # start; the timed region itself can be shorter than one sampling period)
    clocks = ClockSampler(local)
    clocks.start()
    chain.enable_timing(False)
    stage("warm-up")
    main_step = gather_step if G is not None else plain_step
    t_w, n_w = time.perf_counter(), 0
    if world == 1:
        while n_w < max(3, args.warmup) or time.perf_counter() - t_w < 0.4:
            main_step()
            n_w += 1
            if n_w % 8 == 0:
                torch.cuda.synchronize()
    else:
        # every rank issues the same steps between two host synchronisations, and the decision to stop is collective
        # (shard.collective_warmup: a time-based loop per rank deadlocked one N = 4 run)
        def any_rank(flag):
            t = torch.tensor([1 if flag else 0], device=dev, dtype=torch.int64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return bool(int(t.item()))
        n_w = shard.collective_warmup(main_step, torch.cuda.synchronize, any_rank, max(3, args.warmup), 0.4)
    barrier()

    # ---- timed region: K steps, CUDA events on the launching streams, max over ranks
    chain.enable_timing(True)
    stage("timed region")
    launches0 = T.kernel_launches()
    if G is None:
        end_stream = None
    else:
        side = torch.cuda.ExternalStream(G.side_stream, device=dev)
        end_stream = consumer if rank == 0 else side
    ms_per_step = timed(main_step, args.steps, end_stream)
    stage_ms = chain.stage_ms()          # per-run CUDA events, read after the timed region
    launches = T.kernel_launches() - launches0
    clk = clocks.stop()
    chain.enable_timing(False)
    # after the clock sampler stops: the copy and the files belong to no timed step
    if args.dump_outputs and rank == 0:
        stage("dump outputs")
        if G is None:
            last = d_out[:nch].cpu().numpy()
        else:                            # the ordered reassembly of every rank's channels in the root's last slot
            torch.cuda.synchronize()
            last = np.empty((args.channels, nfr * S), np.complex64)
            T.copy_to_host(last, G.wait(step_no[0] - 1, cp))
            torch.cuda.synchronize()
        dump_outputs(args.dump_outputs, last)
    total_samples = args.channels * nfr * S
    value = total_samples / (ms_per_step * 1e-3) / 1e6

    # ---- N > 1 extras: the same step without the reassembly, the int16-sink reassembly, weak scaling
    multi = None
    stage("extras after the timed region")
    if G is not None:
        # the gathered slot must be what the ranks produced: the root compares every rank's last channel of the final
        # slot with the checker (untimed)
        gather_ok = None
        if rank == 0 and not args.no_parity:
            torch.cuda.synchronize()
            last_slot = G.wait(step_no[0] - 1, cp)
            torch.cuda.synchronize()
            gather_ok = True
            worst = 1e9
            for r in range(world):
                c = shard.channels_for_rank(args.channels, world, r)[-1]
                host = np.empty(S, np.complex64)
                src_ptr = last_slot + (offs[r] + (counts[r] - 1) * part_bytes)
                T.copy_to_host(host, src_ptr)
                want, _ = reference_frame(cfg, K.make_ts(nfr * n_ts, seed=K.TS_SEED + c))
                m = mer_db(host, want)
                worst = min(worst, m)
                gather_ok = gather_ok and m >= 90.0
            if not gather_ok:
                raise SystemExit("bench.py: reassembled slot differs from the checker (worst MER %.1f dB)" % worst)
        compute_ms = timed(plain_step, args.steps, None)
        # int16 I/Q sink: halves the bytes every rank pushes
        chain.set_sink(1, 0.2)
        for _ in range(3):
            gather_step(4)
        int16_ms = timed(lambda: gather_step(4), args.steps, end_stream)
        chain.set_sink(0, 1.0)
        # weak scaling: 64 channels on every GPU, no reassembly (round-1 headline, kept for continuity)
        stage("extras: weak scaling")
        wts = torch.empty((weak_nch, pitch), dtype=torch.uint8)
        wnp = wts.numpy()
        for c in range(weak_nch):
            wnp[c, :nfr * n_ts] = ts_np[c % max(nch, 1), :nfr * n_ts]
        d_wts = wts.to(dev)
        d_wout = torch.empty((weak_nch, nfr * S), dtype=torch.complex64, device=dev)

        def weak_step():
            chain.run_device(d_wts.data_ptr(), pitch, weak_nch, nfr, 0, d_wout.data_ptr(), sp)
        for _ in range(3):
            weak_step()
        weak_ms = timed(weak_step, args.steps, None)
        del d_wts, d_wout
        # root-weighted shares: GPU 0 computes as many channels itself as it can in the time the others' channels take to
        # arrive over its NVLink ingest (its own channels cost no transfer); the rest is spread over the other GPUs.
        # c1 = one channel's compute time in a full batch (from the 64-channel step above), t_in = its transfer time.
        stage("extras: root-weighted reassembly")
        c1 = weak_ms / weak_nch
        t_in = part_bytes / (NVLINK_PEER_GBS * 1e9) * 1e3
        n_root = max(1, min(args.channels - (world - 1), int(args.channels * t_in / (c1 + t_in) + 0.5)))
        counts_w = [n_root] + [len(shard.channels_for_rank(args.channels - n_root, world - 1, r)) for r in range(world - 1)]
        first_w = sum(counts_w[:rank])
        nw = counts_w[rank]
        wts2 = torch.empty((max(nw, 1), pitch), dtype=torch.uint8)
        for i in range(nw):
            wts2.numpy()[i, :nfr * n_ts] = K.make_ts(nfr * n_ts, seed=K.TS_SEED + first_w + i)
        d_wts2 = wts2.to(dev)
        offs_w, sizes_w, slot_w = shard.slot_layout(counts_w, part_bytes)
        G2 = T.Gather(rank, world, 0, local, slot_w, sizes_w[rank], n_slots=2)
        blobs = [None] * world
        dist.all_gather_object(blobs, G2.export())
        G2.connect(blobs)
        barrier()
        step_w = [0]

        def weighted_step():
            k = step_w[0]
            step_w[0] += 1
            p2 = G2.acquire(k, offs_w[rank], sp)
            chain.run_device(d_wts2.data_ptr(), pitch, nw, nfr, 0, p2, sp)
            G2.push(k, offs_w[rank], sizes_w[rank], sp)
            if rank == 0:
                G2.wait(k, cp)
                G2.release(k, cp)
        for _ in range(3):
            weighted_step()
        end_w = consumer if rank == 0 else torch.cuda.ExternalStream(G2.side_stream, device=dev)
        weighted_ms = timed(weighted_step, args.steps, end_w)
        weighted_ok = None
        if rank == 0 and not args.no_parity:        # the last channel of the last rank, as it sits in the root's slot
            torch.cuda.synchronize()
            slot2 = G2.wait(step_w[0] - 1, cp)
            torch.cuda.synchronize()
            host = np.empty(S, np.complex64)
            T.copy_to_host(host, slot2 + (offs_w[-1] + (counts_w[-1] - 1) * part_bytes))
            want, _ = reference_frame(cfg, K.make_ts(nfr * n_ts, seed=K.TS_SEED + args.channels - 1))
            weighted_ok = bool(mer_db(host, want) >= 90.0)
            if not weighted_ok:
                raise SystemExit("bench.py: root-weighted reassembly differs from the checker")
        barrier()
        G2.close()
        del d_wts2
        into_root_w = slot_w - sizes_w[0]
        into_root = slot_bytes - sizes[0]
        multi = {
            "reassembly": {"api": "dvbt2ll_gather_acquire/push/wait/release (NVLink peer copy per rank on a side stream, 2-slot ring on GPU 0, "
                                  "device-side arrival/release counters)", "in_value": True,
                           "bytes_into_root_per_step": int(into_root), "ingest_gbs_achieved": into_root / (ms_per_step * 1e-3) / 1e9,
                           "ingest_gbs_bound": NVLINK_PEER_GBS, "ingest_bound_source": "B200_PROFILING.md: measured peer copy 770 GB/s per direction per GPU (900 nominal)",
                           "ms_per_step_floor_from_ingest": into_root / (NVLINK_PEER_GBS * 1e9) * 1e3,
                           "gather_parity_ok": gather_ok},
            "compute_only": {"value": total_samples / (compute_ms * 1e-3) / 1e6, "ms_per_step": compute_ms,
                             "note": "same sharded step, every rank keeps its frames (no reassembly)"},
            "reassembly_int16_sink": {"value": total_samples / (int16_ms * 1e-3) / 1e6, "ms_per_step": int16_ms,
                                      "bytes_into_root_per_step": int(into_root // 2),
                                      "ingest_gbs_achieved": (into_root // 2) / (int16_ms * 1e-3) / 1e9},
            "weak": {"value": world * weak_nch * nfr * S / (weak_ms * 1e-3) / 1e6, "ms_per_step": weak_ms,
                     "channels_per_gpu": weak_nch, "note": "64 channels on every GPU, no reassembly (round-1 headline)"},
            "reassembly_root_weighted": {"value": total_samples / (weighted_ms * 1e-3) / 1e6, "ms_per_step": weighted_ms,
                                         "channels_per_gpu": counts_w, "bytes_into_root_per_step": int(into_root_w),
                                         "ingest_gbs_achieved": into_root_w / (weighted_ms * 1e-3) / 1e9, "gather_parity_ok": weighted_ok,
                                         "note": "same 64 channels and the same ordered reassembly, but GPU 0 takes the share it can compute "
                                                 "while the other GPUs' channels arrive (its own cost no transfer): root compute time = "
                                                 "root ingest time; not the headline, which keeps 64 / N channels per GPU"},
            "limiter": "one GPU's NVLink ingest: all but 1/N of every step's samples must enter GPU 0",
        }

    stage("e2e through host buffers")
    # ---- e2e: HOST TS in, HOST samples out through the C ABI (pinned buffers), copies inside the timed region
    out_host = torch.empty((max(nch, 1), nfr * S), dtype=torch.complex64).pin_memory()
    out_np = out_host.numpy()
    chain.run_host(ts_np, nch, nfr, 0, out=out_np)      # warm-up (allocates staging)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        chain.run_host(ts_np, nch, nfr, 0, out=out_np)
    torch.cuda.synchronize()
    e2e_s = allmax((time.perf_counter() - t0) / args.e2e_steps)
    e2e_value = total_samples / e2e_s / 1e6
    checksum = float(np.abs(out_np[0, :4096]).sum())

    # ---- extra (SURVEY 8(f) item 3): the flowgraph's sink side folded into the last kernel -- x0.2 gain and
    # 16-bit I/Q output, which halves the device-to-host bytes.  Reported beside e2e, not instead of it.
    out16_host = torch.empty((max(nch, 1), nfr * S, 2), dtype=torch.int16).pin_memory()
    out16_np = out16_host.numpy()
    chain.set_sink(1, 0.2)
    chain.run_host(ts_np, nch, nfr, 0, out=out16_np)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        chain.run_host(ts_np, nch, nfr, 0, out=out16_np)
    torch.cuda.synchronize()
    e2e16_s = allmax((time.perf_counter() - t0) / args.e2e_steps)
    chain.set_sink(0, 1.0)
    e2e16_value = total_samples / e2e16_s / 1e6

    # ---- the box's device->host ceiling: every GPU copies 1 GB to pinned host memory at the same time, no kernels
    probe_bytes = 1 << 30
    d_probe = torch.empty(probe_bytes, dtype=torch.uint8, device=dev)
    h_probe = torch.empty(probe_bytes, dtype=torch.uint8).pin_memory()
    h_probe.copy_(d_probe, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        h_probe.copy_(d_probe, non_blocking=True)
    torch.cuda.synchronize()
    probe_s = allmax((time.perf_counter() - t0) / 3)
    pcie_ceiling = world * probe_bytes / probe_s / 1e9
    del d_probe, h_probe
    e2e_d2h = args.channels * nfr * S * 8
    e2e_gbs = (e2e_d2h + args.channels * nfr * n_ts) / e2e_s / 1e9

    if rank != 0:
        if G is not None:
            G.close()           # peers unmap the root's ring before the root frees it
            barrier()
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f)["hbm_gbs"]); peak_src = "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        pass
    roofline = stage_roofline(chain, cfg, frames, stage_ms, peak, peak_src)
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "ofdm_traffic.json")) as f:
            tj = json.load(f)
            # measured once under `ncu --set full` for 64 T2 frames per launch; scaled to this launch's frame count
            traffic = tj.get("dram_bytes_per_launch") * frames / float(tj.get("frames_per_launch", 64))
            traffic_src = "profiles/ofdm_traffic.json (static: one ncu --set full capture, not measured in this run)"
    except Exception:
        pass
    roofline["traffic"] = traffic
    roofline["traffic_source"] = traffic_src

    extras = {}
    stage("N = 1 extras / cpu baseline")
    if world == 1 and not args.no_extras:
        try:
            extras["dropin_e2e"] = dropin_extras(torch, T, K, args.config, 8)
        except Exception as e:      # pragma: no cover  (an extra must never cost the headline line)
            extras["dropin_e2e"] = {"error": str(e)[:300]}
        try:
            extras["per_block_device"] = per_block_device_extras(torch, T, K, dev, stream, peak, peak_src, args.config, 32, max(5, args.steps // 2))
        except Exception as e:      # pragma: no cover
            extras["per_block_device"] = {"error": str(e)[:300]}
            torch.cuda.synchronize()
        try:
            extras["per_config"] = per_config_extras(torch, T, K, dev, stream, peak, peak_src, max(5, args.steps // 2))
        except Exception as e:      # pragma: no cover
            extras["per_config"] = {"error": str(e)[:300]}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(cfg, 1, args.cpu_frames, 1)
        if r is not None:
            v = r["samples"] / r["seconds"] / 1e6
            fft_share = r["stage_seconds"].get("fft", 0.0) / max(1e-9, sum(x for k, x in r["stage_seconds"].items() if k != "fft"))
            cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "reference",
                   "fft_share_of_cpu_time": fft_share, "value_without_fft": v / (1 - fft_share) if fft_share < 1 else None,
                   "sample": "%d consecutive T2 frames of one %s channel on %s, unmodified reference sources via oracle/_ref "
                             "(GNU Radio shim, single-precision radix-4 FFT stand-in for FFTW), one frame per general_work call; "
                             "stage CPU-seconds %s" % (r["frames"], args.config, cpu_model(), json.dumps(r["stage_seconds"]))}

    cell_size = (64800 if cfg["framesize"] else 16200) // (2 * (cfg["constellation"] + 1))
    conf = config_dict(args, S, F)
    conf.update({"channels_per_gpu": counts, "l2": "working set per step per GPU (%.0f MB 16-bit cells + %.0f MB samples) %s the 126 MB L2; no explicit flush" % (
        frames * F * cell_size * 2 / 1e6, frames * S * 8 / 1e6, "exceeds" if frames * S * 8 > 126e6 else "is below")})
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": n_w,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8/f32", "data": "synthetic", "config": conf,
        "x_realtime": value / K.REALTIME_MSPS, "x_realtime_per_gpu": value / K.REALTIME_MSPS / world,
        "fecframes_per_s": args.channels * nfr * F / (ms_per_step * 1e-3),
        "parity_ok_ranks": parity_ok_ranks, "parity": parity,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(args.channels * nfr * n_ts), "d2h_bytes_per_step": int(e2e_d2h),
                "api": "dvbt2ll_chain_run_host (pinned host buffers), every rank on its own channels", "checksum": checksum,
                "pcie_gbs_achieved": e2e_gbs, "pcie_ceiling_gbs": pcie_ceiling,
                "pcie_ceiling_how": "all %d GPU(s) copying 1 GiB device->pinned host concurrently, no kernels (3 copies each, max over ranks)" % world,
                "frac_of_ceiling": e2e_gbs / pcie_ceiling},
        "e2e_int16_sink": {"value": e2e16_value, "unit": UNIT, "d2h_bytes_per_step": int(e2e_d2h // 2),
                           "pcie_gbs_achieved": (e2e_d2h // 2 + args.channels * nfr * n_ts) / e2e16_s / 1e9,
                           "note": "same call with dvbt2ll_chain_set_sink(format=int16 I/Q, gain=0.2): the flowgraph's multiply_const + sc16 conversion fused into the last kernel"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "clocks": clk,
    }
    if multi is not None:
        line["multi_gpu"] = multi
    line.update(extras)
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))
    if G is not None:
        barrier()
        G.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
