#!/usr/bin/env python
"""k_ldpc accumulation scheme per code (run on the GPU box): times the LDPC stage of the fused chain for every T2 code
with a lane per (row, word) [mode 0] and a lane per row [mode 1]; the faster one per code is what
LdpcStage::ldpc_lane_per_row_default encodes.  Output: profiles/r2_ldpc_modes.txt"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "gr-dvbt2ll_b200", "python"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import dvbt2ll_b200 as T  # noqa: E402
from dvbt2ll_b200 import configs as K  # noqa: E402

dev = torch.device("cuda", 0)
stream = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(stream)
NAMES = {K.C1_2: "1/2", K.C3_5: "3/5", K.C2_3: "2/3", K.C3_4: "3/4", K.C4_5: "4/5", K.C5_6: "5/6", K.C1_3: "1/3", K.C2_5: "2/5"}
cases = [("c3", r, 64, 1) for r in (K.C1_2, K.C3_5, K.C2_3, K.C3_4, K.C4_5, K.C5_6)] + \
        [("c1", r, 64, 8) for r in (K.C1_3, K.C2_5, K.C1_2, K.C3_5, K.C2_3, K.C3_4, K.C4_5, K.C5_6)]
print("config rate  q   frames  ldpc_ms(mode0)  ldpc_ms(mode1)")
for base, rate, nch, nfr in cases:
    res = []
    for mode in ("0", "1"):
        os.environ["DVBT2LL_LDPC_MODE"] = mode
        cfg = K.resolve(dict(K.CONFIGS[base], rate=rate))
        ch = T.Chain(cfg, max_frames=nch * nfr, device=0)
        n_ts, S = ch.ts_bytes_per_frame, ch.samples_per_frame
        pitch = (nfr * n_ts + 255) // 256 * 256
        ts = np.zeros((nch, pitch), np.uint8)
        for c in range(nch):
            ts[c, :nfr * n_ts] = K.make_ts(nfr * n_ts, seed=K.TS_SEED + c)
        d_ts = torch.from_numpy(ts).to(dev)
        d_out = torch.empty((nch, nfr * S), dtype=torch.complex64, device=dev)
        for _ in range(5):
            ch.run_device(d_ts.data_ptr(), pitch, nch, nfr, 0, d_out.data_ptr(), stream.cuda_stream)
        torch.cuda.synchronize()
        ch.enable_timing(True)
        for _ in range(30):
            ch.run_device(d_ts.data_ptr(), pitch, nch, nfr, 0, d_out.data_ptr(), stream.cuda_stream)
        torch.cuda.synchronize()
        res.append(ch.stage_ms()["ldpc"])
        q = int(ch.plan("bb.dims", np.int32)[2])
        del ch, d_ts, d_out
    print("%s  %s  %3d  %5d  %.4f  %.4f  %s" % (base, NAMES[rate], q, nch * nfr * cfg["fecblocks"], res[0], res[1], "mode1" if res[1] < res[0] else "mode0"))
