"""Dense appearance cost (north_star kernel 2): M tracks x 30 bank rows x 128 against N detections through the public
call, CUDA events around whole calls with L2 flushed in front of each + max error against a float64 reference.  One
JSON line per shape, each with the device name, power limit and library read in the same run.

usage: python tools/app_cost_bench.py [MxN ...]        (default: 512x512, BASELINE config 4)"""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import alufe_b200
from alufe_b200 import _lib, cost

T, K = 30, 5
shapes = [tuple(int(v) for v in a.lower().split("x")) for a in sys.argv[1:]] or [(512, 512)]
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                   capture_output=True, text=True).stdout.strip().split(",")
info = {"device": torch.cuda.get_device_name(0), "power_limit_w": float(q[1]) if len(q) > 1 else None,
        "lib": os.path.basename(_lib.LIB_PATH)}
flush = torch.empty(64 * 1024 * 1024, device="cuda")
for M, N in shapes:
    tc = M * N >= 64 * 64                       # smaller problems run the float32 FFMA kernel (app_cost_tc.cu)
    g = torch.Generator(device="cuda").manual_seed(0)
    bank = torch.nn.functional.normalize(torch.randn((M, T, 128), device="cuda", generator=g), dim=2)
    det = torch.nn.functional.normalize(torch.randn((N, 128), device="cuda", generator=g), dim=1)
    lens = torch.full((M,), T, dtype=torch.int32, device="cuda")
    for _ in range(3):
        C = cost.app_cost_topk(bank, lens, det, topk=K)
    ts = []
    for _ in range(30):
        flush.zero_()                           # flushes L2; the second pass gives the host a head start, so that the
        flush.zero_()                           # events time the GPU work of the call and not its enqueue
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        C = cost.app_cost_topk(bank, lens, det, topk=K)
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    sims = torch.einsum("mtd,nd->mtn", bank.double(), det.double())
    want = 1.0 - sims.topk(K, dim=1).values.mean(dim=1)
    err = (C.double() - want).abs().max().item()
    us = float(np.median(ts))
    print(json.dumps({"M": M, "N": N, "T": T, "kernel": "tcgen05 bf16x3 split (6 products)" if tc else "float32 FFMA",
                      "us_median": round(us, 2), "us_best": round(min(ts), 2), "max_abs_err_vs_f64": err,
                      "useful_tflops": round(2.0 * M * T * N * 128 / us / 1e6, 2),
                      "bf16_tensor_tflops": round(6 * 2.0 * M * 32 * N * 128 / us / 1e6, 2) if tc else None, **info}),
          flush=True)
