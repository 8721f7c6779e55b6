"""Device timing of the attention backward: the mma.sync kernel (vdk_attention_bwd, <= 208 tokens) and the tcgen05 pair
(vdk_attention_bwd_tc, any token count).  CUDA events over many launches after warm-up; every shape's working set (qkv, out, d_out,
dqkv) is larger than the 126 MB L2.  At 197 tokens the two kernels alternate launch by launch in one window pair, and their dqkv
are compared on the same inputs.  Prints one JSON line per shape.

    python tools/time_attention_bwd.py [iters]

Algorithmic work is 10 N^2 64 flops per (image, head) (S, dP, dV, dQ, dK); the tcgen05 pair executes 14 N^2 64 (it recomputes S and dP
on the key side instead of accumulating dQ with atomics).
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from visiondk_b200 import _lib

ITERS = int(sys.argv[1]) if len(sys.argv) > 1 else 20


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def inputs(B, N, H):
    torch.manual_seed(0)
    qkv = torch.randn(B, N, 3, H, 64, device="cuda").to(torch.bfloat16)
    dout = torch.randn(B, N, H * 64, device="cuda").to(torch.bfloat16)
    out = torch.empty((B, N, H * 64), dtype=torch.bfloat16, device="cuda")
    lse = torch.empty((B, H, N), dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().vdk_attention_fwd_lse(qkv.data_ptr(), B, N, H, 64, out.data_ptr(), lse.data_ptr(), _lib.stream_ptr()),
               "vdk_attention_fwd_lse")
    return qkv, dout, out, lse


def main():
    lib = _lib.load()
    _lib.require_device()
    dev = card()
    s = _lib.stream_ptr()
    for B, H, N, kernels in [(128, 12, 197, ("mma_sync", "tcgen05")), (128, 12, 785, ("tcgen05",)), (64, 16, 577, ("tcgen05",))]:
        qkv, dout, out, lse = inputs(B, N, H)
        dq = {k: torch.empty_like(qkv) for k in kernels}
        ws_bytes = lib.vdk_attention_bwd_tc_workspace_bytes(B, N, H, 64)
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")

        def run(k):
            if k == "mma_sync":
                rc = lib.vdk_attention_bwd(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), B, N, H, 64, dq[k].data_ptr(), s)
            else:
                rc = lib.vdk_attention_bwd_tc(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), B, N, H, 64, dq[k].data_ptr(),
                                              ws.data_ptr(), ws_bytes, s)
            _lib.check(rc, k)

        for _ in range(3):
            for k in kernels:
                run(k)
        torch.cuda.synchronize()
        ev = {k: [] for k in kernels}
        for _ in range(ITERS):  # alternated launch by launch: both kernels see the same clocks and neighbours
            for k in kernels:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(k)
                e1.record()
                ev[k].append((e0, e1))
        torch.cuda.synchronize()
        alg = 10.0 * B * H * N * N * 64
        res = {"B": B, "H": H, "N": N, "device": dev, "iters": ITERS}
        for k in kernels:
            t = sorted(a.elapsed_time(b) for a, b in ev[k])
            ms = t[len(t) // 2]
            executed = alg * (1.4 if k == "tcgen05" else 1.0)
            res[k] = {"ms_median": round(ms, 4), "ms_min": round(t[0], 4), "ms_max": round(t[-1], 4),
                      "alg_tflops": round(alg / ms / 1e9, 1), "executed_tflops": round(executed / ms / 1e9, 1)}
        if len(kernels) == 2:
            a, b = dq["tcgen05"].float(), dq["mma_sync"].float()
            res["rel_l2_tcgen05_vs_mma_sync"] = {n: ((a[:, :, i] - b[:, :, i]).norm() / b[:, :, i].norm()).item() for i, n in enumerate("qkv")}
            res["max_abs_diff"] = (a - b).abs().max().item()
        print(json.dumps(res), flush=True)
        del qkv, dout, out, lse, dq, ws
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
