#!/usr/bin/env python
"""bench.py — the hot-path benchmark (driver contract: ONE JSON line on rank 0).

    python bench.py --gpus N --steps K --warmup W [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

BASELINE.json's metric is "embeddings/sec and query x gallery pairs/sec, ConvNeXt-B 224^2".  The line's headline (`metric`,
`value`, `e2e`, `roofline`, `cpu_baseline`) is the faceX TRAIN STEP of configs[1] (ConvNeXt-B 224^2 + ArcFace C=1000, per-GPU
batch 128, DDP all-reduce overlapped with the backward); the other legs ride in sub-objects with the same fields:

  train_vit       configs[2]: ViT-B/16 224^2 + CircleLoss train step (secondary)
  extract         embeddings/sec of the CBIR eval path: one batch of 256 synthetic 224^2 images per GPU through
                  TimmWrapper.embed(l2_normalize=True) (= FeatureExtractor.extract_cbir's model(x) + F.normalize,
                  face_model.py:137-139), bf16 activations; N GPUs: independent images, no collective -> weak scaling
  extract_vit     the same with ViT-B/16 (secondary)
  extract_vitl    configs[4]: the same with the CLIP ViT-L/14 tower at 336^2 (timm vit_large_patch14_clip_336), batch 64 per GPU;
                  its retrieval half is the `retrieval` leg (512-d embeddings, gallery sharded over the GPUs)
  retrieval       pairs/sec of configs[3]: one full search, 10 000 queries x 1 000 000 gallery rows, 512-d, cosine top-100
                  (rows_prepare -> tcgen05 score/filter over the gallery ranges -> select -> canonical re-rank); N GPUs:
                  gallery rows sharded, all-gather of queries and of per-shard lists + merge -> strong scaling

`value` is measured with inputs resident in HBM; `e2e` goes through the reference-facing call with HOST buffers (pinned):
train: every step's batch crosses PCIe through visiondk_b200.train.DevicePrefetcher and every step's loss is read back;
extraction: images H2D + embeddings D2H per step (FeatureExtractor.extract_cbir); retrieval: query H2D + (scores, ids) D2H.
`roofline` times the dominant kernel alone with CUDA events (tensor bound, peaks from MEASURED_PEAKS.json; `traffic` = DRAM bytes
per launch from the ncu captures under profiles/).  `cpu_baseline` is the oracle's port of the reference CPU formulation on the
host cores (thread count calibrated, samples bounded); `--impl reference` prints the same line for that CPU port alone.

`--dump-outputs DIR` writes what the last timed step of each leg returned to its caller, as DIR/<name>.npy (float32; ids as
float64): train_loss, train_vit_loss, extract_embeddings, extract_vit_embeddings, extract_vitl_embeddings, retrieval_scores,
retrieval_ids.  Inputs and weights are seeded, so two builds run with the same arguments can be compared file by file.  Above
64 MB in all, every array keeps the same fixed, seeded sample of its rows.  bench.py writes nothing else to disk.
Embeddings, scores and ids repeat bit for bit from run to run.  The train losses do not: the weight-gradient reductions add
with float atomics, and after the default 3 warm-up + 20 timed steps two runs differ by up to about 1e-2 relative (6e-3 seen
for train_vit_loss over three runs on one B200, 1000 W power limit).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NQ, NG, DIM, K = 10000, 1000000, 512, 100
MODEL, IMG, FEAT, BATCH = "convnext_base", 224, 512, 256
GFLOP_PER_EMBEDDING = 30.76  # SURVEY.md §8(d)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--nq", type=int, default=NQ)
    ap.add_argument("--ng", type=int, default=NG)
    ap.add_argument("--k", type=int, default=K)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity check of the retrieval leg")
    ap.add_argument("--train-batch", type=int, default=128)
    ap.add_argument("--only", default="all", choices=["all", "both", "train", "extract", "retrieval"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of each leg returned as DIR/<name>.npy (at most 64 MB in all)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------------
# clocks during the timed region: one persistent nvidia-smi -lms process, parsed afterwards
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line)

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = [[c.strip() for c in l.split(",")] for l in self.lines if l.strip()]
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[j] for r in rows for j in range(4) if len(r) > 2 + j and r[2 + j] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------
# CPU legs (oracle port of the reference formulation; the only place bench.py executes oracle/)
# ------------------------------------------------------------------------------------------------------
def cpu_embeddings_pass(model, x):
    import torch
    with torch.no_grad():
        return torch.nn.functional.normalize(model(x))  # face_model.py:137-139


def cpu_retrieval_pass(q, g, k, slice_rows=256):
    """engine/cbir/evaluation.py:190-195: 256-query slices against the whole index, top-k per slice."""
    import torch
    outs = []
    for i in range(0, q.shape[0], slice_rows):
        s = q[i:i + slice_rows] @ g.t()
        outs.append(torch.topk(s, min(k, g.shape[0]), dim=1))
    return outs


def usable_threads():
    """Thread count for the CPU legs.  os.cpu_count() may exceed what the container is allowed to run (CPU quota /
    affinity): 128 threads on a throttled box were measured 10-25x slower than 8 threads on 8 real cores.  So the count
    is calibrated: the candidate (all visible CPUs, then halves down to 8) that runs a fixed fp32 GEMM + conv fastest."""
    import torch
    try:
        visible = len(os.sched_getaffinity(0))
    except AttributeError:
        visible = os.cpu_count() or 1
    cands, c = [], visible
    while c >= 1:
        cands.append(c)
        if c <= 8:
            break
        c //= 2
    a = torch.randn(1536, 1536)
    xconv = torch.randn(4, 256, 28, 28)
    wconv = torch.randn(256, 1, 7, 7)
    best, best_t = cands[-1], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        a @ a
        t0 = time.perf_counter()
        for _ in range(3):
            a @ a
            torch.nn.functional.conv2d(xconv, wconv, padding=3, groups=256)
        dt = time.perf_counter() - t0
        if dt < best_t * 0.95:  # prefer more threads only when they actually help
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_baselines(args, want_retrieval=True, want_train=False, target_s=10.0):
    import torch
    from oracle.convnext import TimmWrapperOracle
    cores = usable_threads()
    out = {}
    model = TimmWrapperOracle(MODEL, FEAT, IMG).eval()
    x = torch.randn(16, 3, IMG, IMG)
    cpu_embeddings_pass(model, x[:4])
    t0 = time.perf_counter()
    n = 0
    while True:
        cpu_embeddings_pass(model, x)
        n += 16
        if time.perf_counter() - t0 > target_s or n >= 512:
            break
    dt = time.perf_counter() - t0
    out["embeddings"] = {"value": n / dt, "unit": "embeddings/s", "cores": cores, "kind": "port",
                         "sample": f"{n} images (bs 16, fp32 oracle ConvNeXt-B 224 + F.normalize), {dt:.1f} s"}
    if want_train:
        from oracle import heads as H
        model.train()
        head_w = torch.nn.Parameter(H.init_head_weight(FEAT, 1000))
        opt = torch.optim.SGD(list(model.parameters()) + [head_w], lr=0.01, momentum=0.937, weight_decay=5e-4)
        xt, yt = torch.randn(16, 3, IMG, IMG), torch.randint(0, 1000, (16,))

        def tstep():
            loss = H.cross_entropy(H.arcface_logits(model(xt), head_w, yt, 0.35, 0.0, 32.0), yt, 0.1)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(list(model.parameters()) + [head_w], 10.0)
            opt.step()
            opt.zero_grad()

        tstep()  # warm-up (allocator, thread pool)
        t0 = time.perf_counter()
        reps, per = 0, []
        while True:
            t1 = time.perf_counter()
            tstep()
            per.append(time.perf_counter() - t1)
            reps += 1
            if time.perf_counter() - t0 > 2 * target_s or reps >= 8:
                break
        dt = time.perf_counter() - t0
        out["train"] = {"value": reps * 16 / dt, "unit": "embeddings/s", "cores": cores, "kind": "port",
                        "spread": {"min": 16 / max(per), "max": 16 / min(per), "unit": "embeddings/s per step"},
                        "sample": f"{reps} train steps of 16 images (fp32 oracle fwd + ArcFace/CE + bwd + clip + SGD), {dt:.1f} s"}
        model.eval()
    if want_retrieval:
        gen = torch.Generator().manual_seed(5)
        g = torch.nn.functional.normalize(torch.randn(args.ng, DIM, generator=gen))
        q = torch.nn.functional.normalize(torch.randn(256, DIM, generator=gen))
        cpu_retrieval_pass(q[:64], g, args.k)
        t0 = time.perf_counter()
        reps = 0
        while True:
            cpu_retrieval_pass(q, g, args.k)
            reps += 1
            if time.perf_counter() - t0 > target_s or reps >= 40:
                break
        dt = time.perf_counter() - t0
        out["retrieval"] = {"value": reps * 256 * args.ng / dt, "unit": "pairs/s", "cores": cores, "kind": "port",
                            "sample": f"{reps} x (256 queries x {args.ng} gallery x {DIM}-d fp32, q@g.T + top-{args.k}), {dt:.1f} s"}
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU formulation on the host cores (oracle port; timm/faiss cannot be
    installed here, DESIGN.md §2).  Primary metric = the faceX train step (fwd + CE + bwd + clip + SGD + EMA of the fp32
    oracle, engine/procedure/train.py:196-215); one step = a bounded sample of 2 images so that K steps stay within minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import copy
    import torch
    from oracle.convnext import TimmWrapperOracle
    from oracle import heads as H
    cores = usable_threads()
    bs = 16  # a bounded sample of the 128-image step: ~3 s per step on the box's host cores, K = 20 steps stay within minutes
    backbone = TimmWrapperOracle(MODEL, FEAT, IMG).train()
    head_w = torch.nn.Parameter(H.init_head_weight(FEAT, 1000))
    params = list(backbone.parameters()) + [head_w]
    opt = torch.optim.SGD([{"params": list(backbone.parameters()), "lr": 0.01}, {"params": [head_w], "lr": 0.1}], lr=0.01,
                          momentum=0.937, weight_decay=5e-4)
    ema = copy.deepcopy(backbone).eval()
    x = torch.randn(bs, 3, IMG, IMG)
    y = torch.randint(0, 1000, (bs,))

    def step():
        logits = H.arcface_logits(backbone(x), head_w, y, 0.35, 0.0, 32.0)
        loss = H.cross_entropy(logits, y, 0.1)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 10.0)
        opt.step()
        opt.zero_grad()
        with torch.no_grad():
            for e, p in zip(ema.state_dict().values(), backbone.state_dict().values()):
                if e.dtype.is_floating_point:
                    e.mul_(0.999).add_(p.detach(), alpha=0.001)
        return float(loss)

    for _ in range(max(1, min(args.warmup, 2))):
        step()
    per_step = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        t1 = time.perf_counter()
        step()
        per_step.append(time.perf_counter() - t1)
    dt = time.perf_counter() - t0
    value = args.steps * bs / dt
    srt = sorted(per_step)
    spread = {"min": bs / srt[-1], "median": bs / srt[len(srt) // 2], "max": bs / srt[0], "unit": "embeddings/s per step"}
    # secondary: inference embeddings and retrieval, bounded samples
    backbone.eval()
    xe = torch.randn(8, 3, IMG, IMG)
    cpu_embeddings_pass(backbone, xe[:2])
    t0 = time.perf_counter()
    cpu_embeddings_pass(backbone, xe)
    evalue = 8 / (time.perf_counter() - t0)
    gen = torch.Generator().manual_seed(5)
    g = torch.nn.functional.normalize(torch.randn(args.ng, DIM, generator=gen))
    q = torch.nn.functional.normalize(torch.randn(256, DIM, generator=gen))
    cpu_retrieval_pass(q[:32], g, args.k)
    t0 = time.perf_counter()
    reps = 2
    for _ in range(reps):
        cpu_retrieval_pass(q, g, args.k)
    rvalue = reps * 256 * args.ng / (time.perf_counter() - t0)
    zero = {"h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    line = {
        "impl": "reference", "metric": "embeddings/sec (ConvNeXt-B 224^2 faceX ArcFace train step)", "value": value,
        "unit": "embeddings/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "faceX train step: ConvNeXt-B 224^2 + ArcFace(C=1000) + CE + clip + SGD + EMA",
                   "note": f"reference CPU path restated (fp32 oracle + torch.optim.SGD); each step = a bounded sample of {bs} images"},
        "cpu_baseline": {"value": value, "unit": "embeddings/s", "cores": cores, "kind": "port", "spread": spread,
                         "sample": f"each step = {bs} images through fwd + ArcFace/CE + bwd + clip + SGD + EMA (fp32 oracle)"},
        "e2e": dict(value=value, unit="embeddings/s", **zero), "gpu_launches": 0,
        "extract": {"metric": "embeddings/sec (ConvNeXt-B 224^2, CBIR extract, inference)", "value": evalue,
                    "unit": "embeddings/s", "cpu_baseline": {"value": evalue, "unit": "embeddings/s", "cores": cores,
                                                             "kind": "port", "sample": "8 images, bs 8, fp32 oracle"},
                    "e2e": dict(value=evalue, unit="embeddings/s", **zero)},
        "retrieval": {"metric": "query x gallery pairs/sec (cosine top-100, 512-d)", "value": rvalue, "unit": "pairs/s",
                      "cpu_baseline": {"value": rvalue, "unit": "pairs/s", "cores": cores, "kind": "port",
                                       "sample": f"{reps} x (256 queries x {args.ng} gallery, q@g.T + top-{args.k})"},
                      "e2e": dict(value=rvalue, unit="pairs/s", **zero)},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------
# GPU legs
# ------------------------------------------------------------------------------------------------------
class Ctx:
    pass


def timed(ctx, fn, steps, warmup):
    """W warm-up calls, then K calls bracketed by barrier + synchronize; CUDA events; max over ranks.
    Returns the ms per call and what the last call returned."""
    import torch
    import torch.distributed as dist
    for _ in range(max(3, warmup)):
        fn()
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = None
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    ctx.barrier()
    ms = e0.elapsed_time(e1)
    if ctx.world > 1:
        t = torch.tensor([ms], device=ctx.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms / steps, out


MAX_DUMP_BYTES = 60 * 10**6  # array data; with the .npy headers the files stay under 64 MB however it is counted


def keep_outputs(ctx, args, **tensors):
    """--dump-outputs: host copies of what a leg's last timed step returned, taken right after its timed loop (the untimed
    calls that follow may reuse the same buffers)."""
    if args.dump_outputs:
        ctx.outputs.update({name: t.detach().cpu() for name, t in tensors.items()})


def dump_outputs(outputs, out_dir):
    """DIR/<name>.npy in float32 (float64 kept; integers as float64, exact below 2**53).  Above MAX_DUMP_BYTES in all, every
    array keeps the same fraction of its rows, chosen by a fixed seed, so a given set of arguments always dumps the same rows."""
    import numpy as np
    import torch
    arrays = {}
    for name, t in outputs.items():
        dt = torch.float64 if t.dtype == torch.float64 or not t.is_floating_point() else torch.float32
        arrays[name] = t.to(dt).numpy()
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if total > MAX_DUMP_BYTES and a.ndim > 0:
            keep = max(1, a.shape[0] * MAX_DUMP_BYTES // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def peak_tflops():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["bf16_tflops"]), "MEASURED_PEAKS.json bf16_tflops (burst: kernel timed alone)"
    except Exception:
        return 1590.0, "fallback 1590 TFLOP/s (B200_PROFILING.md)"


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def ncu_traffic(key):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of a kernel / shape from the committed ncu captures:
    profiles/r02_traffic.json maps a key to {"bytes_per_launch": ..., "source": "<csv under profiles/>"}; None when not captured."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        return t.get(key)
    except Exception:
        return None


def live_profile(fn):
    """One extra, UNTIMED call of `fn` with the library's event profile open (vdk_prof_begin / vdk_prof_end): per kernel
    category the launches, the summed CUDA-event time on the launching stream and the algorithmic FLOPs / bytes of that call."""
    import torch
    from visiondk_b200 import _lib
    torch.cuda.synchronize()
    with _lib.profile() as p:
        fn()
        torch.cuda.synchronize()
    return p.totals


def step_roofline(totals, step_ms, what, sustained=True, traffic_key=None):
    """The `roofline` object of a leg from a live profile of ONE of its steps: the dominant kernel class is the tcgen05 GEMM
    (tensor bound); the depthwise / attention classes ride along as `secondary` with their own bounds."""
    pk = measured_peaks()
    if sustained:
        peak, src = float(pk.get("bf16_tflops_sustained", 1422.7)), "MEASURED_PEAKS.json bf16_tflops_sustained (kernels timed inside a long step)"
    else:
        peak, src = float(pk.get("bf16_tflops", 1590.0)), "MEASURED_PEAKS.json bf16_tflops (burst)"
    hbm = float(pk.get("hbm_gbs", 6485.2))
    g = totals["gemm"]
    if g["launches"] == 0:
        return None
    ach = g["flops"] / (g["ms"] * 1e-3) / 1e12
    tr = ncu_traffic(traffic_key) if traffic_key else None
    roof = {"bound": "tensor", "kernel": f"gemm_tn_kernel: every tcgen05 GEMM launch of one {what} (timed live, CUDA events around each launch)",
            "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "peak_source": src,
            "launches": g["launches"], "launch_ms": g["ms"] / g["launches"], "algorithmic_flops_per_launch": g["flops"] / g["launches"],
            "algorithmic_bytes_per_launch": g["bytes"] / g["launches"], "share_of_step": g["ms"] / step_ms,
            "traffic": tr["bytes_per_launch"] if tr else None, "traffic_source": tr["source"] if tr else None, "secondary": {}}
    d = totals["depthwise"]
    if d["launches"]:
        roof["secondary"]["depthwise7x7"] = {
            "bound": "hbm", "kernel": "dwconv7 forward(+LayerNorm) / data-gradient / weight-gradient launches of the step",
            "achieved": d["bytes"] / (d["ms"] * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "frac": d["bytes"] / (d["ms"] * 1e-3) / 1e9 / hbm,
            "fp32_tflops": d["flops"] / (d["ms"] * 1e-3) / 1e12,
            "fp32_peak_note": "FFMA2 measured at 118 FMA/clk/SM = 67 TFLOP/s (tools/ubench_fma.cu): 49 FMA per 4 bytes puts this operator at the FP32 pipe and the HBM roofline at the same time",
            "launches": d["launches"], "share_of_step": d["ms"] / step_ms}
    a = totals["attention"]
    if a["launches"]:
        roof["secondary"]["attention"] = {"bound": "tensor", "achieved": a["flops"] / (a["ms"] * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s",
                                          "frac": a["flops"] / (a["ms"] * 1e-3) / 1e12 / peak, "launches": a["launches"],
                                          "share_of_step": a["ms"] / step_ms}
    return roof


def bench_extract(ctx, args):
    import ctypes as C
    import torch
    from visiondk_b200 import _lib
    from visiondk_b200.backbone import TimmWrapper
    lib = _lib.load()
    B = args.batch
    torch.manual_seed(0)
    model = TimmWrapper(MODEL, FEAT, IMG, pretrained=False).to(ctx.dev).eval()
    # random-init weights of the named architecture; visible layer scale so every block contributes
    with torch.no_grad():
        for n, p in model.named_parameters():
            if n.endswith("gamma"):
                p.fill_(0.1)
    gen = torch.Generator(device=ctx.dev).manual_seed(ctx.rank)
    pool = [torch.randn(B, 3, IMG, IMG, device=ctx.dev, generator=gen) for _ in range(2)]  # 2 x 154 MB > 126 MB L2
    state = {"i": 0}

    def step_dev():
        x = pool[state["i"] & 1]
        state["i"] += 1
        return model.embed(x, l2_normalize=True)

    ms, emb = timed(ctx, step_dev, args.steps, args.warmup)
    keep_outputs(ctx, args, extract_embeddings=emb)
    value = ctx.world * B / (ms * 1e-3)

    # e2e: the reference-facing call FeatureExtractor.extract_cbir(dataloader, device) -> numpy, fed from pinned host
    # batches (what DataLoader(pin_memory=True) yields); every step's images cross PCIe and every step's embeddings
    # come back to the host inside the timed region
    from visiondk_b200.cbir import FeatureExtractor
    host_x = [torch.randn(B, 3, IMG, IMG).pin_memory() for _ in range(2)]
    extractor = FeatureExtractor(model)

    def run_e2e(n_steps):
        loader = (host_x[i & 1] for i in range(n_steps))
        return extractor.extract_cbir(loader, ctx.dev)  # numpy float32 [n_steps*B, FEAT] on the host

    run_e2e(max(3, args.steps))  # warm-up of the same length: the extractor's pinned staging pool reaches its steady size
    ctx.barrier()
    t0 = time.perf_counter()
    out = run_e2e(args.steps)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    assert out.shape == (args.steps * B, FEAT)
    if ctx.world > 1:
        import torch.distributed as dist
        t = torch.tensor([e2e_ms], device=ctx.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())

    roof = None
    if ctx.rank == 0:
        roof = step_roofline(live_profile(step_dev), ms, f"extraction forward (batch {B})", sustained=True, traffic_key=f"extract_gemm_b{B}")
        if roof is not None:
            peak = roof["peak"]
            roof["whole_step"] = {"achieved": B * GFLOP_PER_EMBEDDING / ms, "frac": B * GFLOP_PER_EMBEDDING / ms / peak,
                                  "note": "30.76 GFLOP per embedding over the whole forward"}
    n_blocks = sum(model.model.depths)
    return {"value": value, "ms": ms, "e2e_ms": e2e_ms, "roofline": roof,
            "launches_per_step": 2 + 3 * n_blocks + 6 + 1 + 2,
            "h2d": B * 3 * IMG * IMG * 4, "d2h": B * FEAT * 4, "batch": B}


def bench_extract_vit(ctx, args, name="vit_base_patch16_224", img=IMG, batch=None, title="ViT-B/16", leg="extract_vit"):
    """Secondary row (BASELINE config 5 family): CBIR extraction with a Transformer backbone, ViT-B/16 224^2, random-init
    weights, batch = --batch per GPU.  Device-resident and end-to-end (FeatureExtractor.extract_cbir from pinned host batches)."""
    import torch
    from visiondk_b200.vit import ViTWrapper, VIT_ARCHS
    from visiondk_b200.cbir import FeatureExtractor
    B = batch or args.batch
    IMG_ = img
    torch.manual_seed(0)
    model = ViTWrapper(name, FEAT, IMG_, pretrained=False).to(ctx.dev).eval()
    gen = torch.Generator(device=ctx.dev).manual_seed(ctx.rank)
    pool = [torch.randn(B, 3, IMG_, IMG_, device=ctx.dev, generator=gen) for _ in range(2)]
    state = {"i": 0}

    def step_dev():
        x = pool[state["i"] & 1]
        state["i"] += 1
        return model.embed(x, l2_normalize=True)

    ms, emb = timed(ctx, step_dev, args.steps, args.warmup)
    keep_outputs(ctx, args, **{f"{leg}_embeddings": emb})
    host_x = [torch.randn(B, 3, IMG_, IMG_).pin_memory() for _ in range(2)]
    extractor = FeatureExtractor(model)

    def run_e2e(n_steps):
        return extractor.extract_cbir((host_x[i & 1] for i in range(n_steps)), ctx.dev)

    run_e2e(max(3, args.steps))  # warm-up of the same length: the extractor's pinned staging pool reaches its steady size
    ctx.barrier()
    t0 = time.perf_counter()
    out = run_e2e(args.steps)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    assert out.shape == (args.steps * B, FEAT)
    if ctx.world > 1:
        import torch.distributed as dist
        t = torch.tensor([e2e_ms], device=ctx.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    patch, dim, depth, heads = VIT_ARCHS[name]
    T = (IMG_ // patch) ** 2 + 1
    gflop = (depth * (24.0 * T * dim * dim + 4.0 * T * T * dim) + 2.0 * (T - 1) * 3 * patch * patch * dim + 2.0 * T * dim * FEAT) / 1e9
    peak = float(measured_peaks().get("bf16_tflops_sustained", 1422.7))
    ach = B * gflop / ms
    roof = step_roofline(live_profile(step_dev), ms, f"{title} extraction forward (batch {B})") if ctx.rank == 0 else None
    if roof is None:
        roof = {"bound": "tensor"}
    roof["whole_step"] = {"achieved": ach, "unit": "TFLOP/s", "peak": peak, "frac": ach / peak,
                          "note": f"{gflop:.2f} GFLOP per embedding over the whole forward"}
    return {"metric": f"embeddings/sec ({title} {IMG_}^2, CBIR extract, inference)", "value": ctx.world * B / (ms * 1e-3),
            "unit": "embeddings/s", "ms_per_step": ms, "scaling": "weak", "dtype": "bf16",
            "config": {"workload": f"CBIR eval extract: {title} {IMG_}^2 ({T} tokens, timm {name}) -> {FEAT}-d L2-normalised embeddings, batch {B} "
                                   f"per GPU, random-init weights", "l2": "two alternating input batches, together larger than the 126 MB L2"},
            "e2e": {"value": ctx.world * B / (e2e_ms * 1e-3), "unit": "embeddings/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": B * 3 * IMG_ * IMG_ * 4, "d2h_bytes_per_step": B * FEAT * 4},
            "gpu_launches": (3 + 7 * depth + 4) * args.steps,
            "roofline": roof}


def bench_train(ctx, args):
    """BASELINE configs[1]: ConvNeXt-B 224^2 faceX ArcFace (C=1000) train step, bf16 activations / fp32 master weights,
    per-GPU batch fixed (weak scaling), DDP = one NCCL all-reduce(mean) of the flat gradient buffers per step."""
    import torch
    from visiondk_b200.train import FaceTrainingModel, FaceTrainer
    B = args.train_batch
    torch.manual_seed(0)
    cfg = {"backbone": {f"timm-{MODEL}": {"pretrained": False, "image_size": IMG, "feat_dim": FEAT}},
           "head": {"arcface": {"feat_dim": FEAT, "num_class": 1000, "margin_arc": 0.35, "margin_am": 0.0, "scale": 32}}}
    model = FaceTrainingModel(cfg).to(ctx.dev)
    with torch.no_grad():
        for n, p in model.named_parameters():
            if n.endswith("gamma"):
                p.fill_(0.1)
    trainer = FaceTrainer(model, lr0=0.01, momentum=0.937, weight_decay=5e-4, label_smooth=0.1, layer_wise=True, warm_steps=0,
                          total_steps=100000, use_ema=(ctx.rank == 0))  # EMA on rank 0 only (vision_engine.py:165)
    gen = torch.Generator(device=ctx.dev).manual_seed(100 + ctx.rank)
    pool = [torch.randn(B, 3, IMG, IMG, device=ctx.dev, generator=gen) for _ in range(2)]
    labels = [torch.randint(0, 1000, (B,), device=ctx.dev, generator=gen) for _ in range(2)]
    state = {"i": 0}

    def step_dev():
        i = state["i"] & 1
        state["i"] += 1
        return trainer.step(pool[i], labels[i])

    ms, loss = timed(ctx, step_dev, args.steps, args.warmup)
    keep_outputs(ctx, args, train_loss=loss)
    value = ctx.world * B / (ms * 1e-3)

    host_x = [torch.randn(B, 3, IMG, IMG).pin_memory() for _ in range(2)]
    host_y = [torch.randint(0, 1000, (B,)).pin_memory() for _ in range(2)]

    # end to end: every step's batch comes from pinned host memory (train.py:225) through the library's prefetcher (copy of
    # batch i+1 on a side stream under step i) and every step's loss is read back (train.py:233: loss.item())
    from visiondk_b200.train import DevicePrefetcher
    n_e2e = max(3, args.warmup) + args.steps
    feed = DevicePrefetcher(((host_x[j & 1], host_y[j & 1]) for j in range(n_e2e + 1)), ctx.dev)

    def step_e2e():
        x, y = next(feed)
        loss = trainer.step(x, y)
        return loss.item()

    e2e_ms, _ = timed(ctx, step_e2e, args.steps, args.warmup)
    peak_s = 1422.7
    try:
        peak_s = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
    except Exception:
        pass
    gflop_img = 3 * GFLOP_PER_EMBEDDING  # fwd + dgrad + wgrad (SURVEY.md §8d: 92.3 GFLOP per image)
    ach = B * gflop_img / ms
    nb = sum(model.trainingwrapper["backbone"].model.depths)
    launches = (5 * nb + 6) + (3 * nb + 12) + (14 * nb + 30) + 14 + 8
    roof = None
    if ctx.world == 1:  # the profile needs a step without collectives in flight; N>1 lines carry the whole-step figure only
        roof = step_roofline(live_profile(step_dev), ms, f"train step (batch {B}: forward, dgrad x gelu', weight-gradient slabs, neck, head)",
                             sustained=True, traffic_key=f"train_gemm_b{B}")
    return {"value": value, "ms": ms, "e2e_ms": e2e_ms, "batch": B, "h2d": B * 3 * IMG * IMG * 4 + B * 8, "d2h": 4,
            "launches_per_step": launches, "roofline": roof,
            "whole_step": {"achieved": ach, "unit": "TFLOP/s", "peak": peak_s, "frac": ach / peak_s,
                           "note": "92.3 GFLOP per image (3 x forward) over the whole step incl. head, clip+SGD+EMA; peak = "
                                   "MEASURED_PEAKS.json bf16_tflops_sustained (kernel inside a long step)"}}


def bench_train_vit(ctx, args):
    """Secondary row, BASELINE config 3: ViT-B/16 224^2 + CircleLoss (C=1000) train step, same contract as bench_train."""
    import torch
    from visiondk_b200.train import FaceTrainingModel, FaceTrainer, DevicePrefetcher
    B = args.train_batch
    torch.manual_seed(0)
    cfg = {"backbone": {"timm-vit_base_patch16_224": {"pretrained": False, "image_size": IMG, "feat_dim": FEAT}},
           "head": {"circleloss": {"feat_dim": FEAT, "num_class": 1000, "margin": 0.25, "gamma": 256}}}
    model = FaceTrainingModel(cfg).to(ctx.dev)
    trainer = FaceTrainer(model, lr0=0.01, momentum=0.937, weight_decay=5e-4, label_smooth=0.1, layer_wise=True, warm_steps=0,
                          total_steps=100000, use_ema=(ctx.rank == 0))
    gen = torch.Generator(device=ctx.dev).manual_seed(200 + ctx.rank)
    pool = [torch.randn(B, 3, IMG, IMG, device=ctx.dev, generator=gen) for _ in range(2)]
    labels = [torch.randint(0, 1000, (B,), device=ctx.dev, generator=gen) for _ in range(2)]
    state = {"i": 0}

    def step_dev():
        i = state["i"] & 1
        state["i"] += 1
        return trainer.step(pool[i], labels[i])

    ms, loss = timed(ctx, step_dev, args.steps, args.warmup)
    keep_outputs(ctx, args, train_vit_loss=loss)
    host_x = [torch.randn(B, 3, IMG, IMG).pin_memory() for _ in range(2)]
    host_y = [torch.randint(0, 1000, (B,)).pin_memory() for _ in range(2)]
    n_e2e = max(3, args.warmup) + args.steps
    feed = DevicePrefetcher(((host_x[j & 1], host_y[j & 1]) for j in range(n_e2e + 1)), ctx.dev)

    def step_e2e():
        x, y = next(feed)
        return trainer.step(x, y).item()

    e2e_ms, _ = timed(ctx, step_e2e, args.steps, args.warmup)
    gflop = 3 * 35.28
    peak_s = 1422.7
    try:
        peak_s = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
    except Exception:
        pass
    ach = B * gflop / ms
    roof = step_roofline(live_profile(step_dev), ms, f"ViT-B/16 train step (batch {B})") if ctx.world == 1 else None
    if roof is None:
        roof = {"bound": "tensor"}
    roof["whole_step"] = {"achieved": ach, "unit": "TFLOP/s", "peak": peak_s, "frac": ach / peak_s,
                          "note": "105.8 GFLOP per image (3 x forward) over the whole step"}
    del trainer, model
    return {"metric": "embeddings/sec (ViT-B/16 224^2 faceX CircleLoss train step)", "value": ctx.world * B / (ms * 1e-3),
            "unit": "embeddings/s", "ms_per_step": ms, "scaling": "weak", "dtype": "bf16",
            "config": {"workload": f"faceX train step: ViT-B/16 {IMG}^2 + CircleLoss(C=1000) + CE(label_smooth 0.1) + clip + SGD + EMA, "
                                   f"batch {B} per GPU, DDP all-reduce(mean) over {ctx.world} GPU(s)"},
            "e2e": {"value": ctx.world * B / (e2e_ms * 1e-3), "unit": "embeddings/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": B * 3 * IMG * IMG * 4 + B * 8, "d2h_bytes_per_step": 4},
            "roofline": roof}


def bench_retrieval(ctx, args):
    import ctypes as C
    import torch
    from visiondk_b200 import _lib, sharding
    from visiondk_b200.retrieval import FlatIPIndex, PreparedRows, sharded_flat_search
    lib = _lib.load()
    nq, ng, dim, k = args.nq, args.ng, DIM, args.k
    lo, hi = sharding.shard_bounds(ng, ctx.world, ctx.rank)
    gen = torch.Generator(device=ctx.dev).manual_seed(5)
    chunks = []
    for a in range(0, ng, 125000):  # one generator stream so that shards are slices of the same 1M rows
        b = min(ng, a + 125000)
        blk = torch.nn.functional.normalize(torch.randn(b - a, dim, device=ctx.dev, generator=gen))
        s0, s1 = max(a, lo), min(b, hi)
        if s1 > s0:
            chunks.append(blk[s0 - a:s1 - a].clone())
        del blk
    q_full = torch.nn.functional.normalize(torch.randn(nq, dim, device=ctx.dev, generator=gen))
    index = FlatIPIndex(dim, ctx.dev, normalize=True, id_offset=lo)
    for c in chunks:
        index.add(c)
    del chunks
    index._finalize()
    q_lo, q_hi = sharding.shard_bounds(nq, ctx.world, ctx.rank)
    q_sizes = sharding.shard_sizes(nq, ctx.world)
    q_local = q_full[q_lo:q_hi].contiguous()

    def step_dev():  # device-resident: no host synchronisation inside a search; overflow is checked once after the timed loop
        return sharded_flat_search(index, q_local, q_sizes, k, defer_check=True)

    ms, (s_last, i_last) = timed(ctx, step_dev, args.steps, args.warmup)
    index.check_status(all_ranks=True)  # raises on every rank if any shard overflowed its candidate lists during the loop
    keep_outputs(ctx, args, retrieval_scores=s_last, retrieval_ids=i_last)
    value = nq * ng / (ms * 1e-3)

    # parity check, outside the timed region: 64 sampled query rows of THIS search (single GPU or sharded) against the
    # oracle's exact top-k over the whole gallery, ids and canonical scores bit for bit
    got_s, got_i = step_dev()
    parity = None
    if not args.no_parity:
        sample = torch.arange(0, nq, max(1, nq // 64), device=ctx.dev)[:64]
        if ctx.rank == 0:
            import numpy as np
            from oracle import retrieval as oret  # the checker (never the thing measured)
            gen2 = torch.Generator(device=ctx.dev).manual_seed(5)
            g_host = torch.cat([torch.nn.functional.normalize(torch.randn(min(ng, a + 125000) - a, dim, device=ctx.dev, generator=gen2)).cpu()
                                for a in range(0, ng, 125000)]).numpy()
            t0 = time.perf_counter()
            ref_s, ref_i = oret.flat_ip_search_candidates(oret.l2_normalize(q_full[sample].cpu().numpy()), oret.l2_normalize(g_host), k)
            ids_ok = bool(np.array_equal(got_i[sample].cpu().numpy(), ref_i))
            sc_ok = bool(np.array_equal(got_s[sample].cpu().numpy().view(np.uint32), ref_s.view(np.uint32)))
            parity = {"rows_checked": int(sample.numel()), "ids_bit_exact": ids_ok, "scores_bit_exact": sc_ok,
                      "against": "oracle.retrieval.flat_ip_search_candidates over the full gallery", "path": f"{ctx.world} shard(s)",
                      "oracle_seconds": round(time.perf_counter() - t0, 1)}
            del g_host
            if not (ids_ok and sc_ok):
                raise SystemExit(f"bench.py: retrieval parity check FAILED {parity}")

    q_host = torch.empty((nq, dim), dtype=torch.float32).pin_memory()
    q_host.copy_(q_full.cpu())
    s_host = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    i_host = torch.empty((nq, k), dtype=torch.int64).pin_memory()

    def step_e2e():
        qd = q_host[q_lo:q_hi].to(ctx.dev, non_blocking=True)
        s, i = sharded_flat_search(index, qd, q_sizes, k)
        if ctx.rank == 0:
            s_host.copy_(s, non_blocking=True)
            i_host.copy_(i, non_blocking=True)
        torch.cuda.synchronize()

    e2e_ms, _ = timed(ctx, step_e2e, args.steps, args.warmup)

    roof = None
    ngl = hi - lo
    plan = index.last_plan  # the plan of the timed searches (sharded: the common range schedule of all shards)
    ends = sorted({min(int(plan.stage_end[j]), ngl) for j in range(plan.n_stages)})  # padded (empty) trailing ranges collapse
    if ctx.rank == 0:
        qp = PreparedRows(q_full, True)
        r_lo = ends[-2] if len(ends) > 1 else 0
        dense = 1 if len(ends) == 1 else 0
        ws = index._ws  # thresholds of the last search are still in the workspace

        def score_only():
            _lib.check(lib.vdk_score_range(C.byref(plan), qp.xh.data_ptr(), index._rows.xh.data_ptr(), r_lo, ngl, dense,
                                           ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "vdk_score_range")

        score_only()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record()
        for _ in range(reps):
            score_only()
        e1.record()
        torch.cuda.synchronize()
        k_ms = e0.elapsed_time(e1) / reps
        flops = 2.0 * dim * nq * (ngl - r_lo)
        peak, src = peak_tflops()
        ach = flops / (k_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "score_filter_kernel<sparse> over the last gallery range", "rows": [int(r_lo), int(ngl)], "achieved": ach,
                "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "traffic": (ncu_traffic(f"retrieval_last_range_nq{nq}_ng{ng}_w{ctx.world}") or {}).get("bytes_per_launch"),
                "traffic_unit": "bytes/launch (profiles/r02_traffic.json)",
                "peak_source": src, "launch_ms": k_ms,
                "algorithmic_flops_per_launch": flops, "share_of_step": k_ms / ms,
                "whole_step": {"achieved": 2.0 * dim * nq * ngl / (ms * 1e-3) / 1e12,
                               "frac": 2.0 * dim * nq * ngl / (ms * 1e-3) / 1e12 / peak,
                               "note": "2*D FLOP per pair over the whole search (all ranges, select, re-rank)"}}
    # rows_prepare + eps; per range: score_filter + select (+ tighten, rank sketch, bound when sharded); re-rank (+ pack, merge)
    launches = 2 + len(ends) * (2 if ctx.world == 1 else 5) + 1 + (2 if ctx.world > 1 else 0)
    return {"value": value, "ms": ms, "e2e_ms": e2e_ms, "roofline": roof, "launches_per_step": launches, "parity_check": parity,
            "h2d": nq * dim * 4, "d2h": nq * k * 12}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from visiondk_b200 import _lib

    ctx = Ctx()
    ctx.outputs = {}
    ctx.world = int(os.environ.get("WORLD_SIZE", "1"))
    ctx.rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the hot path")
    torch.cuda.set_device(local_rank)
    ctx.dev = torch.device("cuda", local_rank)
    if ctx.world > 1:
        dist.init_process_group("nccl", device_id=ctx.dev)
    _lib.load()  # the library build() left in the tree; bench.py compiles nothing, so the tree may be read-only
    _lib.require_device()

    def barrier():
        if ctx.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx.barrier = barrier

    sampler = ClockSampler(local_rank) if ctx.rank == 0 else None
    if sampler:
        sampler.start()
    want = lambda name: args.only in ("all", name) or (args.only == "both" and name in ("extract", "retrieval"))
    tr = bench_train(ctx, args) if want("train") else None
    torch.cuda.empty_cache()
    trv = bench_train_vit(ctx, args) if want("train") else None
    torch.cuda.empty_cache()
    ex = bench_extract(ctx, args) if want("extract") else None
    torch.cuda.empty_cache()
    exv = bench_extract_vit(ctx, args) if want("extract") else None
    torch.cuda.empty_cache()
    # BASELINE configs[4]: the CLIP ViT-L/14 tower at 336^2 (timm vit_large_patch14_clip_336: 577 tokens, width 1024, 24 blocks)
    exl = bench_extract_vit(ctx, args, name="vit_large_patch14_clip_336", img=336, batch=max(8, args.batch // 4),
                            title="ViT-L/14 (CLIP tower)", leg="extract_vitl") if want("extract") else None
    torch.cuda.empty_cache()
    rt = bench_retrieval(ctx, args) if want("retrieval") else None
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(ctx.outputs, args.dump_outputs)

    cpu = {}
    if ctx.rank == 0 and ctx.world == 1 and not args.no_cpu_baseline and (ex is not None or tr is not None):
        cpu = cpu_baselines(args, want_retrieval=rt is not None, want_train=tr is not None)

    if ctx.rank == 0:
        W = max(3, args.warmup)
        retrieval = extract = None
        if rt is not None:
            retrieval = {
                "metric": "query x gallery pairs/sec (cosine top-100, 512-d)", "value": rt["value"], "unit": "pairs/s",
                "ms_per_step": rt["ms"], "scaling": "strong", "dtype": "f16 candidates + f64 canonical re-rank",
                "config": {"workload": f"{args.nq} queries x {args.ng} gallery x {DIM}-d, cosine top-{args.k}, gallery "
                                       f"sharded by rows over {ctx.world} GPU(s)",
                           "l2": "gallery (fp16 1.0 GB + fp32 2.0 GB per 1M rows) exceeds the 126 MB L2; no flush needed",
                           "exactness": "see parity_check: sampled rows of this very search vs the oracle, bit for bit"},
                "parity_check": rt["parity_check"],
                "e2e": {"value": args.nq * args.ng / (rt["e2e_ms"] * 1e-3), "unit": "pairs/s", "ms_per_step": rt["e2e_ms"],
                        "h2d_bytes_per_step": rt["h2d"], "d2h_bytes_per_step": rt["d2h"]},
                "gpu_launches": rt["launches_per_step"] * args.steps,
                "roofline": rt["roofline"], "cpu_baseline": cpu.get("retrieval"),
            }
        if ex is not None:
            extract = {
                "metric": "embeddings/sec (ConvNeXt-B 224^2, CBIR extract, inference)", "value": ex["value"],
                "unit": "embeddings/s", "ms_per_step": ex["ms"], "scaling": "weak", "dtype": "bf16",
                "config": {"workload": f"CBIR eval extract: ConvNeXt-B {IMG}^2 -> {FEAT}-d L2-normalised embeddings, "
                                       f"batch {ex['batch']} per GPU, random-init weights",
                           "l2": "two alternating input batches (2 x 154 MB) exceed the 126 MB L2"},
                "e2e": {"value": ctx.world * ex["batch"] / (ex["e2e_ms"] * 1e-3), "unit": "embeddings/s",
                        "ms_per_step": ex["e2e_ms"], "h2d_bytes_per_step": ex["h2d"], "d2h_bytes_per_step": ex["d2h"]},
                "gpu_launches": ex["launches_per_step"] * args.steps,
                "roofline": ex["roofline"], "cpu_baseline": cpu.get("embeddings"),
            }
        common = {"n_gpus": ctx.world, "steps": args.steps, "warmup": W, "higher_is_better": True, "vs_baseline": None,
                  "data": "synthetic", "clocks": clocks}
        if tr is not None:
            roof = tr.get("roofline")
            if roof is not None:
                roof["whole_step"] = tr["whole_step"]
            line = {
                "metric": "embeddings/sec (ConvNeXt-B 224^2 faceX ArcFace train step)", "value": tr["value"],
                "unit": "embeddings/s", "ms_per_step": tr["ms"], "scaling": "weak", "dtype": "bf16",
                "config": {"workload": f"faceX train step: ConvNeXt-B {IMG}^2 + ArcFace(C=1000) + CE(label_smooth 0.1) + "
                                       f"clip + SGD + EMA, batch {tr['batch']} per GPU, DDP all-reduce(mean) over {ctx.world} GPU(s)",
                           "l2": "two alternating input batches; saved activations (~93 MB/image) stream through HBM",
                           "other_metrics": "see `extract` (inference embeddings/sec) and `retrieval` (pairs/sec)"},
                "e2e": {"value": ctx.world * tr["batch"] / (tr["e2e_ms"] * 1e-3), "unit": "embeddings/s",
                        "ms_per_step": tr["e2e_ms"], "h2d_bytes_per_step": tr["h2d"], "d2h_bytes_per_step": tr["d2h"]},
                "gpu_launches": tr["launches_per_step"] * args.steps,
                "roofline": roof if roof is not None else {"bound": "tensor", "whole_step": tr["whole_step"]},
                "cpu_baseline": cpu.get("train"),
                "train_vit": trv, "extract": extract, "extract_vit": exv, "extract_vitl": exl, "retrieval": retrieval,
            }
        elif ex is not None:
            line = dict(extract)
            line["extract_vit"] = exv
            line["extract_vitl"] = exl
            line["retrieval"] = retrieval
        else:
            line = dict(retrieval)
        line.update(common)
        print(json.dumps(line), flush=True)
    if ctx.world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
