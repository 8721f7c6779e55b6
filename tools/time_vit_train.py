"""Quick device timing of a ViT + CircleLoss train step (BASELINE config 3 by default; not the bench contract).
argv: batch iters [model image_size], default 128 5 vit_base_patch16_224 224.  After the timed steps one profiled step reports the
attention kernels' share (forward and backward together: the library profile has one attention category)."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from visiondk_b200 import _lib
from visiondk_b200.train import FaceTrainingModel, FaceTrainer
from visiondk_b200.vit import VIT_ARCHS

B = int(sys.argv[1]) if len(sys.argv) > 1 else 128
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 5
name = sys.argv[3] if len(sys.argv) > 3 else "vit_base_patch16_224"
S = int(sys.argv[4]) if len(sys.argv) > 4 else 224
cfg = {"backbone": {f"timm-{name}": {"pretrained": False, "image_size": S, "feat_dim": 512}},
       "head": {"circleloss": {"feat_dim": 512, "num_class": 1000, "margin": 0.25, "gamma": 256}}}
torch.manual_seed(0)
model = FaceTrainingModel(cfg).cuda()
trainer = FaceTrainer(model, lr0=0.01, momentum=0.937, weight_decay=5e-4, label_smooth=0.1, layer_wise=True, warm_steps=0,
                      total_steps=100000, use_ema=True)
x = [torch.randn(B, 3, S, S, device="cuda") for _ in range(2)]
y = [torch.randint(0, 1000, (B,), device="cuda") for _ in range(2)]
for i in range(3):
    loss = trainer.step(x[i & 1], y[i & 1])
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for i in range(iters):
    loss = trainer.step(x[i & 1], y[i & 1])
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / iters
with _lib.profile() as prof:
    trainer.step(x[0], y[0])
    torch.cuda.synchronize()
att = prof.totals["attention"]
# forward GFLOP per image: patch embedding, per block the four Linears (12 C^2 per token) and Q K^T + P V (4 T^2 C), the neck Linear
P, C, depth, _ = VIT_ARCHS[name]
N = (S // P) ** 2
T = N + 1
gflop = (2 * N * 3 * P * P * C + depth * (2 * T * 12 * C * C + 4 * T * T * C) + 2 * T * C * 512) / 1e9
print(json.dumps({"model": f"{name} {S}^2 + CircleLoss(C=1000)", "tokens": T, "batch": B, "ms_per_step": ms, "img_per_s": B / ms * 1e3,
                  "tflops": B * 3 * gflop / ms, "loss": float(loss), "device": torch.cuda.get_device_name(),
                  "profiled_step_attention": {"launches": att["launches"], "ms": att["ms"]}}))
