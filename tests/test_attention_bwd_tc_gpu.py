"""GPU parity of the tcgen05 attention backward (csrc/attention_bwd_tc.cu, vdk_attention_bwd_tc) and of ViT training above the
208 tokens the mma.sync backward holds: against fp32 autograd on the same bf16 inputs, and against the fp32 oracle for whole nets."""
import pytest
import torch

from oracle.vit import ViTWrapperOracle, randomize_
from visiondk_b200 import _lib
from visiondk_b200.vit import VIT_ARCHS, ViTWrapper

pytestmark = pytest.mark.gpu

# the toy net above 208 tokens: 128^2 image, patch 8 -> 16^2 + 1 = 257 tokens (3 tiles of 128, the last with one row)
TOY = dict(feat_dim=64, image_size=128, patch=8, dim=128, depth=2, heads=2)
# exact gradient 0: a constant shift in front of a batch-statistics BatchNorm1d is normalised away
VIT_INVARIANT = {"output_layer.2.bias", "output_layer.0.bias"}


def rel(a, b):
    return ((a.float() - b.float()).norm() / (b.float().norm() + 1e-12)).item()


def attention_inputs(B, N, H, seed):
    torch.manual_seed(seed)
    qkv = torch.randn(B, N, 3, H, 64, device="cuda").to(torch.bfloat16)
    dout = torch.randn(B, N, H * 64, device="cuda").to(torch.bfloat16)
    out = torch.empty((B, N, H * 64), dtype=torch.bfloat16, device="cuda")
    lse = torch.empty((B, H, N), dtype=torch.float32, device="cuda")
    _lib.check(_lib.load().vdk_attention_fwd_lse(qkv.data_ptr(), B, N, H, 64, out.data_ptr(), lse.data_ptr(), _lib.stream_ptr()),
               "attention fwd+lse")
    return qkv, dout, out, lse


def backward_tc(lib, qkv, out, dout, lse, dqkv):
    B, N, _, H, _ = qkv.shape
    ws_bytes = lib.vdk_attention_bwd_tc_workspace_bytes(B, N, H, 64)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
    _lib.check(lib.vdk_attention_bwd_tc(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), B, N, H, 64, dqkv.data_ptr(),
                                        ws.data_ptr(), ws_bytes, _lib.stream_ptr()), "vdk_attention_bwd_tc")
    torch.cuda.synchronize()


@pytest.mark.parametrize("B,N,H", [(2, 17, 1), (3, 50, 2), (2, 197, 3), (1, 208, 2), (2, 209, 2), (2, 257, 2), (1, 577, 4),
                                   (1, 785, 2)])
def test_attention_backward_tc_matches_torch_autograd(lib, B, N, H):
    """dqkv against fp32 autograd on the same bf16 inputs (P and dS are rounded to bf16 inside the kernels, as in the mma.sync kernel:
    rel L2 <= 2e-2 per operand).  dqkv is followed by one image of NaN sentinel that must survive: rows >= N are never written."""
    qkv, dout, out, lse = attention_inputs(B, N, H, seed=N + H)
    buf = torch.full((B + 1, N, 3, H, 64), float("nan"), dtype=torch.bfloat16, device="cuda")
    backward_tc(lib, qkv, out, dout, lse, buf)
    dqkv = buf[:B]
    assert torch.isnan(buf[B].float()).all(), "the backward wrote past dqkv"
    x = qkv.float().requires_grad_(True)
    q, k, v = x.permute(2, 0, 3, 1, 4).unbind(0)
    ref = (torch.softmax((q @ k.transpose(-2, -1)) * 0.125, dim=-1) @ v).transpose(1, 2).reshape(B, N, H * 64)
    ref.backward(dout.float())
    assert torch.isfinite(dqkv.float()).all()
    for i, name in enumerate("qkv"):
        assert rel(dqkv[:, :, i], x.grad[:, :, i]) <= 2e-2, (name, rel(dqkv[:, :, i], x.grad[:, :, i]))


def test_attention_backward_tc_same_bits_on_every_call(lib):
    """No atomics: two calls on the same inputs give the same bits."""
    B, N, H = 2, 577, 4
    qkv, dout, out, lse = attention_inputs(B, N, H, seed=11)
    a = torch.full_like(qkv, float("nan"))
    b = torch.full_like(qkv, float("nan"))
    backward_tc(lib, qkv, out, dout, lse, a)
    backward_tc(lib, qkv, out, dout, lse, b)
    assert torch.equal(a.view(torch.int16), b.view(torch.int16))


def test_attention_backward_tc_agrees_with_mma_sync_at_197_tokens(lib):
    """The two backward kernels on one input: both round P and dS to bf16, they differ in summation order only."""
    B, N, H = 2, 197, 3
    qkv, dout, out, lse = attention_inputs(B, N, H, seed=5)
    a = torch.full_like(qkv, float("nan"))
    b = torch.full_like(qkv, float("nan"))
    backward_tc(lib, qkv, out, dout, lse, a)
    _lib.check(lib.vdk_attention_bwd(qkv.data_ptr(), out.data_ptr(), dout.data_ptr(), lse.data_ptr(), B, N, H, 64, b.data_ptr(),
                                     _lib.stream_ptr()), "vdk_attention_bwd")
    torch.cuda.synchronize()
    for i in range(3):
        assert rel(a[:, :, i], b[:, :, i]) <= 1e-2, (i, rel(a[:, :, i], b[:, :, i]))


def test_attention_forward_and_lse_at_785_tokens(lib):
    """The forward at 7 query tiles (ViT-B/8 at 224^2) and the log2-domain log-sum-exp the backward consumes."""
    B, N, H = 2, 785, 3
    qkv, _, out, lse = attention_inputs(B, N, H, seed=3)
    q, k, v = qkv.float().permute(2, 0, 3, 1, 4).unbind(0)
    s = (q @ k.transpose(-2, -1)) * 0.125
    ref = (torch.softmax(s, dim=-1) @ v).transpose(1, 2).reshape(B, N, H * 64)
    assert torch.isfinite(out.float()).all()
    assert (out.float() - ref).abs().max().item() <= 2e-2 * v.abs().max().item()
    assert rel(out, ref) <= 1e-2
    assert (lse - torch.logsumexp(s, dim=-1) * 1.4426950408889634).abs().max().item() <= 2e-2


def build(seed, **kw):
    oracle = randomize_(ViTWrapperOracle("x", **kw), seed=seed)
    ours = ViTWrapper("x", kw["feat_dim"], kw["image_size"], pretrained=False, patch=kw["patch"], dim=kw["dim"], depth=kw["depth"],
                      heads=kw["heads"])
    ours.load_state_dict(oracle.state_dict(), strict=True)
    return oracle, ours.cuda()


def grads_match(ours, oracle, rel_tol, cos_tol, vec_rel_tol=None, vec_cos_tol=None):
    import torch.nn.functional as F
    ref = dict(oracle.named_parameters())
    bad, worst = [], []
    for n, p in ours.named_parameters():
        gr, g = ref[n].grad, p.grad.detach().cpu()
        assert torch.isfinite(g).all(), n
        if n in VIT_INVARIANT or gr.norm() < 1e-7 * (1 + gr.numel() ** 0.5):
            continue
        r = rel(g, gr)
        c = F.cosine_similarity(g.flatten(), gr.flatten(), dim=0).item()
        worst.append((r, c, n))
        rt, ct = (rel_tol, cos_tol) if g.dim() >= 2 else (vec_rel_tol or rel_tol, vec_cos_tol or cos_tol)
        if not (r <= rt and c >= ct):
            bad.append(f"{n}: rel {r:.4f} cos {c:.5f}")
    for r, c, n in sorted(worst, reverse=True)[:8]:
        print(f"  rel {r:.4f} cos {c:.5f} {n}")
    assert not bad, "\n".join(bad[:20])


def test_vit_toy_training_above_208_tokens_matches_oracle_autograd(lib):
    oracle, ours = build(7, **TOY)
    oracle.train()
    ours.train()
    torch.manual_seed(1)
    x = torch.randn(6, 3, 128, 128)
    wout = torch.randn(6, 64)
    out_ref = oracle(x)
    (out_ref * wout).sum().backward()
    out = ours(x.cuda())
    (out * wout.cuda()).sum().backward()
    assert rel(out.detach().cpu(), out_ref.detach()) <= 3e-2
    grads_match(ours, oracle, 6e-2, 0.995)


def test_vit_backward_above_208_tokens_in_unit_ranges_equals_single_call(lib):
    _, ours = build(9, **TOY)
    ours.train()
    torch.manual_seed(3)
    x = torch.randn(6, 3, 128, 128, device="cuda")
    wout = torch.randn(6, 64, device="cuda")
    for p in ours.parameters():
        p.grad = torch.zeros_like(p)
    (ours(x) * wout).sum().backward()
    one_call = {n: p.grad.clone() for n, p in ours.named_parameters()}
    for p in ours.parameters():
        p.grad.zero_()
    seen = []
    ours.grad_section_hook = lambda names: seen.extend(names)
    (ours(x) * wout).sum().backward()
    ours.grad_section_hook = None
    assert sorted(seen) == sorted(n for n, _ in ours.named_parameters())
    for n, p in ours.named_parameters():
        a, b = p.grad, one_call[n]
        assert (a - b).abs().max().item() <= 1e-4 * (b.abs().max().item() + 1e-6) + 1e-6, n


@pytest.mark.slow
def test_vit_base_patch8_224_training_gradients_match_oracle(lib):
    """ViT-B/8 at 224^2 (785 tokens, the tcgen05 backward in all 12 blocks), batch 8: every parameter gradient vs fp32 autograd of the
    oracle, at the ViT-B/16 bounds (weight matrices rel <= 0.15, cos >= 0.99; 1-D parameters rel <= 0.25, cos >= 0.97)."""
    torch.set_num_threads(min(16, torch.get_num_threads()))
    patch, dim, depth, heads = VIT_ARCHS["vit_base_patch8_224"]
    oracle = randomize_(ViTWrapperOracle("vit_base_patch8_224", 512, 224, patch=patch, dim=dim, depth=depth, heads=heads),
                        seed=5).train()
    ours = ViTWrapper("vit_base_patch8_224", 512, 224, pretrained=False)
    ours.load_state_dict(oracle.state_dict(), strict=True)
    ours = ours.cuda().train()
    torch.manual_seed(2)
    x = torch.randn(8, 3, 224, 224)
    wout = torch.randn(8, 512)
    (oracle(x) * wout).sum().backward()
    (ours(x.cuda()) * wout.cuda()).sum().backward()
    grads_match(ours, oracle, 0.15, 0.99, vec_rel_tol=0.25, vec_cos_tol=0.97)


def test_vit_train_step_above_208_tokens_with_circleloss(lib):
    """One config-3 style step on a 257-token toy ViT: forward -> CircleLoss + CE -> backward -> clip + SGD + EMA; loss decreases
    over 8 steps."""
    from visiondk_b200.train import FaceTrainingModel, FaceTrainer
    cfg = {"backbone": {"timm-vit_toy": {"pretrained": False, "image_size": 128, "feat_dim": 64, "patch": 8, "dim": 128, "depth": 2,
                                         "heads": 2}},
           "head": {"circleloss": {"feat_dim": 64, "num_class": 10, "margin": 0.25, "gamma": 64}}}
    torch.manual_seed(0)
    model = FaceTrainingModel(cfg).cuda()
    trainer = FaceTrainer(model, lr0=0.02, momentum=0.9, weight_decay=5e-4, label_smooth=0.0, layer_wise=True, warm_steps=0,
                          total_steps=100, use_ema=True)
    x = torch.randn(16, 3, 128, 128, device="cuda")
    y = torch.randint(0, 10, (16,), device="cuda")
    losses = [float(trainer.step(x, y)) for _ in range(8)]
    assert all(l == l for l in losses) and losses[-1] < losses[0], losses
