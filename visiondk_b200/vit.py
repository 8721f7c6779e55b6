"""ViT backbones for the CBIR extract path (inference) on the B200 kernels.

Mirrors what `TimmWrapper(model_name='vit_*', feat_dim, image_size)` builds in the reference
(models/faceX/backbone/timm_wrapper.py:16-21 + the Transformer neck of :39-47): the parameter tree and state_dict keys of
timm 0.9.16's VisionTransformer (`model.patch_embed.proj`, `model.cls_token`, `model.pos_embed`, `model.blocks.{i}.{norm1,
attn.qkv, attn.proj, norm2, mlp.fc1, mlp.fc2}`, `model.norm`) and `output_layer.{0: LayerNorm, 2: Linear, 3: BatchNorm1d}`,
so reference checkpoints load with `strict=True`.  The eval forward runs in `vdk_vit_forward`, the train-mode forward and
backward (BASELINE config 3) in `vdk_vit_train_forward` / `vdk_vit_train_backward` (csrc/vit.cu) as ONE autograd node;
training needs 3*patch^2 % 8 == 0 and takes any token count: the attention backward runs the mma.sync kernel up to 208 tokens
(ViT-*/16 at 224^2) and the tcgen05 pair of csrc/attention_bwd_tc.cu beyond (ViT-*/8 at 224^2: 785 tokens; ViT-*/16 at 384^2: 577).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import torch
import torch.nn as nn

from . import _lib

VIT_ARCHS = {
    # timm name -> (patch, embed_dim, depth, heads)
    "vit_tiny_patch16_224": (16, 192, 12, 3),
    "vit_small_patch16_224": (16, 384, 12, 6),
    "vit_base_patch16_224": (16, 768, 12, 12),
    "vit_large_patch16_224": (16, 1024, 24, 16),
    "vit_small_patch8_224": (8, 384, 12, 6),
    "vit_base_patch8_224": (8, 768, 12, 12),
    "vit_small_patch16_384": (16, 384, 12, 6),
    "vit_base_patch16_384": (16, 768, 12, 12),
    "vit_large_patch16_384": (16, 1024, 24, 16),
    "vit_base_patch16_clip_224": (16, 768, 12, 12),
    "vit_large_patch14_clip_224": (14, 1024, 24, 16),
    "vit_large_patch14_clip_336": (14, 1024, 24, 16),
}
# timm 0.9.16 `vit_*_clip_*` (the CLIP image towers; BASELINE config 5's ViT-L/14 at 336^2): VisionTransformer(pre_norm=True,
# norm_layer=nn.LayerNorm): a `norm_pre` LayerNorm after cls / position, NO bias in patch_embed.proj, LayerNorm eps 1e-5,
# standard GELU (the `*_clip_quickgelu_*` architectures are separate timm entries and are not built).
VIT_PRE_NORM = {"vit_base_patch16_clip_224", "vit_large_patch14_clip_224", "vit_large_patch14_clip_336"}
MAX_BLOCKS = 48


class _Attention(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.qkv = nn.Linear(dim, 3 * dim, bias=True)
        self.proj = nn.Linear(dim, dim)


class _Mlp(nn.Module):
    def __init__(self, dim):
        super().__init__()
        self.fc1 = nn.Linear(dim, 4 * dim)
        self.fc2 = nn.Linear(4 * dim, dim)


class _Block(nn.Module):
    def __init__(self, dim, eps=1e-6):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=eps)
        self.attn = _Attention(dim)
        self.norm2 = nn.LayerNorm(dim, eps=eps)
        self.mlp = _Mlp(dim)


class _PatchEmbed(nn.Module):
    def __init__(self, patch, dim, bias=True):
        super().__init__()
        self.proj = nn.Conv2d(3, dim, kernel_size=patch, stride=patch, bias=bias)


class ViTParams(nn.Module):
    """timm 0.9.16 `VisionTransformer(num_classes=0, global_pool='')` parameter tree (timm/models/vision_transformer.py)."""

    def __init__(self, image_size, patch, dim, depth, heads, pre_norm=False):
        super().__init__()
        self.image_size, self.patch, self.dim, self.depth, self.heads = image_size, patch, dim, depth, heads
        self.pre_norm = bool(pre_norm)
        self.ln_eps = 1e-5 if pre_norm else 1e-6
        n = (image_size // patch) ** 2
        self.patch_embed = _PatchEmbed(patch, dim, bias=not pre_norm)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, dim))
        self.pos_embed = nn.Parameter(torch.randn(1, n + 1, dim) * 0.02)
        if pre_norm:
            self.norm_pre = nn.LayerNorm(dim, eps=self.ln_eps)
        self.blocks = nn.Sequential(*[_Block(dim, self.ln_eps) for _ in range(depth)])
        self.norm = nn.LayerNorm(dim, eps=self.ln_eps)
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.trunc_normal_(m.weight, std=0.02)
                nn.init.zeros_(m.bias)
        nn.init.normal_(self.cls_token, std=1e-6)


class _VitBlockC(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("ln1_w", "ln1_b", "qkv_w", "qkv_b", "proj_w", "proj_b", "ln2_w", "ln2_b", "fc1_w", "fc1_b",
                                          "fc2_w", "fc2_b")]


class _VitBlockTensorsC(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("ln1_w", "ln1_b", "qkv_w", "qkv_b", "proj_w", "proj_b", "ln2_w", "ln2_b", "fc1_w", "fc1_b",
                                          "fc2_w", "fc2_b")]


class VitTensorsC(C.Structure):
    """vdk_vit_tensors: fp32 tensors in timm layouts (parameters, or their gradients)."""
    _fields_ = [("patch_w", C.c_void_p), ("patch_b", C.c_void_p), ("cls_token", C.c_void_p), ("pos_embed", C.c_void_p),
                ("blocks", _VitBlockTensorsC * MAX_BLOCKS),
                ("norm_w", C.c_void_p), ("norm_b", C.c_void_p), ("neck_ln_w", C.c_void_p), ("neck_ln_b", C.c_void_p),
                ("lin_w", C.c_void_p), ("lin_b", C.c_void_p),
                ("bn1_w", C.c_void_p), ("bn1_b", C.c_void_p), ("bn1_running_mean", C.c_void_p), ("bn1_running_var", C.c_void_p)]


class VitNetC(C.Structure):
    """vdk_vit_net (include/vdk_b200.h)."""
    _fields_ = [("image_size", C.c_int), ("patch", C.c_int), ("dim", C.c_int), ("depth", C.c_int), ("heads", C.c_int),
                ("feat_dim", C.c_int),
                ("patch_w", C.c_void_p), ("patch_b", C.c_void_p), ("cls_token", C.c_void_p), ("pos_embed", C.c_void_p),
                ("ones", C.c_void_p), ("blocks", _VitBlockC * MAX_BLOCKS),
                ("norm_w", C.c_void_p), ("norm_b", C.c_void_p), ("neck_ln_w", C.c_void_p), ("neck_ln_b", C.c_void_p),
                ("neck_w", C.c_void_p), ("neck_b", C.c_void_p),
                ("norm_pre_w", C.c_void_p), ("norm_pre_b", C.c_void_p), ("ln_eps", C.c_float)]


class ViTWrapper(nn.Module):
    """Drop-in for the reference's TimmWrapper when the timm model is a VisionTransformer (eval / extract path)."""

    def __init__(self, model_name: str, feat_dim: int, image_size: int, pretrained: bool = True, patch=None, dim=None, depth=None,
                 heads=None, pre_norm=None, **kwargs):
        super().__init__()
        if dim is None:
            if model_name not in VIT_ARCHS:
                raise ValueError(f"backbone '{model_name}' is not built for B200 yet; available: {sorted(VIT_ARCHS)}")
            patch, dim, depth, heads = VIT_ARCHS[model_name]
        if pre_norm is None:
            pre_norm = model_name in VIT_PRE_NORM
        if image_size % patch != 0 or dim != heads * 64 or depth > MAX_BLOCKS:
            raise ValueError("ViT on B200: image_size must be a multiple of patch, head_dim must be 64, depth <= 48")
        self.model_name, self.feat_dim, self.image_size = model_name, int(feat_dim), int(image_size)
        self.model = ViTParams(image_size, patch, dim, depth, heads, pre_norm=pre_norm)
        tokens = (image_size // patch) ** 2 + 1
        self.output_layer = nn.Sequential(nn.LayerNorm(dim), nn.Flatten(1), nn.Linear(tokens * dim, feat_dim),
                                          nn.BatchNorm1d(feat_dim))
        self._packed: Optional[Dict] = None
        self._packed_key = None
        self._ws = None
        self._train = None
        if pretrained:
            raise RuntimeError("pretrained timm weights cannot be downloaded here (no network): pass pretrained=False and "
                               "load a checkpoint with load_state_dict (keys are timm's)")

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if self.training and self.model.pre_norm:
            raise NotImplementedError("pre_norm ViT variants (CLIP towers) are built for inference / extraction only")
        if self.training:
            return _ViTTrainFn.apply(self, x, *[p for _, p in self.named_parameters()])
        return self.embed(x, l2_normalize=False)

    # ---- training path (csrc/vit.cu: vdk_vit_train_forward / vdk_vit_train_backward) -------------------------------------
    def _tensors_struct(self, get) -> VitTensorsC:
        t = VitTensorsC()
        t.patch_w, t.patch_b = get("model.patch_embed.proj.weight"), get("model.patch_embed.proj.bias")
        t.cls_token, t.pos_embed = get("model.cls_token"), get("model.pos_embed")
        for i in range(self.model.depth):
            b, pre = t.blocks[i], f"model.blocks.{i}."
            b.ln1_w, b.ln1_b = get(pre + "norm1.weight"), get(pre + "norm1.bias")
            b.qkv_w, b.qkv_b = get(pre + "attn.qkv.weight"), get(pre + "attn.qkv.bias")
            b.proj_w, b.proj_b = get(pre + "attn.proj.weight"), get(pre + "attn.proj.bias")
            b.ln2_w, b.ln2_b = get(pre + "norm2.weight"), get(pre + "norm2.bias")
            b.fc1_w, b.fc1_b = get(pre + "mlp.fc1.weight"), get(pre + "mlp.fc1.bias")
            b.fc2_w, b.fc2_b = get(pre + "mlp.fc2.weight"), get(pre + "mlp.fc2.bias")
        t.norm_w, t.norm_b = get("model.norm.weight"), get("model.norm.bias")
        t.neck_ln_w, t.neck_ln_b = get("output_layer.0.weight"), get("output_layer.0.bias")
        t.lin_w, t.lin_b = get("output_layer.2.weight"), get("output_layer.2.bias")
        t.bn1_w, t.bn1_b = get("output_layer.3.weight"), get("output_layer.3.bias")
        t.bn1_running_mean, t.bn1_running_var = get("output_layer.3.running_mean"), get("output_layer.3.running_var")
        return t

    def backward_sections(self):
        """[((unit_begin, unit_end), [parameter names final after that range]), ...]: neck + final norm + the last third of the
        blocks; the middle third; the first third + patch / cls / position embeddings — each a contiguous run of named_parameters()."""
        d = self.model.depth
        names = [n for n, _ in self.named_parameters()]

        def blk(n):
            return int(n.split(".")[2]) if n.startswith("model.blocks.") else None

        c1, c2 = d - d // 3, d - 2 * (d // 3)  # blocks >= c1 | c2 <= blocks < c1 | blocks < c2
        sec = [
            ((0, 1 + (d - c1)), [n for n in names if n.startswith("output_layer.") or n.startswith("model.norm.") or
                                 (blk(n) is not None and blk(n) >= c1)]),
            ((1 + (d - c1), 1 + (d - c2)), [n for n in names if blk(n) is not None and c2 <= blk(n) < c1]),
            ((1 + (d - c2), d + 2), [n for n in names if (blk(n) is not None and blk(n) < c2) or n in ("model.cls_token", "model.pos_embed")
                                     or n.startswith("model.patch_embed.")]),
        ]
        if sum(len(ns) for _, ns in sec) != len(names):
            raise RuntimeError("backward_sections: parameters not covered exactly once")
        return [x for x in sec if x[0][0] < x[0][1] and x[1]]

    def _train_structs(self, device):
        m = self.model
        if self._train is None or self._train["device"] != device:
            def buf(*shape):
                return torch.empty(shape, dtype=torch.bfloat16, device=device)
            tokens = (m.image_size // m.patch) ** 2 + 1
            self._train = {"device": device, "ws": None, "gflat": None, "last": None,
                           "patch_w": buf(m.dim, 3 * m.patch * m.patch),
                           "blocks": [{"qkv_w": buf(3 * m.dim, m.dim), "proj_w": buf(m.dim, m.dim), "fc1_w": buf(4 * m.dim, m.dim),
                                       "fc2_w": buf(m.dim, 4 * m.dim)} for _ in range(m.depth)],
                           "neck_w": buf(self.feat_dim, tokens * m.dim),
                           "ones": torch.ones(m.dim, dtype=torch.float32, device=device)}
        st = self._train
        named = dict(self.named_parameters())
        named.update(dict(self.named_buffers()))
        for n, t in named.items():
            if t.is_floating_point() and (t.device != device or t.dtype != torch.float32 or not t.is_contiguous()):
                raise RuntimeError(f"{n}: training needs contiguous fp32 parameters on {device}")
        params = self._tensors_struct(lambda n: named[n].data_ptr())
        net = VitNetC()
        net.image_size, net.patch, net.dim, net.depth, net.heads, net.feat_dim = (m.image_size, m.patch, m.dim, m.depth, m.heads,
                                                                                 self.feat_dim)
        net.patch_w, net.patch_b = st["patch_w"].data_ptr(), params.patch_b
        net.cls_token, net.pos_embed, net.ones = params.cls_token, params.pos_embed, st["ones"].data_ptr()
        for i in range(m.depth):
            b, pb, bb = net.blocks[i], params.blocks[i], st["blocks"][i]
            b.ln1_w, b.ln1_b, b.qkv_b, b.proj_b = pb.ln1_w, pb.ln1_b, pb.qkv_b, pb.proj_b
            b.ln2_w, b.ln2_b, b.fc1_b, b.fc2_b = pb.ln2_w, pb.ln2_b, pb.fc1_b, pb.fc2_b
            b.qkv_w, b.proj_w = bb["qkv_w"].data_ptr(), bb["proj_w"].data_ptr()
            b.fc1_w, b.fc2_w = bb["fc1_w"].data_ptr(), bb["fc2_w"].data_ptr()
        net.norm_w, net.norm_b, net.neck_ln_w, net.neck_ln_b = params.norm_w, params.norm_b, params.neck_ln_w, params.neck_ln_b
        net.neck_w, net.neck_b = st["neck_w"].data_ptr(), params.lin_b
        return st, net, params

    def _train_forward(self, x: torch.Tensor) -> torch.Tensor:
        lib = _lib.load()
        if x.device.type != "cuda":
            raise RuntimeError("visiondk_b200.ViTWrapper runs on CUDA (sm_100a) only; there is no CPU fallback")
        x = x.contiguous().float()
        B = x.shape[0]
        st, net, params = self._train_structs(x.device)
        need = lib.vdk_vit_train_workspace_bytes(C.byref(net), B)
        if need == 0:
            raise RuntimeError("vdk_vit_train_workspace_bytes: " + _lib.last_error())
        if st["ws"] is None or st["ws"].numel() < need:
            st["ws"] = torch.empty((need,), dtype=torch.uint8, device=x.device)
        out = torch.empty((B, self.feat_dim), dtype=torch.float32, device=x.device)
        bn = self.output_layer[3]
        with torch.cuda.device(x.device):
            s = _lib.stream_ptr()
            _lib.check(lib.vdk_vit_pack(C.byref(params), C.byref(net), s), "vdk_vit_pack")
            _lib.check(lib.vdk_vit_train_forward(C.byref(net), C.byref(params), x.data_ptr(), B, float(bn.momentum), out.data_ptr(),
                                                 st["ws"].data_ptr(), st["ws"].numel(), s), "vdk_vit_train_forward")
        bn.num_batches_tracked += 1
        st["last"] = (net, params, B)
        return out

    def _train_backward(self, dout: torch.Tensor):
        """Gradients of every parameter: accumulated straight into pre-allocated fp32 `.grad` buffers when every parameter owns
        one (the fused optimizer's flat buffer), else produced in a scratch buffer and returned to autograd."""
        lib = _lib.load()
        st = self._train
        net, params, B = st["last"]
        plist = list(self.named_parameters())
        direct = all(p.grad is not None and p.grad.dtype == torch.float32 and p.grad.is_contiguous() and
                     p.grad.device == dout.device for _, p in plist)
        if direct:
            ptrs = {n: p.grad.data_ptr() for n, p in plist}
        else:
            total = sum(p.numel() for _, p in plist)
            if st["gflat"] is None or st["gflat"].numel() != total:
                st["gflat"] = torch.empty((total,), dtype=torch.float32, device=dout.device)
            gflat = st["gflat"]
            gflat.zero_()
            offs, off = {}, 0
            for n, p in plist:
                offs[n] = off
                off += p.numel()
            ptrs = {n: gflat.data_ptr() + 4 * offs[n] for n, _ in plist}
        grads = self._tensors_struct(lambda n: ptrs.get(n, 0))
        dout = dout.contiguous().float()
        hook = getattr(self, "grad_section_hook", None)
        with torch.cuda.device(dout.device):
            if hook is not None and direct:  # DDP overlap: reduce the gradients a unit range completed while the next one runs
                for (u0, u1), names in self.backward_sections():
                    _lib.check(lib.vdk_vit_train_backward_range(C.byref(net), C.byref(params), C.byref(grads), dout.data_ptr(), B,
                                                                st["ws"].data_ptr(), st["ws"].numel(), _lib.stream_ptr(), u0, u1),
                               "vdk_vit_train_backward_range")
                    hook(names)
            else:
                _lib.check(lib.vdk_vit_train_backward(C.byref(net), C.byref(params), C.byref(grads), dout.data_ptr(), B,
                                                      st["ws"].data_ptr(), st["ws"].numel(), _lib.stream_ptr()),
                           "vdk_vit_train_backward")
        if direct:
            return [None] * len(plist)
        return [gflat[offs[n]:offs[n] + p.numel()].view_as(p) for n, p in plist]

    def _version_key(self, device):
        return (str(device),) + tuple(int(t._version) for t in list(self.parameters()) + list(self.buffers()))

    def _pack(self, device) -> VitNetC:
        key = self._version_key(device)
        if self._packed is not None and self._packed_key == key:
            return self._packed["net"]
        keep = []

        def f32(t):
            t = t.detach().to(device, torch.float32).contiguous()
            keep.append(t)
            return t.data_ptr()

        def bf16(t):
            t = t.detach().to(device, torch.float32).contiguous().to(torch.bfloat16)
            keep.append(t)
            return t.data_ptr()

        m, net = self.model, VitNetC()
        net.image_size, net.patch, net.dim, net.depth, net.heads, net.feat_dim = (m.image_size, m.patch, m.dim, m.depth, m.heads,
                                                                                 self.feat_dim)
        k = 3 * m.patch * m.patch
        kp = (k + 7) // 8 * 8
        w = m.patch_embed.proj.weight.detach().reshape(m.dim, k)  # (c, kh, kw) order
        if kp != k:
            w = torch.cat([w, torch.zeros(m.dim, kp - k, dtype=w.dtype, device=w.device)], dim=1)
        net.patch_w = bf16(w)
        net.patch_b = f32(m.patch_embed.proj.bias) if m.patch_embed.proj.bias is not None else 0
        if m.pre_norm:
            net.norm_pre_w, net.norm_pre_b = f32(m.norm_pre.weight), f32(m.norm_pre.bias)
        net.ln_eps = float(m.ln_eps)
        net.cls_token, net.pos_embed = f32(m.cls_token.reshape(-1)), f32(m.pos_embed.reshape(-1, m.dim))
        net.ones = f32(torch.ones(m.dim))
        for i, blk in enumerate(m.blocks):
            b = net.blocks[i]
            b.ln1_w, b.ln1_b = f32(blk.norm1.weight), f32(blk.norm1.bias)
            b.qkv_w, b.qkv_b = bf16(blk.attn.qkv.weight), f32(blk.attn.qkv.bias)
            b.proj_w, b.proj_b = bf16(blk.attn.proj.weight), f32(blk.attn.proj.bias)
            b.ln2_w, b.ln2_b = f32(blk.norm2.weight), f32(blk.norm2.bias)
            b.fc1_w, b.fc1_b = bf16(blk.mlp.fc1.weight), f32(blk.mlp.fc1.bias)
            b.fc2_w, b.fc2_b = bf16(blk.mlp.fc2.weight), f32(blk.mlp.fc2.bias)
        net.norm_w, net.norm_b = f32(m.norm.weight), f32(m.norm.bias)
        ln, lin, bn = self.output_layer[0], self.output_layer[2], self.output_layer[3]
        net.neck_ln_w, net.neck_ln_b = f32(ln.weight), f32(ln.bias)
        # BatchNorm1d (eval statistics) folded into the Linear: y = s * (W x + b - mean) + beta, s = gamma / sqrt(var + eps)
        s = (bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + bn.eps))
        wn = lin.weight.detach().double() * s[:, None]
        bnb = (lin.bias.detach().double() - bn.running_mean.detach().double()) * s + bn.bias.detach().double()
        net.neck_w, net.neck_b = bf16(wn.float()), f32(bnb.float())
        self._packed, self._packed_key = {"net": net, "keep": keep}, key
        return net

    @torch.no_grad()
    def embed(self, x: torch.Tensor, l2_normalize: bool = False) -> torch.Tensor:
        """[B,3,S,S] fp32 NCHW -> fp32 [B, feat_dim] (TimmWrapper.forward in eval mode; optionally F.normalize fused)."""
        lib = _lib.load()
        if x.device.type != "cuda":
            raise RuntimeError("visiondk_b200.ViTWrapper runs on CUDA (sm_100a) only; there is no CPU fallback")
        if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] != self.image_size or x.shape[3] != self.image_size:
            raise ValueError(f"expected [B,3,{self.image_size},{self.image_size}], got {tuple(x.shape)}")
        x = x.contiguous().float()
        net = self._pack(x.device)
        B = x.shape[0]
        out = torch.empty((B, self.feat_dim), dtype=torch.float32, device=x.device)
        need = lib.vdk_vit_workspace_bytes(C.byref(net), B)
        if need == 0:
            raise RuntimeError("vdk_vit_workspace_bytes: " + _lib.last_error())
        if self._ws is None or self._ws.numel() < need or self._ws.device != x.device:
            self._ws = torch.empty((need,), dtype=torch.uint8, device=x.device)
        with torch.cuda.device(x.device):
            _lib.check(lib.vdk_vit_forward(C.byref(net), x.data_ptr(), B, int(l2_normalize), out.data_ptr(), self._ws.data_ptr(),
                                           self._ws.numel(), _lib.stream_ptr()), "vdk_vit_forward")
        return out


class _ViTTrainFn(torch.autograd.Function):
    """Train-mode forward/backward of the whole ViT + neck as one autograd node (csrc/vit.cu)."""

    @staticmethod
    def forward(ctx, module, x, *params):
        ctx.module = module
        return module._train_forward(x)

    @staticmethod
    def backward(ctx, dout):
        grads = ctx.module._train_backward(dout)
        return (None, None, *grads)

