"""CPU checks of the long-sequence ViT architectures (ViT-*/8 at 224^2, ViT-*/16 at 384^2) and of the host side of the tcgen05
attention backward: factory resolution, parameter trees against the oracle, workspace sizing and the no-GPU failure mode."""
import pytest
import torch

from oracle import vit as oracle_vit
from oracle.vit import ViTWrapperOracle
from visiondk_b200 import _lib
from visiondk_b200.backbone import BackboneFactory
from visiondk_b200.vit import VIT_ARCHS, ViTWrapper

# timm 0.9.16 name (with a pretrained tag, as the reference's configs write them) -> image size
NEW_ARCHS = {
    "vit_small_patch8_224.dino": 224,
    "vit_base_patch8_224.dino": 224,
    "vit_small_patch16_384.augreg_in21k_ft_in1k": 384,
    "vit_base_patch16_384.augreg_in21k_ft_in1k": 384,
    "vit_large_patch16_384.augreg_in21k_ft_in1k": 384,
}


@pytest.mark.parametrize("tagged", sorted(NEW_ARCHS))
def test_factory_builds_long_sequence_vits(tagged):
    name, size = tagged.split(".")[0], NEW_ARCHS[tagged]
    patch, dim, depth, heads = VIT_ARCHS[name]
    tokens = (size // patch) ** 2 + 1
    with torch.device("meta"):
        ours = BackboneFactory({f"timm-{tagged}": {"pretrained": False, "image_size": size, "feat_dim": 8}}).get_backbone()
        oracle = ViTWrapperOracle(name, 8, size, patch=patch, dim=dim, depth=depth, heads=heads)
    assert isinstance(ours, ViTWrapper) and not ours.model.pre_norm
    assert ours.model.heads * 64 == ours.model.dim and ours.model.ln_eps == 1e-6
    assert ours.output_layer[2].in_features == tokens * dim
    assert set(ours.state_dict()) == set(oracle.state_dict())
    assert sum(p.numel() for p in ours.parameters()) == sum(p.numel() for p in oracle.parameters())


def test_long_sequence_token_counts():
    assert (224 // VIT_ARCHS["vit_base_patch8_224"][0]) ** 2 + 1 == 785
    assert (384 // VIT_ARCHS["vit_base_patch16_384"][0]) ** 2 + 1 == 577


def test_arch_tables_agree_on_shared_names():
    shared = set(VIT_ARCHS) & set(oracle_vit.VIT_ARCHS)
    assert shared
    for name in shared:
        assert VIT_ARCHS[name] == oracle_vit.VIT_ARCHS[name], name


@pytest.mark.parametrize("B,N,H", [(1, 1, 1), (2, 209, 2), (128, 785, 12), (64, 577, 16)])
def test_attention_bwd_tc_workspace_is_host_only(lib, B, N, H):
    need = lib.vdk_attention_bwd_tc_workspace_bytes(B, N, H, 64)
    assert need >= B * H * N * 4
    assert lib.vdk_attention_bwd_tc_workspace_bytes(B, N, H, 128) == 0
    assert lib.vdk_attention_bwd_tc_workspace_bytes(0, N, H, 64) == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_attention_bwd_tc_fails_loudly_without_gpu(lib):
    B, N, H = 2, 257, 2
    fake = 1 << 20  # never dereferenced: the call must fail before it touches memory
    need = lib.vdk_attention_bwd_tc_workspace_bytes(B, N, H, 64)
    rc = lib.vdk_attention_bwd_tc(fake, fake, fake, fake, B, N, H, 64, fake, fake, need, 0)
    assert rc != _lib.VDK_OK
    with pytest.raises(RuntimeError):
        _lib.check(rc, "vdk_attention_bwd_tc")
    assert lib.vdk_attention_bwd_tc(0, 0, 0, 0, B, N, H, 64, 0, 0, 0, 0) == _lib.VDK_ERR_INVALID
