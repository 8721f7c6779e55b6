"""The oracle's TimmWrapper restatements (oracle/convnext.py::TimmWrapperOracle, oracle/vit.py::ViTWrapperOracle) against
tests/golden/neck_ref.npz, minted by executing the REFERENCE's own models/faceX/backbone/timm_wrapper.py:5-54 around a stub
`timm` (oracle/make_golden.py::neck): state_dict key set, both neck branches (CNN: BatchNorm2d -> Flatten -> Linear ->
BatchNorm1d, :30-38; Transformer: LayerNorm -> Flatten -> Linear -> BatchNorm1d, :39-47) in eval and in train mode
(batch statistics, running-stat update, gradients)."""
import os

import numpy as np
import pytest
import torch

from oracle.convnext import TimmWrapperOracle, randomize_ as rand_cnx
from oracle.vit import ViTWrapperOracle, randomize_ as rand_vit

GOLD = os.path.join(os.path.dirname(__file__), "golden", "neck_ref.npz")


def build(tag, z):
    if tag == "cnn":
        m = rand_cnx(TimmWrapperOracle("toy", 64, 64, depths=(1, 1, 2, 1), dims=(64, 128, 128, 256)), seed=int(z["cnn_seed"]))
    else:
        m = rand_vit(ViTWrapperOracle("toy", 64, 64, patch=16, dim=128, depth=2, heads=2), seed=int(z["vit_seed"]))
    return m


@pytest.fixture
def golden_threads():
    """neck_ref.npz was minted with 8 intra-op CPU threads.  The CPU kernels split their reductions by thread count, and the
    train-mode gradients of the 6-image batch are ill-conditioned: at any other count the Transformer neck's Linear weight
    gradient moves by up to 3e-4 (float64 misses the golden by as much).  The test runs with the golden's 8 threads."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("tag", ["cnn", "vit"])
def test_oracle_wrapper_reproduces_the_reference_wrapper(tag, golden_threads):
    z = np.load(GOLD)
    m = build(tag, z)
    sd = m.state_dict()
    assert list(sd.keys()) == [str(k) for k in z[f"{tag}_keys"]], "state_dict keys differ from the reference TimmWrapper's"
    body = sum(v.double().abs().sum().item() for k, v in sd.items() if k.startswith("model."))
    assert abs(body - float(z[f"{tag}_body_abs_sum"])) <= 1e-9 * body
    for k in sd:
        if k.startswith("output_layer."):
            assert np.array_equal(sd[k].numpy(), z[f"{tag}_sd/{k}"]), k
    x = torch.from_numpy(z["x"])
    m.eval()
    with torch.no_grad():
        np.testing.assert_allclose(m.model(x).numpy(), z[f"{tag}_feat"], rtol=0, atol=1e-6)
        np.testing.assert_allclose(m(x).numpy(), z[f"{tag}_eval"], rtol=0, atol=2e-6)
    m.train()
    feat = torch.from_numpy(z[f"{tag}_feat"]).requires_grad_(True)
    y = m.output_layer(feat)
    (y * torch.from_numpy(z[f"{tag}_w_out"])).sum().backward()
    np.testing.assert_allclose(y.detach().numpy(), z[f"{tag}_train"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(feat.grad.numpy(), z[f"{tag}_dfeat"], rtol=1e-4, atol=1e-6)
    for k, p in m.output_layer.named_parameters():
        np.testing.assert_allclose(p.grad.numpy(), z[f"{tag}_grad/output_layer.{k}"], rtol=1e-4, atol=1e-5, err_msg=k)
    for k, b in m.output_layer.named_buffers():
        np.testing.assert_allclose(b.numpy(), z[f"{tag}_after/output_layer.{k}"], rtol=1e-6, atol=1e-7, err_msg=k)
