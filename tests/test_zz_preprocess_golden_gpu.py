"""The device preprocessing (csrc/preprocess.cu) against tensors produced by the reference's OWN eval-time input pipeline
(tests/golden/preprocess_ref.npz: dataset/transforms.py `create_AugTransforms` on the val augment list of
configs/faceX/cbir.yaml, minted by oracle/make_golden.py::preprocess) — bit for bit, one mixed-size batch per image size.
(The oracle is held to the same file by tests/test_oracle_preprocess_cpu.py, the kernels to the oracle by
tests/test_preprocess_gpu.py; this closes the triangle directly.)"""
import os

import numpy as np
import pytest

from visiondk_b200.preprocess import resize_pad_normalize

pytestmark = pytest.mark.gpu


def test_device_pipeline_reproduces_the_reference_tensors(lib):
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "preprocess_ref.npz"))
    mean, std = tuple(float(v) for v in z["mean"]), tuple(float(v) for v in z["std"])
    by_size = {}
    for n in range(int(z["count"])):
        if min(z[f"img{n}"].shape[:2]) >= 2:  # the 1 x 1 source image is held to the golden on the oracle side only
            by_size.setdefault(int(z[f"size{n}"]), []).append(n)
    assert sum(len(v) for v in by_size.values()) >= 12
    for size, idx in by_size.items():
        out = resize_pad_normalize([z[f"img{n}"] for n in idx], size=size, mean=mean, std=std).cpu().numpy()
        for row, n in enumerate(idx):
            ref = z[f"out{n}"]
            assert np.array_equal(out[row].view(np.uint32), ref.view(np.uint32)), (n, z[f"img{n}"].shape, size)
