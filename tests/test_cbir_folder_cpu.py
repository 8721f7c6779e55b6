"""engine/cbir/folder.py — the reference's local CBIRDatasets layout (dataset/basedataset.py:463-596) as the data source of
`valuate`: file lists, identity labels, positives, decoding order, the supported val transform list.  Host logic only (the
device half — preprocessing, extraction, search — has its own GPU tests)."""
import os

import numpy as np
import pytest
import torch

from engine.cbir.folder import CBIRFolderData, parse_val_augment, read_image
from oracle import preprocess as P

PIL = pytest.importorskip("PIL")
from PIL import Image  # noqa: E402

AUGMENT = [{"resize_and_padding": {"size": 64, "training": False}}, {"to_tensor": "no_params"},
           {"normalize": {"mean": [0.485, 0.456, 0.406], "std": [0.229, 0.224, 0.225]}}]


def make_tree(root, n_ids=4, per_gallery=3, per_query=2, seed=0):
    rng = np.random.default_rng(seed)
    images = {}
    for split, per in (("gallery", per_gallery), ("query", per_query)):
        for i in range(n_ids if split == "gallery" else n_ids - 1):  # the last identity has no query: a strict subset
            d = os.path.join(root, split, f"id_{i:02d}")
            os.makedirs(d)
            for j in range(per):
                w, h = int(rng.integers(20, 90)), int(rng.integers(20, 90))
                arr = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
                ext = "png" if j % 2 else "jpg"
                path = os.path.join(d, f"img_{j}.{ext}")
                Image.fromarray(arr).save(path, quality=95)
                images[path] = arr
    os.makedirs(os.path.join(root, "gallery", ".hidden"))  # dot entries are ignored (basedataset.py:589-590)
    return images


def test_lists_labels_and_positives(tmp_path):
    make_tree(str(tmp_path))
    data = CBIRFolderData(str(tmp_path), AUGMENT, batch=4, device="cpu", nw=2)
    assert data.identities == ["id_00", "id_01", "id_02", "id_03"]
    assert len(data.gallery_files) == 12 and len(data.query_files) == 6
    # jpg files of an identity come before its png files (basedataset.py:503-504), identities in sorted order
    assert [os.path.basename(f) for f in data.gallery_files[:3]] == ["img_0.jpg", "img_2.jpg", "img_1.png"]
    assert data.gallery_labels().tolist() == [0, 0, 0, 1, 1, 1, 2, 2, 2, 3, 3, 3]
    assert data.query_labels().tolist() == [0, 0, 1, 1, 2, 2]
    assert data.query_labels(3).tolist() == [0, 0, 1] and data.gallery_labels(4).tolist() == [0, 0, 0, 1]
    pos = data.positives()
    assert len(pos) == 6 and all(len(p) == 3 for p in pos)
    for q, p in zip(data.query_files, pos):  # a query's positives = the gallery files of its identity folder
        ident = os.path.basename(os.path.dirname(q))
        assert all(os.path.basename(os.path.dirname(g)) == ident for g in p)
    assert (data.size, data.mean, data.std) == (64, (0.485, 0.456, 0.406), (0.229, 0.224, 0.225))


def test_layout_errors_like_the_reference(tmp_path):
    with pytest.raises(ValueError, match="query dir and gallery dir"):
        CBIRFolderData(str(tmp_path), AUGMENT, 4, "cpu")
    make_tree(str(tmp_path))
    os.makedirs(tmp_path / "query" / "stranger")
    with pytest.raises(ValueError, match="not subset"):
        CBIRFolderData(str(tmp_path), AUGMENT, 4, "cpu")


def test_decoding_order_and_content(tmp_path):
    images = make_tree(str(tmp_path))
    data = CBIRFolderData(str(tmp_path), AUGMENT, batch=5, device="cpu", nw=3)
    batches = list(data.decoded_batches(data.gallery_files))
    assert [len(b) for b in batches] == [5, 5, 2]
    flat = [im for b in batches for im in b]
    for path, im in zip(data.gallery_files, flat):
        assert im.dtype == np.uint8 and im.ndim == 3 and im.shape[2] == 3
        ref = np.asarray(Image.open(path).convert("RGB"))
        assert np.array_equal(im, ref)
        if path.endswith(".png"):  # lossless: the stored array itself
            assert np.array_equal(im, images[path])
    assert list(data.decoded_batches([])) == []
    grey = tmp_path / "grey.png"
    Image.fromarray(np.arange(64, dtype=np.uint8).reshape(8, 8)).save(grey)
    assert read_image(str(grey)).shape == (8, 8, 3)  # .convert('RGB') like basedataset.py:236


def test_file_to_tensor_equals_the_reference_transform(tmp_path):
    """file -> read_image -> oracle preprocessing == file -> PIL -> the reference's val transform steps (the device pipeline is
    held to the oracle bit for bit by tests/test_preprocess_gpu.py)."""
    import torchvision.transforms as T
    from PIL import ImageOps
    make_tree(str(tmp_path))
    data = CBIRFolderData(str(tmp_path), AUGMENT, batch=4, device="cpu")
    for path in data.query_files:
        image = Image.open(path).convert("RGB")
        w, h = image.size
        s = data.size / max(w, h)
        nw, nh = int(w * s), int(h * s)
        image = image.resize((nw, nh), Image.BILINEAR)
        pw, ph = (data.size - nw) // 2, (data.size - nh) // 2
        image = ImageOps.expand(image, (pw, ph, data.size - nw - pw, data.size - nh - ph), fill=(0, 0, 0))
        ref = T.Normalize(mean=data.mean, std=data.std)(T.ToTensor()(image)).numpy()
        got = P.resize_pad_normalize(read_image(path), data.size, data.mean, data.std)
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_val_augment_parsing():
    assert parse_val_augment(AUGMENT) == (64, (0.485, 0.456, 0.406), (0.229, 0.224, 0.225))
    assert parse_val_augment([{"resize_and_padding": {"size": 336}}, {"to_tensor": "no_params"}, {"normalize": "no_params"}])[0] == 336
    with pytest.raises(NotImplementedError, match="center_crop"):
        parse_val_augment([{"center_crop": {"size": 224}}, {"to_tensor": "no_params"}, {"normalize": "no_params"}])
    with pytest.raises(NotImplementedError, match="training=True"):
        parse_val_augment([{"resize_and_padding": {"size": 224, "training": True}}, {"to_tensor": "no_params"}, {"normalize": "no_params"}])


def test_reference_cbir_yaml_val_list_is_the_supported_one():
    """The val augment list of the reference's own configs/faceX/cbir.yaml (written out by value, and checked against the
    file's fixture copy tests/golden/ref_configs/cbir.yaml) parses to its image size and the ImageNet statistics."""
    ref_list = [{"resize_and_padding": {"size": 224, "training": False}}, {"to_tensor": "no_params"},
                {"normalize": {"mean": [0.485, 0.456, 0.406], "std": [0.229, 0.224, 0.225]}}]
    assert parse_val_augment(ref_list) == (224, (0.485, 0.456, 0.406), (0.229, 0.224, 0.225))
    import yaml
    with open(os.path.join(os.path.dirname(__file__), "golden", "ref_configs", "cbir.yaml")) as f:
        assert yaml.safe_load(f)["data"]["val"]["augment"] == ref_list
