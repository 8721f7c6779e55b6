"""`valuate` on an image FOLDER in the reference's CBIRDatasets layout (engine/cbir/folder.py): files -> host decode -> device
val transforms -> embed -> index -> search -> metrics, against the same computation assembled by hand from the oracle's
preprocessing of the same files (bit-exact inputs => identical embeddings => identical metrics), plus the vis=True return."""
import os

import numpy as np
import pytest
import torch

from oracle import preprocess as P

pytestmark = pytest.mark.gpu

SIZE = 64
AUGMENT = [{"resize_and_padding": {"size": SIZE, "training": False}}, {"to_tensor": "no_params"},
           {"normalize": {"mean": [0.485, 0.456, 0.406], "std": [0.229, 0.224, 0.225]}}]


def make_tree(root, n_ids=6, per_gallery=4, per_query=2):
    from PIL import Image
    rng = np.random.default_rng(11)
    for i in range(n_ids):
        proto = rng.integers(0, 256, (8, 8, 3), dtype=np.uint8)  # every identity = one low-resolution pattern + noise
        for split, per in (("gallery", per_gallery), ("query", per_query)):
            d = os.path.join(root, split, f"id_{i:02d}")
            os.makedirs(d)
            for j in range(per):
                w, h = int(rng.integers(40, 120)), int(rng.integers(40, 120))
                img = np.asarray(Image.fromarray(proto).resize((w, h), Image.NEAREST)).astype(np.int16)
                img = np.clip(img + rng.integers(-20, 21, img.shape), 0, 255).astype(np.uint8)
                Image.fromarray(img).save(os.path.join(d, f"img_{j}.png"))


def test_valuate_on_an_image_folder(lib, tmp_path):
    from engine.cbir.evaluation import compute_metrics, valuate
    from engine.cbir.folder import CBIRFolderData, read_image
    from visiondk_b200.backbone import TimmWrapper
    from visiondk_b200.retrieval import FlatIPIndex
    make_tree(str(tmp_path))
    # 64-d embeddings: the top-k search takes widths that are multiples of 64 (vdk_topk_plan_default)
    model = TimmWrapper("toy", 64, SIZE, pretrained=False, depths=(1, 1, 1, 1), dims=(64, 64, 128, 128)).cuda().eval()
    metrics_cfg = {"metrics": ["mrr", "recall", "precision", "auc", "ndcg"], "cutoffs": [1, 3, 5]}
    data_cfg = {"root": str(tmp_path), "nw": 2, "val": {"bs": 5, "augment": AUGMENT, "metrics": metrics_cfg}}
    got = valuate(model, data_cfg, "cuda", image_size=SIZE)
    assert {k.split("@")[0] for k in got} == {"MRR", "Recall", "Precision", "AUC", "nDCG"} and len(got) == 13
    assert all(0.0 <= v <= 1.0 or np.isnan(v) for v in got.values())

    # the same evaluation assembled by hand: oracle preprocessing on the host, same batch size
    data = CBIRFolderData(str(tmp_path), AUGMENT, 5, "cuda")

    def embed(files):
        out = []
        for a in range(0, len(files), 5):
            x = np.stack([P.resize_pad_normalize(read_image(f), SIZE, data.mean, data.std) for f in files[a:a + 5]])
            out.append(model.embed(torch.from_numpy(x).cuda(), l2_normalize=True))
        return torch.cat(out)

    index = FlatIPIndex(64, "cuda")
    index.add(embed(data.gallery_files))
    scores, ids = index.search_device(embed(data.query_files), 5, resolve_overflow=True)
    want = compute_metrics(ids, scores, data.query_labels(), data.gallery_labels(), metrics=metrics_cfg["metrics"],
                           cutoffs=metrics_cfg["cutoffs"])
    np.testing.assert_equal({k: float(v) for k, v in want.items()}, got)

    results, vis_scores, positives, queries = valuate(model, data_cfg, "cuda", vis=True, image_size=SIZE)
    assert queries == data.query_files and positives == data.positives()
    assert len(results) == len(queries) and all(len(r) == 5 and all(f in data.gallery_files for f in r) for r in results)
    assert np.array_equal(vis_scores, scores.cpu().numpy())
    assert results == [[data.gallery_files[j] for j in row] for row in ids.cpu().tolist()]


def test_extract_face_names_and_features(lib):
    """FeatureExtractor.extract_face (models/faceX/face_model.py:93-118): keys "<parent dir>/<file>", values = the rows
    extract_cbir_device returns for the same tensors."""
    from visiondk_b200.backbone import TimmWrapper
    from visiondk_b200.cbir import FeatureExtractor
    model = TimmWrapper("toy", 32, SIZE, pretrained=False, depths=(1, 1, 1, 1), dims=(64, 64, 128, 128)).cuda().eval()
    gen = torch.Generator().manual_seed(3)
    batches = [torch.randn(n, 3, SIZE, SIZE, generator=gen) for n in (4, 3)]
    paths = [[f"/data/lfw/person_{i}/img_{j}.jpg" for j in range(b.shape[0])] for i, b in enumerate(batches)]
    ext = FeatureExtractor(model)
    got = ext.extract_face([(None, b, p) for b, p in zip(batches, paths)], "cuda")
    assert list(got) == [f"person_{i}/img_{j}.jpg" for i, b in enumerate(batches) for j in range(b.shape[0])]
    want = ext.extract_cbir_device(batches, "cuda").cpu().numpy()
    assert np.array_equal(np.stack(list(got.values())), want)
    assert np.allclose(np.linalg.norm(want, axis=1), 1.0, atol=1e-5)
    assert ext.extract_face([], "cuda") == {}


def test_face_task_pair_verification(lib, tmp_path):
    """engine/faceX/evaluation.py::valuate: (a) synthetic:// root -> a (mean, std) in range that beats chance on the
    identity-structured images; (b) a pair file over <root>/val/ images == the same protocol assembled by hand."""
    from PIL import Image
    from engine.faceX.evaluation import valuate as valuate_face
    from engine.cbir.folder import read_image
    from visiondk_b200.backbone import TimmWrapper
    from visiondk_b200.metrics import face_verification_accuracy
    model = TimmWrapper("toy", 32, SIZE, pretrained=False, depths=(1, 1, 1, 1), dims=(64, 64, 128, 128)).cuda().eval()
    cfg = {"root": "synthetic://cbir?ids=50&per_id=4&queries=10&noise=0.3", "nw": 2, "val": {"bs": 50, "augment": AUGMENT}}
    mean, std = valuate_face(model, cfg, "cuda", image_size=SIZE, n_pairs=600)
    assert 0.5 < mean <= 1.0 and 0.0 <= std < 0.2

    rng = np.random.default_rng(5)
    rel = []
    for i in range(8):
        proto = rng.integers(0, 256, (8, 8, 3), dtype=np.uint8)
        os.makedirs(tmp_path / "val" / f"p{i}")
        for j in range(3):
            w, h = int(rng.integers(40, 100)), int(rng.integers(40, 100))
            img = np.asarray(Image.fromarray(proto).resize((w, h), Image.NEAREST)).astype(np.int16)
            Image.fromarray(np.clip(img + rng.integers(-25, 26, img.shape), 0, 255).astype(np.uint8)).save(tmp_path / "val" / f"p{i}" / f"{j}.png")
            rel.append(f"p{i}/{j}.png")
    pairs = []
    for n in range(40):  # 10 folds of 4: two genuine, two impostor
        i = int(rng.integers(0, 8))
        if n % 4 < 2:
            a, b = rng.choice(3, 2, replace=False)
            pairs.append((f"p{i}/{a}.png", f"p{i}/{b}.png", 1))
        else:
            o = int((i + 1 + rng.integers(0, 7)) % 8)
            pairs.append((f"p{i}/{int(rng.integers(0, 3))}.png", f"p{o}/{int(rng.integers(0, 3))}.png", 0))
    (tmp_path / "pairs.txt").write_text("\n".join(f"{a} {b} {l}" for a, b, l in pairs) + "\n")
    cfg = {"root": str(tmp_path), "nw": 2, "val": {"bs": 7, "pair_txt": str(tmp_path / "pairs.txt"), "augment": AUGMENT}}
    got = valuate_face(model, cfg, "cuda", image_size=SIZE)

    used = sorted({p for a, b, _ in pairs for p in (a, b)})
    chunks = []
    for a in range(0, len(used), 7):  # same batches as the loader: distinct images in np.unique order, 7 at a time
        x = np.stack([P.resize_pad_normalize(read_image(str(tmp_path / "val" / r)), SIZE) for r in used[a:a + 7]])
        chunks.append(model.embed(torch.from_numpy(x).cuda(), l2_normalize=True))
    feats, row = torch.cat(chunks), {r: i for i, r in enumerate(used)}
    ia = torch.tensor([row[a] for a, _, _ in pairs], device="cuda")
    ib = torch.tensor([row[b] for _, b, _ in pairs], device="cuda")
    scores = (feats[ia] * feats[ib]).sum(dim=1)
    want = face_verification_accuracy(scores, torch.tensor([l for _, _, l in pairs], device="cuda"))
    assert got == want
