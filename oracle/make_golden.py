"""Generates tests/golden/*.npz by executing the REFERENCE's own modules, and copies its two faceX configs there as fixtures.

    python oracle/make_golden.py            # needs /root/reference; never runs on the GPU box

The reference package cannot be imported as a whole (timm / faiss / torchmetrics are not installed), so the
torch-only files are loaded by path: models/faceX/head/{arcface,circleloss}.py, models/losses/loss.py,
models/ema.py, engine/scheduler.py, engine/optimizer.py, dataset/transforms.py (the eval-time input pipeline, built from the
reference's own configs/faceX/cbir.yaml), and models/faceX/backbone/timm_wrapper.py (the neck) around a stub `timm`.  The committed .npz files are what the CPU tests
hold oracle/ to; the GPU tests then hold the CUDA kernels to oracle/.
"""
from __future__ import annotations

import importlib.util
import os
import sys

import numpy as np
import torch

REF = "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def load(rel, name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def heads():
    arc = load("models/faceX/head/arcface.py", "ref_arcface")
    cir = load("models/faceX/head/circleloss.py", "ref_circleloss")
    loss = load("models/losses/loss.py", "ref_loss")
    for name, B, D, Cn, smooth in (("small", 8, 64, 40, 0.0), ("cfg", 24, 512, 160, 0.1)):
        torch.manual_seed(7)
        feats = torch.randn(B, D) * 3.0
        labels = torch.randint(0, Cn, (B,))
        out = {"feats": feats.numpy(), "labels": labels.numpy(), "label_smooth": np.float32(smooth)}
        for kind, mod, kwargs in (("arcface", arc.ArcFace, dict(margin_arc=0.35, margin_am=0.0, scale=32)),
                                  ("arcface_am", arc.ArcFace, dict(margin_arc=0.5, margin_am=0.2, scale=64)),
                                  ("circleloss", cir.CircleLoss, dict(margin=0.25, gamma=256))):
            torch.manual_seed(11)
            head = mod(D, Cn, **kwargs)
            if kind == "arcface_am":
                # make a few rows hit the theta+m > pi fallback branch (cos <= cos(pi - m))
                # (not exactly cos = -1: the reference's sqrt(1 - cos^2) has a NaN gradient there)
                with torch.no_grad():
                    gen = torch.Generator().manual_seed(5)
                    for r in range(0, B, 3):
                        noise = torch.randn(D, generator=gen) * feats[r].norm() / D ** 0.5
                        head.weight[:, labels[r]] = -feats[r] + 0.3 * noise
            f = feats.clone().requires_grad_(True)
            logits = head(f, labels)
            crit = loss.create_Lossfn("ce")(label_smooth=smooth)
            l = crit(logits, labels)
            l.backward()
            out[f"{kind}_weight"] = head.weight.detach().numpy().copy()
            out[f"{kind}_logits"] = logits.detach().numpy()
            out[f"{kind}_loss"] = l.detach().numpy()
            out[f"{kind}_dfeats"] = f.grad.numpy().copy()
            out[f"{kind}_dweight"] = head.weight.grad.numpy().copy()
        np.savez_compressed(os.path.join(OUT, f"heads_{name}.npz"), **out)


def heads_mv():
    mv = load("models/faceX/head/mv_softmax.py", "ref_mv_softmax")
    loss = load("models/losses/loss.py", "ref_loss")
    B, D, Cn, smooth = 16, 64, 40, 0.1
    torch.manual_seed(17)
    feats = torch.randn(B, D) * 2.0
    labels = torch.randint(0, Cn, (B,))
    out = {"feats": feats.numpy(), "labels": labels.numpy(), "label_smooth": np.float32(smooth)}
    for kind, kwargs in (("mv_arc", dict(is_am=False, margin=0.35, mv_weight=1.12, scale=32)),
                         ("mv_am", dict(is_am=True, margin=0.35, mv_weight=1.12, scale=32))):
        torch.manual_seed(19)
        head = mv.MV_Softmax(D, Cn, **kwargs)
        with torch.no_grad():  # pull some class centres towards their samples so that both gt > 0 / gt > margin branches occur
            for r in range(0, B, 2):
                head.weight[:, labels[r]] = feats[r] / feats[r].norm() + 0.4 * head.weight[:, labels[r]]
        f = feats.clone().requires_grad_(True)
        logits = head(f, labels)
        l = loss.create_Lossfn("ce")(label_smooth=smooth)(logits, labels)
        l.backward()
        out[f"{kind}_weight"] = head.weight.detach().numpy().copy()
        out[f"{kind}_logits"] = logits.detach().numpy()
        out[f"{kind}_loss"] = l.detach().numpy()
        out[f"{kind}_dfeats"] = f.grad.numpy().copy()
        out[f"{kind}_dweight"] = head.weight.grad.numpy().copy()
    np.savez_compressed(os.path.join(OUT, "heads_mv.npz"), **out)


def cbir_metrics():
    """The reference's own CBIRMetrics / compute_metrics (engine/cbir/evaluation.py:14-224), executed from their source text (the
    module itself cannot be imported: it pulls in faiss / timm / dataset code at import time), on a synthetic retrieval result."""
    import ast
    from sklearn.metrics import ndcg_score, roc_auc_score
    src = open(os.path.join(REF, "engine/cbir/evaluation.py")).read()
    tree = ast.parse(src)
    ns = {"np": np, "roc_auc_score": roc_auc_score, "ndcg_score": ndcg_score}
    for node in tree.body:
        if (isinstance(node, ast.ClassDef) and node.name == "CBIRMetrics") or \
           (isinstance(node, ast.FunctionDef) and node.name == "compute_metrics"):
            exec(compile(ast.Module(body=[node], type_ignores=[]), "evaluation.py", "exec"), ns)
    rng = np.random.default_rng(23)
    nq, ng, k = 40, 400, 10
    gal_label = rng.integers(0, 25, ng)                      # identity of every gallery item
    q_label = rng.integers(0, 25, nq)
    for c in range(25):                                      # every identity has at least two gallery items
        gal_label[2 * c], gal_label[2 * c + 1] = c, c
    scores = np.sort(rng.random((nq, k)).astype(np.float32), axis=1)[:, ::-1].copy()
    scores[3, 2] = scores[3, 3] = scores[3, 4]               # tied scores: sklearn's tie-averaged DCG / AUC paths
    scores[7, 0] = scores[7, 1]
    ids = np.stack([rng.choice(ng, k, replace=False) for _ in range(nq)]).astype(np.int64)
    for q in range(0, nq, 3):                                # plant some hits
        pos = np.flatnonzero(gal_label == q_label[q])
        ids[q, rng.integers(0, k)] = pos[0]
        if len(pos) > 1 and pos[1] not in ids[q]:
            ids[q, rng.integers(0, k)] = pos[1]
    for q in range(nq):                                      # keep rows duplicate-free
        seen, row = set(), ids[q]
        for j in range(k):
            while row[j] in seen:
                row[j] = (row[j] + 1) % ng
            seen.add(row[j])
    names = np.array([f"gallery/{i:04d}.jpg" for i in range(ng)])
    preds = [names[row] for row in ids]
    labels = [list(names[np.flatnonzero(gal_label == q_label[q])]) for q in range(nq)]
    cutoffs = [1, 3, 10]
    metrics = ns["compute_metrics"](preds, scores, labels, metrics=["mrr", "precision", "recall", "auc", "ndcg"], cutoffs=cutoffs)
    np.savez_compressed(os.path.join(OUT, "cbir_metrics.npz"), ids=ids, scores=scores, gal_label=gal_label, q_label=q_label,
                        cutoffs=np.array(cutoffs), metric_names=np.array(list(metrics.keys())),
                        metric_values=np.array([float(v) for v in metrics.values()], dtype=np.float64))


def face_verification():
    """The reference's own Evaluator.test_one_model / getThreshold (engine/faceX/evaluation.py:34-113: LFW-style 10-fold threshold
    sweep over 6000 pairs), executed from its source text on synthetic unit features."""
    import ast
    src = open(os.path.join(REF, "engine/faceX/evaluation.py")).read()
    ns = {"np": np, "os": os}
    for node in ast.parse(src).body:
        if isinstance(node, ast.ClassDef) and node.name == "Evaluator":
            exec(compile(ast.Module(body=[node], type_ignores=[]), "evaluation.py", "exec"), ns)
    rng = np.random.default_rng(31)
    n_id, per_id, dim = 200, 4, 32
    centres = rng.standard_normal((n_id, dim))
    feats = centres[:, None, :] + 1.1 * rng.standard_normal((n_id, per_id, dim))
    feats = (feats / np.linalg.norm(feats, axis=-1, keepdims=True)).astype(np.float32).reshape(n_id * per_id, dim)
    names = [f"id{i // per_id:03d}/img{i % per_id}.jpg" for i in range(n_id * per_id)]
    pairs = []
    for fold in range(10):                      # 300 genuine + 300 impostor pairs per fold, as in the LFW protocol
        for j in range(600):
            a = int(rng.integers(0, n_id))
            if j < 300:
                i1, i2 = rng.choice(per_id, 2, replace=False)
                pairs.append((a * per_id + i1, a * per_id + i2, 1))
            else:
                b = int((a + 1 + rng.integers(0, n_id - 1)) % n_id)
                pairs.append((a * per_id + int(rng.integers(0, per_id)), b * per_id + int(rng.integers(0, per_id)), 0))
    pair_list = [[names[a], names[b], str(l)] for a, b, l in pairs]
    name2feat = {os.path.normpath(n): f for n, f in zip(names, feats)}
    mean, std = ns["Evaluator"](None).test_one_model(pair_list, name2feat)
    np.savez_compressed(os.path.join(OUT, "face_verification.npz"), feats=feats, pairs=np.array(pairs, dtype=np.int64),
                        mean=np.float64(mean), std=np.float64(std))


def neck():
    """The reference's OWN models/faceX/backbone/timm_wrapper.py (constructor logic, both neck branches, forward) executed
    around a stub `timm` module: `timm.create_model(name, pretrained=..., num_classes=0, global_pool='')` hands back the
    oracle's toy ConvNeXt / ViT body (timm itself is not installed: the body is the unpinned part, the wrapper and its
    BatchNorm2d/LayerNorm -> Flatten -> Linear -> BatchNorm1d neck are the reference's code, pinned here).  Stored: the
    wrapper's state_dict keys as the reference names them, the neck's tensors (the body is rebuilt from its seed), a batch, the body's feature map, the embeddings in eval mode, and in
    train mode the embeddings, the updated BatchNorm running statistics and the gradients of every neck parameter and of
    the feature map for loss = sum(out * w_out)."""
    import types
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from oracle.convnext import ConvNeXt, randomize_ as rand_cnx
    from oracle.vit import VisionTransformer, randomize_ as rand_vit
    calls = []

    def create_model(name, pretrained=False, num_classes=None, global_pool=None, **kw):
        calls.append((name, pretrained, num_classes, global_pool))
        assert num_classes == 0 and global_pool == "", "timm_wrapper.py:16-21 asks for the un-pooled, head-less body"
        if name == "convnext_toy":
            return ConvNeXt((1, 1, 2, 1), (64, 128, 128, 256))
        if name == "vit_toy":
            return VisionTransformer(64, 16, 128, 2, 2)
        raise ValueError(name)

    stub = types.ModuleType("timm")
    stub.create_model = create_model
    sys.modules["timm"] = stub
    try:
        ref = load("models/faceX/backbone/timm_wrapper.py", "ref_timm_wrapper")
    finally:
        del sys.modules["timm"]
    out = {}
    torch.manual_seed(41)
    x = torch.randn(6, 3, 64, 64)
    out["x"] = x.numpy()
    for tag, name, rand, seed in (("cnn", "convnext_toy", rand_cnx, 51), ("vit", "vit_toy", rand_vit, 52)):
        w = ref.TimmWrapper(name, feat_dim=64, image_size=64, pretrained=False)
        rand(w, seed=seed)
        sd = {k: v.detach().clone() for k, v in w.state_dict().items()}
        out[f"{tag}_keys"] = np.array(list(sd.keys()))
        out[f"{tag}_seed"] = np.int32(seed)  # the body is rebuilt from oracle.*.randomize_(wrapper, seed): deterministic
        out[f"{tag}_body_abs_sum"] = np.float64(sum(v.double().abs().sum().item() for k, v in sd.items() if k.startswith("model.")))
        for k, v in sd.items():
            if k.startswith("output_layer."):
                out[f"{tag}_sd/{k}"] = v.numpy()
        w.eval()
        with torch.no_grad():
            out[f"{tag}_feat"] = w.model(x).numpy()
            out[f"{tag}_eval"] = w(x).numpy()
        w.train()
        feat = w.model(x).detach().requires_grad_(True)
        y = w.output_layer(feat)
        g = torch.Generator().manual_seed(61)
        w_out = torch.randn(y.shape, generator=g)
        (y * w_out).sum().backward()
        out[f"{tag}_train"] = y.detach().numpy()
        out[f"{tag}_w_out"] = w_out.numpy()
        out[f"{tag}_dfeat"] = feat.grad.numpy()
        for k, p_ in w.output_layer.named_parameters():
            out[f"{tag}_grad/output_layer.{k}"] = p_.grad.numpy()
        for k, b in w.output_layer.named_buffers():
            out[f"{tag}_after/output_layer.{k}"] = b.detach().numpy()
    assert [c[0] for c in calls] == ["convnext_toy", "vit_toy"]
    np.savez_compressed(os.path.join(OUT, "neck_ref.npz"), **out)


def preprocess():
    """The reference's OWN eval-time input pipeline: dataset/transforms.py is loaded by path and its `create_AugTransforms`
    builds the val transform list of the reference's OWN configs/faceX/cbir.yaml (`data.val.augment`: resize_and_padding ->
    to_tensor -> normalize, transforms.py:325-365, 466-477, 530-555) at the config's image size and at two smaller sizes.
    Stored: the uint8 source images (seeded noise and smooth ramps, landscape / portrait / square / tiny / one-pixel-off
    shapes) and the float32 tensors the reference pipeline returns for them."""
    import yaml
    from PIL import Image
    ref = load("dataset/transforms.py", "ref_transforms")
    with open(os.path.join(REF, "configs/faceX/cbir.yaml")) as f:
        cfg = yaml.safe_load(f)
    augment = cfg["data"]["val"]["augment"]
    assert [list(a.keys())[0] for a in augment] == ["resize_and_padding", "to_tensor", "normalize"]
    cfg_size = int(augment[0]["resize_and_padding"]["size"])
    out = {"cfg_size": np.int32(cfg_size), "mean": np.array(augment[2]["normalize"]["mean"], np.float64),
           "std": np.array(augment[2]["normalize"]["std"], np.float64)}
    shapes = [(320, 240), (100, 300), (96, 96), (500, 37), (50, 60), (133, 200), (7, 5), (97, 96), (31, 97), (1, 1)]
    rng = np.random.default_rng(2025)
    n = 0
    for size, use in ((cfg_size, shapes[:2]), (96, shapes), (64, shapes[3:7])):  # kept small: the fixture is committed
        aug = [dict(a) for a in augment]
        aug[0] = {"resize_and_padding": {"size": size, "training": False}}
        pipeline = ref.create_AugTransforms(aug)
        for (w, h) in use:
            if n % 2 == 0:
                img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
            else:  # smooth content: exercises the fixed-point rounding differently from noise
                yy, xx = np.mgrid[0:h, 0:w]
                img = np.stack([(xx * 255 // max(w - 1, 1)), (yy * 255 // max(h - 1, 1)), ((xx + yy) * 7 % 256)], axis=2).astype(np.uint8)
            t = pipeline(Image.fromarray(img))
            assert tuple(t.shape) == (3, size, size) and t.dtype == torch.float32
            out[f"img{n}"] = img
            out[f"size{n}"] = np.int32(size)
            out[f"out{n}"] = t.numpy()
            n += 1
    out["count"] = np.int32(n)
    np.savez_compressed(os.path.join(OUT, "preprocess_ref.npz"), **out)


def configs():
    """The reference's own configs/faceX/{cbir,face}.yaml, byte for byte: tests/test_config_surface_cpu.py parses them through
    engine.vision_engine.yaml_load + check, tests/test_cbir_folder_cpu.py reads their val augment list."""
    import shutil
    os.makedirs(os.path.join(OUT, "ref_configs"), exist_ok=True)
    for name in ("cbir.yaml", "face.yaml"):
        shutil.copyfile(os.path.join(REF, "configs", "faceX", name), os.path.join(OUT, "ref_configs", name))


def ema_sgd_sched():
    ema_mod = load("models/ema.py", "ref_ema")
    sched = load("engine/scheduler.py", "ref_sched")
    torch.manual_seed(3)
    model = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.BatchNorm1d(5), torch.nn.Linear(5, 3))
    ema = ema_mod.ModelEMA(model)
    opt = torch.optim.SGD([{"params": model[0].parameters(), "lr": 0.01},
                           {"params": list(model[1].parameters()) + list(model[2].parameters()), "lr": 0.1}],
                          lr=0.01, momentum=0.8, weight_decay=5e-4)
    sc = sched.create_Scheduler("cosine_with_warm", opt, warm_ep=4, epochs=20, lr0=0.01, lrf_ratio=0.1)
    rec = {"init": np.concatenate([p.detach().numpy().ravel() for p in model.state_dict().values()])}
    xs, ys, lrs, params, emas, gnorms = [], [], [], [], [], []
    for step in range(12):
        x = torch.randn(16, 6)
        y = torch.randint(0, 3, (16,))
        lrs.append([g["lr"] for g in opt.param_groups])  # learning rates in effect during this step
        loss = torch.nn.functional.cross_entropy(model(x) * 30, y)
        loss.backward()
        gn = torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=10.0)  # train.py:209
        opt.step()
        opt.zero_grad()
        ema.update(model)  # train.py:214-215
        sc.step()          # train.py:230 (per batch)
        xs.append(x.numpy()); ys.append(y.numpy()); gnorms.append(float(gn))
        params.append(np.concatenate([p.detach().numpy().ravel() for p in model.state_dict().values()]))
        emas.append(np.concatenate([p.detach().numpy().ravel().astype(np.float32) for p in ema.ema.state_dict().values()]))
    np.savez_compressed(os.path.join(OUT, "step_sgd_ema.npz"), init=rec["init"], x=np.stack(xs), y=np.stack(ys),
                        lrs=np.array(lrs), params=np.stack(params), emas=np.stack(emas), gnorms=np.array(gnorms))


if __name__ == "__main__":
    if not os.path.isdir(REF):
        sys.exit("make_golden.py needs /root/reference (authoring container only)")
    os.makedirs(OUT, exist_ok=True)
    heads()
    heads_mv()
    cbir_metrics()
    face_verification()
    ema_sgd_sched()
    neck()
    preprocess()
    configs()
    print("golden vectors written to", OUT)
