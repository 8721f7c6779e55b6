"""The configs/*.yaml surface (SURVEY.md §5, north_star "keeping the ... configs/*.yaml surface"): the reference's own
configs/faceX/{face,cbir}.yaml parse unchanged through engine.vision_engine.yaml_load and satisfy engine.vision_engine.check's
schema (utils/checks.py:225-229) once `data.root` points at data that exists here; the class-count assert (checks.py:111-143) fires
like the reference's.  The reference files are byte-for-byte copies kept as fixtures (tests/golden/ref_configs/,
oracle/make_golden.py::configs)."""
import copy
import os

import pytest

from engine.vision_engine import check, yaml_load
from visiondk_b200.backbone import BackboneFactory

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "tests", "golden", "ref_configs")


def test_own_config_passes_the_checks():
    cfgs = yaml_load(os.path.join(ROOT, "configs", "faceX", "cbir_convnext_b200.yaml"))
    check("cbir", cfgs)
    bad = copy.deepcopy(cfgs)
    bad["model"]["head"]["arcface"]["num_class"] = 999
    with pytest.raises(AssertionError, match="Number of classes mismatch"):
        check("cbir", bad)
    bad = copy.deepcopy(cfgs)
    bad["model"]["backbone"] = {"resnet50": bad["model"]["backbone"]["timm-convnext_base"]}
    with pytest.raises(ValueError, match="timm-ModelName"):
        check("cbir", bad)
    with pytest.raises(ValueError):
        check("classification", cfgs)


@pytest.mark.parametrize("name,task", [("cbir.yaml", "cbir"), ("face.yaml", "face")])
def test_reference_yaml_parses_unchanged_and_passes_the_schema(name, task):
    cfgs = yaml_load(os.path.join(REF, name))
    assert cfgs["model"]["task"] == task and set(cfgs) >= {"model", "data", "hyp"}
    head = next(iter(cfgs["model"]["head"].values()))
    # the file's data root (a HuggingFace id / a path on the author's machine) does not exist here: same config, synthetic data
    cfgs["data"]["root"] = f"synthetic://cbir?ids={head['num_class']}&per_id=2&queries=4"
    check(task, cfgs)
    # every yaml anchor / alias (image_size, feat_dim) resolved; optimizer / scheduler are the ones the B200 step implements
    assert cfgs["hyp"]["optimizer"][0] == "sgd" and cfgs["hyp"]["scheduler"] == "cosine_with_warm"
    key = next(iter(cfgs["model"]["backbone"]))
    assert key.startswith("timm-")
    # the backbone named by the file is a swin (not built); the factory refuses it loudly instead of substituting
    with pytest.raises(ValueError, match="not built for B200"):
        BackboneFactory(cfgs["model"]["backbone"]).get_backbone()
    # the same file with one of the architectures its own comments list builds through the same factory
    cfgs["model"]["backbone"] = {"timm-convnext_base.clip_laion2b_augreg_ft_in1k": {"pretrained": False, "image_size": 224,
                                                                                   "feat_dim": head["feat_dim"]}}
    m = BackboneFactory(cfgs["model"]["backbone"]).get_backbone()
    assert m.model_name == "convnext_base" and m.feat_dim == head["feat_dim"]


def test_shipped_face_config_passes_the_schema():
    """configs/faceX/face_convnext_b200.yaml: the face task (BASELINE config 2) with the reference's val transform list."""
    from engine.cbir.folder import parse_val_augment
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cfgs = yaml_load(os.path.join(here, "configs", "faceX", "face_convnext_b200.yaml"))
    check("face", cfgs)
    assert cfgs["model"]["task"] == "face" and "arcface" in cfgs["model"]["head"]
    assert parse_val_augment(cfgs["data"]["val"]["augment"]) == (224, (0.485, 0.456, 0.406), (0.229, 0.224, 0.225))
    with pytest.raises(ValueError):
        check("cbir", cfgs)
