"""CPU tests: pin oracle/cubercnn_oracle against the fixture produced by running the reference's own
cubercnn code (tests/golden/make_model_golden.py): same-seed init, losses, logged scalars, gradient
norms, unused parameters and inference detections."""
import os

import pytest
import torch

from omni3d_b200 import synth
from oracle import cubercnn_oracle as co
from oracle import model_io

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = torch.load(os.path.join(ROOT, "tests/golden/model_golden.pt"), weights_only=False)
CASES = {"dla34": ("cubercnn_DLA34_FPN.yaml", (128, 160)), "resnet34": ("cubercnn_ResNet34_FPN.yaml", (128, 128))}
# torch's CPU reductions and convolutions split their work by thread count, which moves results in the last bits; the
# fixture's bit-exact values were produced with this many threads (make_model_golden.py), whatever the core count here
FIXTURE_THREADS = 8


@pytest.fixture
def fixture_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(FIXTURE_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", ["dla34", "resnet34"])
def test_oracle_matches_reference_run(name, fixture_threads):
    from detectron2.utils.events import EventStorage
    cfg_file, (H, W) = CASES[name]
    g = GOLD[name]
    cfg = co.load_cfg(cfg_file)
    torch.manual_seed(0)
    model = co.build_model(cfg)
    sd = model.state_dict()
    assert set(sd) == set(g["init_sum"]), "state_dict key names differ from the reference"
    assert sum(p.numel() for p in model.parameters()) == g["n_params"]
    for k, v in sd.items():   # same-seed init is bit-identical
        assert float(v.double().sum()) == g["init_sum"][k] and float(v.double().abs().sum()) == g["init_abs"][k], k
    model.train()
    torch.manual_seed(123)
    with EventStorage(0) as st:
        losses = model(model_io.to_d2_inputs(synth.make_batch(2, H, W, num_gt=4, seed=1)))
        sum(losses.values()).backward()
        scalars = st.latest()
    assert list(losses) == list(g["losses"])
    for k in losses:
        assert torch.equal(losses[k].detach(), g["losses"][k]), k
    assert scalars == g["scalars"]
    assert sorted(n for n, p in model.named_parameters() if p.grad is None) == g["no_grad"]
    for n, p in model.named_parameters():
        if p.grad is not None:
            ref = g["grad_norm"][n]
            assert abs(float(p.grad.double().norm()) - ref) <= 1e-4 * ref + 1e-7, n
    model.eval()
    with torch.no_grad():
        res = model(model_io.to_d2_inputs(synth.make_batch(2, H, W, with_gt=False, seed=3)))
    for r, d in zip(res, g["detections"]):
        f = r["instances"].get_fields()
        assert set(f) == set(d)
        for k, v in f.items():
            assert torch.equal(v.tensor if hasattr(v, "tensor") else v, d[k]), k


@pytest.mark.parametrize("src", ["repo", "reference"])
def test_config_surface(src):
    """the flattened repo config and the reference's own YAML chain (the values it loads to, stored by
    tests/golden/make_config_golden.py) agree on the model path"""
    path = "cubercnn_DLA34_FPN.yaml"
    if src == "reference":
        path = os.path.join(ROOT, "tests/golden/reference_cubercnn_DLA34_FPN.yaml")
    cfg = co.load_cfg(path)
    if src == "reference":
        repo = co.load_cfg("cubercnn_DLA34_FPN.yaml")
        for sec in ("MODEL", "INPUT", "SOLVER"):
            assert cfg[sec] == repo[sec], sec
    assert cfg.MODEL.META_ARCHITECTURE == "RCNN3D" and cfg.MODEL.ROI_HEADS.NUM_CLASSES == 50
    assert cfg.MODEL.BACKBONE.NAME == "build_dla_from_vision_fpn_backbone"
    assert cfg.MODEL.RPN.IOU_THRESHOLDS == [0.05, 0.05] and cfg.MODEL.ROI_CUBE_HEAD.VIRTUAL_FOCAL == 512.0
    assert cfg.SOLVER.IMS_PER_BATCH == 192 and cfg.SOLVER.STEPS == (69600, 92800)
