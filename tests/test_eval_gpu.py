"""GPU: Omni3DEval (c3d_eval_match / c3d_eval_accumulate) equals the reference's own evaluator run
(tests/golden/omni3d_eval_golden.npz) and the numpy oracle bit for bit: evalImgs, precision / recall / scores tables,
stats and log strings; device-resident Instances evaluate like their COCO-result dicts; launches and copies do not
grow with the number of images."""
import json
import os
import sys

import numpy as np
import pytest
import torch

from oracle import omni3d_eval_oracle as oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import evalgen  # noqa: E402

CASES = [("2D", False), ("2D", True), ("3D", False), ("3D", True)]


@pytest.fixture(scope="module")
def golden():
    z = np.load(os.path.join(ROOT, "tests/golden/omni3d_eval_golden.npz"))
    return {k: z[k] for k in z.files}


def _run(gt, res, mode, prox):
    from omni3d_b200.evaluation import Omni3DEval
    e = Omni3DEval(gt, mode, prox)
    e.add_results(res)
    e.evaluate()
    e.accumulate()
    return e, e.summarize()


def _assert_eval_equal(e, log, prec, rec, sc, stats, want_log):
    assert np.array_equal(e.eval["precision"], prec)
    assert np.array_equal(e.eval["recall"], rec)
    assert np.array_equal(e.eval["scores"], sc)
    assert np.array_equal(e.stats, stats)
    assert log == want_log


@pytest.mark.parametrize("mode,prox", CASES)
def test_kernels_equal_reference_golden(golden, mode, prox):
    gt, res = json.loads(str(golden["A_gt"])), json.loads(str(golden["A_res"]))
    e, log = _run(gt, res, mode, prox)
    pre = f"A_{mode}{'_prox' if prox else ''}_"
    for k, v in oracle.flatten_eval_imgs(e.eval_imgs()).items():
        assert np.array_equal(v, golden[pre + "evalImgs_" + k]), k
    _assert_eval_equal(e, log, golden[pre + "precision"], golden[pre + "recall"], golden[pre + "scores"],
                       golden[pre + "stats"], str(golden[pre + "log"]))


@pytest.mark.parametrize("mode", ["2D", "3D"])
def test_concat_equals_reference_golden(golden, mode):
    from omni3d_b200.evaluation import Omni3DEval
    evs = []
    for s in ("A", "B"):
        e, _ = _run(json.loads(str(golden[s + "_gt"])), json.loads(str(golden[s + "_res"])), mode, False)
        evs.append(e)
    c = Omni3DEval.concat(evs, [int(x) for x in golden[f"AB_{mode}_cat_ids"]])
    log = c.summarize()
    _assert_eval_equal(c, log, *[golden[f"AB_{mode}_{k}"] for k in ("precision", "recall", "scores", "stats")],
                       str(golden[f"AB_{mode}_log"]))


@pytest.fixture(scope="module")
def big():
    return evalgen.make_set(1500, 10, seed=7)


@pytest.mark.parametrize("mode,prox", CASES)
def test_kernels_equal_oracle_randomized(big, mode, prox):
    gt, res = big
    e, log = _run(gt, res, mode, prox)
    p, ev = oracle.evaluate(gt, oracle.load_res(gt, res), mode, prox)
    got, want = oracle.flatten_eval_imgs(e.eval_imgs()), oracle.flatten_eval_imgs(ev)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
    prec, rec, sc = oracle.accumulate(p, oracle.per_cat_area(p, ev))
    stats, want_log = oracle.summarize(p, prec, rec)
    _assert_eval_equal(e, log, prec, rec, sc, stats, want_log)
    assert e.results([f"c{i}" for i in range(10)]) == pytest.approx(
        oracle.derive_results(stats, prec, mode, [f"c{i}" for i in range(10)]), nan_ok=True, rel=0, abs=0)
    e2, log2 = _run(gt, res, mode, prox)                       # two runs are identical
    assert log2 == log and np.array_equal(e2.eval["precision"], e.eval["precision"])


def test_concat_equals_oracle_randomized():
    from omni3d_b200.evaluation import Omni3DEval
    sets = [evalgen.make_set(300, 6, seed=11), evalgen.make_set(200, 4, seed=12, img0=5000, ann0=90000)]
    for mode in ("2D", "3D"):
        evs, per = [], {}
        for gt, res in sets:
            evs.append(_run(gt, res, mode, False)[0])
            p, ev = oracle.evaluate(gt, oracle.load_res(gt, res), mode)
            for key, item in oracle.per_cat_area(p, ev).items():
                per.setdefault(key, [])
                per[key] += item
        cat_ids = sorted({k for k, _ in per})[::-1]               # any explicit order, as summarize_all passes a set's
        c = Omni3DEval.concat(evs, cat_ids)
        prec, rec, sc = oracle.accumulate(oracle.Params(mode), per, cat_ids)
        stats, want_log = oracle.summarize(oracle.Params(mode), prec, rec)
        _assert_eval_equal(c, c.summarize(), prec, rec, sc, stats, want_log)


def test_add_instances_from_model_inference_equals_add_results():
    from omni3d_b200 import cubercnn as pc
    from omni3d_b200 import synth
    from omni3d_b200.evaluation import Omni3DEval
    torch.manual_seed(0)
    model = pc.build_model(pc.load_cfg("cubercnn_DLA34_FPN.yaml", ["MODEL.WEIGHTS_PRETRAIN", "none"])).eval()
    items = synth.make_batch(2, 128, 192, with_gt=False, seed=3)
    with torch.no_grad():
        out = model(items)
    inst = [o["instances"] for o in out]
    assert sum(len(x) for x in inst) > 0
    K = int(max(int(x.pred_classes.max()) for x in inst if len(x))) + 1
    cmap = [(-1 if c % 5 == 4 else 10 + 3 * c) for c in range(K)]     # some classes dropped, as _eval_predictions does
    gt, _ = evalgen.make_set(2, K, seed=5)
    gt["categories"] = [c for i, c in enumerate(gt["categories"]) if i % 3 != 2]   # and some not in the dataset
    cats = {c["id"] for c in gt["categories"]}
    gt["annotations"] = [a for a in gt["annotations"] if a["category_id"] in cats]
    # the instances_to_coco_json form of the same outputs, with the dropped classes removed before loadRes
    res = []
    for j, x in enumerate(inst):
        r = oracle.instances_to_results(j + 1, x.pred_boxes.tensor.cpu().numpy(), x.scores.cpu().numpy(),
                                        x.pred_classes.cpu().numpy(), x.pred_bbox3D.cpu().numpy())
        for d in r:
            if cmap[d["category_id"]] >= 0:
                d["category_id"] = cmap[d["category_id"]]
                res.append(d)
    for mode in ("2D", "3D"):
        a = Omni3DEval(gt, mode)
        a.add_instances([1, 2], inst, cmap)
        b = Omni3DEval(gt, mode)
        b.add_results(res)
        for e in (a, b):
            e.evaluate(); e.accumulate()
        la, lb = a.summarize(), b.summarize()
        assert la == lb
        ga, gb = a._s.groups(100), b._s.groups(100)
        for k in ("id", "score", "box", "area", "depth", "box3d", "img", "cat"):
            assert torch.equal(ga[k], gb[k]), k
        for k in ("precision", "recall", "scores"):
            assert np.array_equal(a.eval[k], b.eval[k])


def _count_work(n_img):
    from omni3d_b200 import _lib
    from omni3d_b200.evaluation import Omni3DEval
    gt, res = evalgen.make_set(n_img, 6, seed=21, quirks=False)
    e2 = Omni3DEval(gt, "2D")
    e2.add_results(res)
    e3 = e2.for_mode("3D")
    torch.cuda.synchronize()
    n0 = _lib.LAUNCHES["n"]
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for e in (e2, e3):
            e.evaluate(); e.accumulate(); e.summarize()
        torch.cuda.synchronize()
    names = [ev.name for ev in prof.events()]
    copies = sum(1 for n in names if "Memcpy" in n and ("HtoD" in n or "DtoH" in n))
    evals = sum(1 for n in names if "eval_match" in n or "eval_accumulate" in n)
    return _lib.LAUNCHES["n"] - n0, copies, evals


def test_launches_and_copies_do_not_grow_with_images():
    small, large = _count_work(100), _count_work(800)
    assert small[0] == large[0] and small[1] == large[1], (small, large)
    assert small[2] == large[2] == 4
