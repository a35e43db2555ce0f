"""CPU: the numpy restatement of the Omni3D evaluator (oracle/omni3d_eval_oracle.py) equals the reference's own
Omni3Deval run (tests/golden/omni3d_eval_golden.npz, generator make_eval_golden.py) bit for bit; Omni3DEval's
result-dict converter and group construction equal the oracle's grouping; the new C entry points reject bad arguments
before any CUDA call."""
import ctypes
import json
import os

import numpy as np
import pytest

from oracle import omni3d_eval_oracle as oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = [("2D", False), ("2D", True), ("3D", False), ("3D", True)]


@pytest.fixture(scope="module")
def golden():
    z = np.load(os.path.join(ROOT, "tests/golden/omni3d_eval_golden.npz"))
    return {k: z[k] for k in z.files}


def _tag(mode, prox):
    return f"{mode}{'_prox' if prox else ''}_"


@pytest.mark.parametrize("mode,prox", CASES)
def test_oracle_equals_reference_run(golden, mode, prox):
    gt, res = json.loads(str(golden["A_gt"])), json.loads(str(golden["A_res"]))
    p, ev = oracle.evaluate(gt, oracle.load_res(gt, res), mode, prox)
    pre = "A_" + _tag(mode, prox)
    for k, v in oracle.flatten_eval_imgs(ev).items():
        assert np.array_equal(v, golden[pre + "evalImgs_" + k]), k
    prec, rec, sc = oracle.accumulate(p, oracle.per_cat_area(p, ev))
    assert np.array_equal(prec, golden[pre + "precision"])
    assert np.array_equal(rec, golden[pre + "recall"])
    assert np.array_equal(sc, golden[pre + "scores"])
    assert (prec == -1).all(axis=(0, 1, 3, 4))[-1]               # the category without GTs keeps the -1 tables
    stats, log = oracle.summarize(p, prec, rec)
    assert np.array_equal(stats, golden[pre + "stats"])
    assert log == str(golden[pre + "log"])


@pytest.mark.parametrize("mode", ["2D", "3D"])
def test_oracle_concatenation_equals_reference(golden, mode):
    per, img_ids = {}, []
    for s in ("A", "B"):
        gt, res = json.loads(str(golden[s + "_gt"])), json.loads(str(golden[s + "_res"]))
        p, ev = oracle.evaluate(gt, oracle.load_res(gt, res), mode)
        for key, item in oracle.per_cat_area(p, ev).items():
            per.setdefault(key, [])
            per[key] += item
    cat_ids = [int(c) for c in golden[f"AB_{mode}_cat_ids"]]
    p = oracle.Params(mode)
    prec, rec, sc = oracle.accumulate(p, per, cat_ids)
    for k, v in (("precision", prec), ("recall", rec), ("scores", sc)):
        assert np.array_equal(v, golden[f"AB_{mode}_{k}"]), k
    stats, log = oracle.summarize(p, prec, rec)
    assert np.array_equal(stats, golden[f"AB_{mode}_stats"]) and log == str(golden[f"AB_{mode}_log"])


def test_golden_covers_the_quirks(golden):
    gt, res = json.loads(str(golden["A_gt"])), json.loads(str(golden["A_res"]))
    assert any(a["id"] == 0 for a in gt["annotations"])
    assert any(a.get("ignore2D") for a in gt["annotations"]) and any(a.get("ignore3D") for a in gt["annotations"])
    assert {a["depth"] for a in gt["annotations"]} >= {10.0, 35.0}
    assert {a["area"] for a in gt["annotations"]} >= {32.0 ** 2, 96.0 ** 2}
    signs = {np.copysign(1, r["score"]) for r in res if r["score"] == 0}
    assert signs == {1.0, -1.0}
    per = {}
    for r in res:
        per[r["image_id"], r["category_id"]] = per.get((r["image_id"], r["category_id"]), 0) + 1
    assert max(per.values()) > 100
    gts = {(a["image_id"], a["category_id"]) for a in gt["annotations"]}
    assert set(per) - gts and gts - set(per)                     # groups with only detections / only GTs
    ev = golden["A_2D_evalImgs_dtMatches"]
    assert (ev > 0).any()


def test_numpy_mean_of_eight_is_the_pairwise_tree():
    import torch
    from omni3d_b200.evaluation import _pairwise_mean8
    rng = np.random.default_rng(0)
    b = (rng.standard_normal((20000, 8)) * np.exp(rng.uniform(-30, 30, (20000, 8)))).astype(np.float32)
    want = np.array([np.array(x.tolist()).mean() for x in b])
    got = _pairwise_mean8(torch.from_numpy(b).double()).numpy()
    assert np.array_equal(got, want)


@pytest.mark.parametrize("mode", ["2D", "3D"])
def test_result_conversion_and_groups_equal_oracle(golden, mode):
    """add_results + the group construction (stable -score order, ties in results order, +-0 tie, truncation to 100)
    give every (image, category) group the detections the oracle's evaluateImg sees, in the same order."""
    from omni3d_b200.evaluation import Omni3DEval
    gt, res = json.loads(str(golden["A_gt"])), json.loads(str(golden["A_res"]))
    e = Omni3DEval(gt, mode, device="cpu")
    e.add_results(res[:70])
    e.add_results(res[70:])
    g = e._s.groups(100)
    p, ev = oracle.evaluate(gt, oracle.load_res(gt, res), mode)
    I = len(p.imgIds)
    off = g["dt_off"].numpy()
    ids = g["id"].numpy()
    for k, cat in enumerate(p.catIds):
        for i, img in enumerate(p.imgIds):
            want = ev[k * len(p.areaRng) * I + i]
            got = ids[off[k * I + i]:off[k * I + i + 1]].tolist()
            assert got == (want["dtIds"] if want is not None else []), (img, cat)
            if want is not None:
                s = g["score"].numpy()[off[k * I + i]:off[k * I + i + 1]]
                assert np.array_equal(s, np.asarray(want["dtScores"], np.float64))
    rng = "area" if mode == "2D" else "depth"
    res_ids = oracle.load_res(gt, res)
    by_id = {r["id"]: r for r in res_ids}
    assert np.array_equal(g[rng].numpy(), np.array([by_id[i][rng] for i in ids], np.float64))
    assert np.array_equal(g["box"].numpy(), np.array([by_id[i]["bbox"] for i in ids], np.float64))


def test_eval_entry_points_reject_bad_arguments_without_gpu():
    from omni3d_b200 import _lib
    from omni3d_b200.evaluation import _bind_eval
    L = _bind_eval()
    L.c3d_last_error.restype = ctypes.c_char_p
    p = ctypes.c_void_p(256)
    start, rng = (ctypes.c_double * 16)(), (ctypes.c_double * 16)()
    assert L.c3d_eval_match_workspace_bytes(100, 4, 10) == 4000
    args = [p] * 10
    rc = L.c3d_eval_match(0, 0, 4, 9, 10, *args, 10, 10, start, rng, 0.3, p, p, p, p, 4000, None)
    assert rc == _lib.C3D_EINVAL and b"eval_match" in L.c3d_last_error()
    rc = L.c3d_eval_match(1, 0, 4, 4, 10, *args[:8], None, None, 10, 10, start, rng, 0.3, p, p, p, p, 4000, None)
    assert rc == _lib.C3D_EINVAL and b"3D mode" in L.c3d_last_error()
    rc = L.c3d_eval_match(0, 0, 4, 4, 10, *args, 10, 10, start, rng, 0.3, p, p, p, p, 10, None)
    assert rc == _lib.C3D_EWORKSPACE
    rc = L.c3d_eval_accumulate(5, 4, 10, 7, 101, *[p] * 7, 10, p, p, p, p, p, None)
    assert rc == _lib.C3D_EINVAL and b"T * M" in L.c3d_last_error()
    rc = L.c3d_eval_accumulate(5, 4, 10, 3, 101, None, *[p] * 6, 10, p, p, p, p, p, None)
    assert rc == _lib.C3D_EINVAL and b"null" in L.c3d_last_error()
    with pytest.raises(_lib.C3DError):
        _lib.check(rc)


def test_use_cats_zero_is_not_supported():
    from omni3d_b200.evaluation import Omni3DEval
    e = Omni3DEval({"images": [{"id": 1}], "categories": [{"id": 1}], "annotations": []}, device="cpu")
    e.params.useCats = 0
    with pytest.raises(NotImplementedError):
        e.evaluate()
