"""Generates tests/golden/omni3d_eval_golden.npz by EXECUTING THE REFERENCE'S OWN Omni3Deval.evaluate / accumulate /
summarize (cubercnn/evaluation/omni3d_evaluation.py:1092-1705) and summarize_all's re-accumulation (:378-447) from a
checkout of the original project (the location make_iou_golden.REF names).

The module is loaded with make_iou_golden's stubs (pytorch3d._C.iou_box3d bound to oracle/iou3d_oracle.c); on top of
that pycocotools' maskUtils.iou is bound to the oracle's bbIou restatement, np.float (gone in NumPy 2) to float, and the
COCO objects are a small fake with getImgIds / getCatIds / getAnnIds / loadAnns in pycocotools' order.  Detections go
through the oracle's restatement of COCO.loadRes.

Needs that checkout:   python tests/golden/make_eval_golden.py
"""
import copy
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

from make_iou_golden import load_reference_eval  # noqa: E402
from oracle import omni3d_eval_oracle as oracle  # noqa: E402
import evalgen  # noqa: E402

CASES = [("2D", False), ("2D", True), ("3D", False), ("3D", True)]


class FakeCOCO:
    def __init__(self, dataset):
        self.dataset = dataset
        self.anns = {a["id"]: a for a in dataset["annotations"]}
        self.imgToAnns = {}
        for a in dataset["annotations"]:
            self.imgToAnns.setdefault(a["image_id"], []).append(a)

    def getImgIds(self):
        return [im["id"] for im in self.dataset["images"]]

    def getCatIds(self):
        return [c["id"] for c in self.dataset["categories"]]

    def getAnnIds(self, imgIds=(), catIds=()):
        anns = [a for i in imgIds if i in self.imgToAnns for a in self.imgToAnns[i]]
        return [a["id"] for a in anns if a["category_id"] in catIds]

    def loadAnns(self, ids):
        return [self.anns[i] for i in ids]


def run_reference(ref, gt, results, mode, prox):
    cgt = FakeCOCO(copy.deepcopy(gt))
    cdt = FakeCOCO({"images": gt["images"], "annotations": oracle.load_res(gt, results)})
    e = ref.Omni3Deval(cgt, cdt, iouType="bbox", mode=mode, eval_prox=prox)
    e.evaluate()
    e.accumulate()
    log = e.summarize()
    return e, log


def reaccumulate(ref, evals, mode, cat_ids, img_ids):
    """summarize_all: the per-dataset evals_per_cat_area concatenated in dataset order, accumulated over cat_ids."""
    per = {}
    for e in evals:
        for key, item in e.evals_per_cat_area.items():
            per.setdefault(key, [])
            per[key] += item
    ev = ref.Omni3Deval(mode=mode)
    ev.params.catIds = list(cat_ids)
    ev.params.imgIds = list(img_ids)
    ev.evalImgs = True
    ev.evals_per_cat_area = per
    ev._paramsEval = copy.deepcopy(ev.params)
    ev.accumulate()
    return ev, ev.summarize()


def store(out, prefix, e, log):
    out[prefix + "precision"] = e.eval["precision"]
    out[prefix + "recall"] = e.eval["recall"]
    out[prefix + "scores"] = e.eval["scores"]
    out[prefix + "stats"] = np.asarray(e.stats)
    out[prefix + "log"] = np.array(log)


def main():
    ref = load_reference_eval()
    np.float = float
    ref.maskUtils = types.SimpleNamespace(iou=lambda d, g, iscrowd: oracle.bb_iou(d, g))
    gtA, resA = evalgen.make_set(40, 5, seed=1)
    gtB, resB = evalgen.make_set(25, 4, seed=2, img0=1001, ann0=5001)
    gtB["categories"].append({"id": 99})                                 # a category only the second dataset has
    out = {"A_gt": np.array(json.dumps(gtA)), "A_res": np.array(json.dumps(resA)),
           "B_gt": np.array(json.dumps(gtB)), "B_res": np.array(json.dumps(resB))}
    for mode, prox in CASES:
        tag = f"{mode}{'_prox' if prox else ''}_"
        e, log = run_reference(ref, gtA, resA, mode, prox)
        store(out, "A_" + tag, e, log)
        for k, v in oracle.flatten_eval_imgs(e.evalImgs).items():
            out["A_" + tag + "evalImgs_" + k] = v
        print(mode, prox, "stats", np.round(e.stats, 4))
        if not prox:
            eB, _ = run_reference(ref, gtB, resB, mode, False)
            cat_ids = sorted({c["id"] for c in gtA["categories"]} | {c["id"] for c in gtB["categories"]})
            img_ids = [im["id"] for im in gtA["images"] + gtB["images"]]
            ec, logc = reaccumulate(ref, [e, eB], mode, cat_ids, img_ids)
            store(out, "AB_" + mode + "_", ec, logc)
            out["AB_" + mode + "_cat_ids"] = np.array(cat_ids)
    np.savez_compressed(os.path.join(ROOT, "tests/golden/omni3d_eval_golden.npz"), **out)
    print("wrote tests/golden/omni3d_eval_golden.npz")


if __name__ == "__main__":
    main()
