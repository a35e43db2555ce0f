"""ORACLE (test infrastructure only): plain-numpy restatement of the Omni3D AP evaluator.

Restates Omni3Deval.evaluate / evaluateImg / accumulate / summarize (cubercnn/evaluation/omni3d_evaluation.py:1019-1087,
1140-1170, 1172-1313, 1315-1357, 1433-1705), _derive_omni_results (:764-840), the multi-dataset re-accumulation of
summarize_all (:378-447), instances_to_coco_json (:970-1013), and the pycocotools pieces the reference reaches without
vendoring them: COCO.loadRes (bbox branch: id = position + 1, area = w * h), getAnnIds / loadAnns order (image order,
then annotation order) and maskApi.c bbIou with iscrowd = 0.

GT datasets are COCO-style dicts {"images": [{"id"}], "categories": [{"id"}], "annotations": [...]} whose annotations
carry id, image_id, category_id, bbox (XYWH), bbox3D (8 x 3), area, depth and optionally ignore2D / ignore3D.
"""
import numpy as np

from . import iou3d


class Params:
    def __init__(self, mode="2D"):
        if mode == "2D":
            self.iouThrs = np.linspace(0.5, 0.95, int(np.round((0.95 - 0.5) / 0.05)) + 1, endpoint=True)
            self.areaRng = [[0 ** 2, 1e5 ** 2], [0 ** 2, 32 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]]
            self.areaRngLbl = ["all", "small", "medium", "large"]
        elif mode == "3D":
            self.iouThrs = np.linspace(0.05, 0.5, int(np.round((0.5 - 0.05) / 0.05)) + 1, endpoint=True)
            self.areaRng = [[0, 1e5], [0, 10], [10, 35], [35, 1e5]]
            self.areaRngLbl = ["all", "near", "medium", "far"]
        else:
            raise ValueError("mode %s not supported" % mode)
        self.recThrs = np.linspace(0.0, 1.00, int(np.round((1.00 - 0.0) / 0.01)) + 1, endpoint=True)
        self.maxDets = [1, 10, 100]
        self.imgIds, self.catIds = [], []
        self.mode = mode
        self.proximity_thresh = 0.3


def bb_iou(d, g):
    """maskApi.c bbIou(dt, gt, iscrowd=0) -> (len(d), len(g)) fp64, or [] when either side is empty (maskUtils.iou)."""
    d, g = np.asarray(d, np.float64).reshape(-1, 4), np.asarray(g, np.float64).reshape(-1, 4)
    if len(d) == 0 or len(g) == 0:
        return []
    o = np.zeros((len(d), len(g)))
    for j, G in enumerate(g):
        ga = G[2] * G[3]
        for i, D in enumerate(d):
            da = D[2] * D[3]
            w = min(D[2] + D[0], G[2] + G[0]) - max(D[0], G[0])
            if w <= 0:
                continue
            h = min(D[3] + D[1], G[3] + G[1]) - max(D[1], G[1])
            if h <= 0:
                continue
            i_ = w * h
            o[i, j] = i_ / (da + ga - i_)
    return o


def instances_to_results(image_id, boxes_xyxy, scores, classes, bbox3D):
    """instances_to_coco_json with BoxMode.convert(XYXY_ABS -> XYWH_ABS) restated on float32 arrays."""
    b = np.asarray(boxes_xyxy, np.float32).copy()
    b[:, 2] -= b[:, 0]
    b[:, 3] -= b[:, 1]
    boxes, sc, cl, b3 = b.tolist(), np.asarray(scores, np.float32).tolist(), np.asarray(classes).tolist(), \
        np.asarray(bbox3D, np.float32).tolist()
    return [{"image_id": image_id, "category_id": cl[k], "bbox": boxes[k], "score": sc[k],
             "depth": np.array(b3[k])[:, 2].mean(), "bbox3D": b3[k]} for k in range(len(boxes))]


def load_res(gt, results):
    """COCO.loadRes, bbox branch: copies of the result dicts with id = position + 1, area = w * h, iscrowd = 0."""
    img_set = {im["id"] for im in gt["images"]}
    assert {r["image_id"] for r in results} <= img_set, "Results do not correspond to current coco set"
    out = []
    for i, r in enumerate(results):
        r = dict(r)
        bb = r["bbox"]
        r["area"] = bb[2] * bb[3]
        r["id"] = i + 1
        r["iscrowd"] = 0
        out.append(r)
    return out


def _by_group(anns, img_ids, cat_ids):
    """getAnnIds(imgIds, catIds) + loadAnns order, bucketed by (image, category) like Omni3Deval._prepare."""
    by_img = {}
    for a in anns:
        by_img.setdefault(a["image_id"], []).append(a)
    cats = set(cat_ids)
    out = {}
    for i in img_ids:
        for a in by_img.get(i, []):
            if a["category_id"] in cats:
                out.setdefault((i, a["category_id"]), []).append(a)
    return out


def evaluate(gt, dts, mode, eval_prox=False, img_ids=None):
    """Omni3Deval.evaluate -> (params, evalImgs list in (category, range, image) order).  dts: load_res output."""
    p = Params(mode)
    p.imgIds = list(np.unique(img_ids if img_ids is not None else [im["id"] for im in gt["images"]]))
    p.catIds = list(np.unique([c["id"] for c in gt["categories"]]))
    ign = "ignore2D" if mode == "2D" else "ignore3D"
    rng_key = "area" if mode == "2D" else "depth"
    gts = _by_group([dict(a) for a in gt["annotations"]], p.imgIds, p.catIds)
    dtg = _by_group(dts, p.imgIds, p.catIds)
    maxDet = p.maxDets[-1]
    T = len(p.iouThrs)
    ious = {}
    for img in p.imgIds:
        for cat in p.catIds:
            g, d = gts.get((img, cat), []), dtg.get((img, cat), [])
            if not g and not d:
                continue
            d = [d[i] for i in np.argsort([-x["score"] for x in d], kind="mergesort")][:maxDet]
            if mode == "2D":
                iou = bb_iou([x["bbox"] for x in d], [x["bbox"] for x in g])
            elif d and g:
                iou = iou3d.box3d_overlap([x["bbox3D"] for x in d], [x["bbox3D"] for x in g])[0]
            else:
                iou = []
            prox = None
            if eval_prox:
                i2 = bb_iou([x["bbox"] for x in d], [x["bbox"] for x in g])
                prox = [] if isinstance(i2, list) else i2 > p.proximity_thresh
            ious[img, cat] = (iou, prox)
    evalImgs = []
    for cat in p.catIds:
        for aRng in p.areaRng:
            for img in p.imgIds:
                g, d = gts.get((img, cat), []), dtg.get((img, cat), [])
                if not g and not d:
                    evalImgs.append(None)
                    continue
                gig = [int(bool(x.get(ign, 0)) or x[rng_key] < aRng[0] or x[rng_key] > aRng[1]) for x in g]
                gtind = np.argsort(gig, kind="mergesort")
                g = [g[i] for i in gtind]
                gtIg = np.array([gig[i] for i in gtind])
                d = [d[i] for i in np.argsort([-x["score"] for x in d], kind="mergesort")[:maxDet]]
                iou, prox = ious[img, cat]
                iou = iou[:, gtind] if len(iou) > 0 else iou
                if eval_prox:
                    prox = prox[:, gtind] if len(prox) > 0 else prox
                G, D = len(g), len(d)
                gtm, dtm, dtIg = np.zeros((T, G)), np.zeros((T, D)), np.zeros((T, D))
                if len(iou) != 0:
                    for ti, t in enumerate(p.iouThrs):
                        for di in range(D):
                            cur, m = min([t, 1 - 1e-10]), -1
                            for gi in range(G):
                                if eval_prox and not prox[di, gi]:
                                    continue
                                if gtm[ti, gi] > 0:
                                    continue
                                if m > -1 and gtIg[m] == 0 and gtIg[gi] == 1:
                                    break
                                if iou[di, gi] < cur:
                                    continue
                                cur, m = iou[di, gi], gi
                            if m == -1:
                                continue
                            dtIg[ti, di] = gtIg[m]
                            dtm[ti, di] = g[m]["id"]
                            gtm[ti, m] = d[di]["id"]
                out = np.array([x[rng_key] < aRng[0] or x[rng_key] > aRng[1] for x in d]).reshape((1, D))
                dtIg = np.logical_or(dtIg, np.logical_and(dtm == 0, np.repeat(out, T, 0)))
                if eval_prox and len(prox) > 0:
                    dtIg = np.logical_or(dtIg, np.repeat((prox.any(1) == 0).reshape((1, D)), T, 0))
                evalImgs.append({"image_id": img, "category_id": cat, "aRng": aRng, "maxDet": maxDet,
                                 "dtIds": [x["id"] for x in d], "gtIds": [x["id"] for x in g], "dtMatches": dtm,
                                 "gtMatches": gtm, "dtScores": [x["score"] for x in d], "gtIgnore": gtIg,
                                 "dtIgnore": dtIg})
    return p, evalImgs


def per_cat_area(p, evalImgs):
    """accumulate's evals_per_cat_area: {(catId, a): [non-None evalImgs in image order]}."""
    I = len(p.imgIds)
    return {(c, a): [e for e in evalImgs[(k * len(p.areaRng) + a) * I:(k * len(p.areaRng) + a + 1) * I] if e is not None]
            for k, c in enumerate(p.catIds) for a in range(len(p.areaRng))}


def accumulate(p, evals_per_cat_area, cat_ids=None):
    """Omni3Deval.accumulate over precomputed {(catId, a): E} -> (precision, recall, scores)."""
    cat_ids = p.catIds if cat_ids is None else cat_ids
    T, R, K, A, M = len(p.iouThrs), len(p.recThrs), len(cat_ids), len(p.areaRng), len(p.maxDets)
    precision, recall, scores = -np.ones((T, R, K, A, M)), -np.ones((T, K, A, M)), -np.ones((T, R, K, A, M))
    for k, cat in enumerate(cat_ids):
        for a in range(A):
            E = evals_per_cat_area[(cat, a)]
            if len(E) == 0:
                continue
            for m, maxDet in enumerate(p.maxDets):
                dtScores = np.concatenate([e["dtScores"][0:maxDet] for e in E])
                inds = np.argsort(-dtScores, kind="mergesort")
                dtScoresSorted = dtScores[inds]
                dtm = np.concatenate([e["dtMatches"][:, 0:maxDet] for e in E], axis=1)[:, inds]
                dtIg = np.concatenate([e["dtIgnore"][:, 0:maxDet] for e in E], axis=1)[:, inds]
                gtIg = np.concatenate([e["gtIgnore"] for e in E])
                npig = np.count_nonzero(gtIg == 0)
                if npig == 0:
                    continue
                tp_sum = np.cumsum(np.logical_and(dtm, np.logical_not(dtIg)), axis=1).astype(float)
                fp_sum = np.cumsum(np.logical_and(np.logical_not(dtm), np.logical_not(dtIg)), axis=1).astype(float)
                for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
                    nd = len(tp)
                    rc = tp / npig
                    pr = tp / (fp + tp + np.spacing(1))
                    recall[t, k, a, m] = rc[-1] if nd else 0
                    env = np.maximum.accumulate(pr[::-1])[::-1]          # the reference's backward "if pr[i] > pr[i-1]" pass
                    q, ss = np.zeros(R), np.zeros(R)
                    idx = np.searchsorted(rc, p.recThrs, side="left")
                    ok = idx < nd                                        # its try/except stops at the first index past the end
                    upto = int(np.argmin(ok)) if not ok.all() else R
                    q[:upto] = env[idx[:upto]]
                    ss[:upto] = dtScoresSorted[idx[:upto]]
                    precision[t, :, k, a, m] = q
                    scores[t, :, k, a, m] = ss
    return precision, recall, scores


def summarize(p, precision, recall):
    """Omni3Deval.summarize -> (stats (13,), log string)."""
    mode = p.mode

    def one(ap=1, iouThr=None, areaRng="all", maxDets=100, log_str=""):
        if mode == "2D":
            iStr = " {:<18} {} @[ IoU={:<9} | area={:>6s} | maxDets={:>3d} ] = {:0.3f}"
        else:
            iStr = " {:<18} {} @[ IoU={:<9} | depth={:>6s} | maxDets={:>3d} ] = {:0.3f}"
        titleStr = "Average Precision" if ap == 1 else "Average Recall"
        typeStr = "(AP)" if ap == 1 else "(AR)"
        iouStr = "{:0.2f}:{:0.2f}".format(p.iouThrs[0], p.iouThrs[-1]) if iouThr is None else "{:0.2f}".format(iouThr)
        aind = [i for i, a in enumerate(p.areaRngLbl) if a == areaRng]
        mind = [i for i, m in enumerate(p.maxDets) if m == maxDets]
        if ap == 1:
            s = precision
            if iouThr is not None:
                s = s[np.where(np.isclose(iouThr, p.iouThrs.astype(float)))[0]]
            s = s[:, :, :, aind, mind]
        else:
            s = recall
            if iouThr is not None:
                s = s[np.where(iouThr == p.iouThrs)[0]]
            s = s[:, :, aind, mind]
        mean_s = -1 if len(s[s > -1]) == 0 else np.mean(s[s > -1])
        if log_str != "":
            log_str += "\n"
        return mean_s, log_str + "mode={} ".format(mode) + iStr.format(titleStr, typeStr, iouStr, areaRng, maxDets, mean_s)

    thres = [0.5, 0.75, 0.95] if mode == "2D" else [0.15, 0.25, 0.50]
    L, md = p.areaRngLbl, p.maxDets
    calls = [dict(ap=1), dict(ap=1, iouThr=thres[0], maxDets=md[2]), dict(ap=1, iouThr=thres[1], maxDets=md[2]),
             dict(ap=1, iouThr=thres[2], maxDets=md[2]), dict(ap=1, areaRng=L[1], maxDets=md[2]),
             dict(ap=1, areaRng=L[2], maxDets=md[2]), dict(ap=1, areaRng=L[3], maxDets=md[2]),
             dict(ap=0, maxDets=md[0]), dict(ap=0, maxDets=md[1]), dict(ap=0, maxDets=md[2]),
             dict(ap=0, areaRng=L[1], maxDets=md[2]), dict(ap=0, areaRng=L[2], maxDets=md[2]),
             dict(ap=0, areaRng=L[3], maxDets=md[2])]
    stats, log_str = np.zeros((13,)), ""
    for i, kw in enumerate(calls):
        stats[i], log_str = one(log_str=log_str, **kw)
    return stats, log_str


def derive_results(stats, precision, mode, class_names=None):
    """_derive_omni_results without the logging: the x100 metrics and per-category AP."""
    metrics = {"2D": ["AP", "AP50", "AP75", "AP95", "APs", "APm", "APl"],
               "3D": ["AP", "AP15", "AP25", "AP50", "APn", "APm", "APf"]}[mode]
    res = {m: float(stats[i] * 100 if stats[i] >= 0 else "nan") for i, m in enumerate(metrics)}
    if class_names is None or len(class_names) <= 1:
        return res
    for idx, name in enumerate(class_names):
        pr = precision[:, :, idx, 0, -1]
        pr = pr[pr > -1]
        res["AP-" + name] = float((np.mean(pr) if pr.size else float("nan")) * 100)
    return res


def flatten_eval_imgs(evalImgs):
    """evalImgs (list of dict | None) -> dict of flat arrays (npz-storable; `present` marks the non-None entries)."""
    present = np.array([e is not None for e in evalImgs], bool)
    E = [e for e in evalImgs if e is not None]
    cat = lambda f, dt, ax=0: (np.concatenate([np.asarray(f(e), dt) for e in E], axis=ax) if E else np.zeros(0, dt))
    return {
        "present": present,
        "nd": np.array([len(e["dtIds"]) for e in E], np.int64), "ng": np.array([len(e["gtIds"]) for e in E], np.int64),
        "image_id": np.array([e["image_id"] for e in E], np.int64),
        "category_id": np.array([e["category_id"] for e in E], np.int64),
        "dtIds": cat(lambda e: e["dtIds"], np.int64), "gtIds": cat(lambda e: e["gtIds"], np.int64),
        "dtScores": cat(lambda e: e["dtScores"], np.float64), "gtIgnore": cat(lambda e: e["gtIgnore"], np.int64),
        "dtMatches": cat(lambda e: e["dtMatches"].T.reshape(-1), np.float64),
        "gtMatches": cat(lambda e: e["gtMatches"].T.reshape(-1), np.float64),
        "dtIgnore": cat(lambda e: e["dtIgnore"].T.reshape(-1), bool),
    }
