"""Device-side Omni3D evaluation: the batched 3D-IoU front-end (SURVEY 8f-1) and Omni3DEval (SURVEY 8f-5).

The reference's only caller of box3d_overlap is Omni3Deval.computeIoU
(cubercnn/evaluation/omni3d_evaluation.py:1359-1431), evaluated once per (image, category) from the dict
comprehension at :1339-1343: tens of thousands of calls with N <= maxDets detections x M <= ~30 ground truths,
each doing two host->device copies, one tiny op and one device->host copy (or, with MAX_DTS_CROSS_GTS_FOR_IOU3D = 0
at :62, a serial CPU loop).  Here ALL (image, category) groups go through ONE segmented launch
(c3d_box3d_overlap_segmented: CSR offsets over the groups, one H2D of the boxes, one D2H of the packed IoUs).

    compute_ious_3d(dts, gts, img_ids, cat_ids, max_dets)  ->  {(imgId, catId): ious}   == self.ious of the reference
    box3d_overlap_segmented(dt_groups, gt_groups)          ->  list of (n_i, m_i) IoU matrices

Semantics kept from the reference: detections sorted by -score with a stable (merge) sort, truncated to maxDets[-1];
`[]` when a group has no detections and no ground truths, or when either side is empty (:1414-1415); dt rows that fail the
planarity / non-zero-volume checks are zeroed and counted in the printed warning (:158-164), once for the whole batch.
"""
import ctypes
import datetime

import numpy as np
import torch

from . import _lib
from .box3d import _device_of, _workspace

_bound = False


def _bind():
    global _bound
    L = _lib.lib()
    if not _bound:
        vp, i32, i64, f32, sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_size_t
        L.c3d_box3d_overlap_segmented_workspace_bytes.restype = sz
        L.c3d_box3d_overlap_segmented_workspace_bytes.argtypes = [i64, i64, i64]
        L.c3d_box3d_overlap_segmented.restype = i32
        L.c3d_box3d_overlap_segmented.argtypes = [vp, i64, vp, i64, vp, vp, vp, i32, i64, f32, f32, vp, vp, vp, sz, vp]
        _bound = True
    return L


def _as_boxes(x):
    a = np.asarray(x, dtype=np.float32)
    if a.size == 0:
        return np.zeros((0, 8, 3), np.float32)
    if a.ndim != 3 or a.shape[1:] != (8, 3):
        raise ValueError(f"boxes must be (n, 8, 3), got {a.shape}")
    return a


def box3d_overlap_segmented(dt_groups, gt_groups, eps_coplanar=1e-4, eps_nonzero=1e-8, device=None, return_bad_counts=False):
    """dt_groups[i] (n_i,8,3), gt_groups[i] (m_i,8,3) (arrays / tensors / nested lists) -> [iou_i (n_i, m_i) float32 numpy].
    One launch for all groups; equals box3d_overlap(dt_i, gt_i) of every group bit for bit."""
    if len(dt_groups) != len(gt_groups):
        raise ValueError("dt_groups and gt_groups must have the same length")
    L = _bind()
    G = len(dt_groups)
    dts = [_as_boxes(d.cpu() if isinstance(d, torch.Tensor) else d) for d in dt_groups]
    gts = [_as_boxes(g.cpu() if isinstance(g, torch.Tensor) else g) for g in gt_groups]
    nd = np.array([len(d) for d in dts], np.int64)
    ng = np.array([len(g) for g in gts], np.int64)
    dt_off = np.zeros(G + 1, np.int32); dt_off[1:] = np.cumsum(nd)
    gt_off = np.zeros(G + 1, np.int32); gt_off[1:] = np.cumsum(ng)
    pair_off = np.zeros(G + 1, np.int64); pair_off[1:] = np.cumsum(nd * ng)
    n_dt, n_gt, total = int(dt_off[-1]), int(gt_off[-1]), int(pair_off[-1])
    bad = [0, 0]
    out = np.zeros(total, np.float32)
    if n_dt > 0:
        dev = device if device is not None else _device_of()
        with torch.cuda.device(dev):
            up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev, non_blocking=False)
            b1 = up(np.concatenate(dts) if n_dt else np.zeros((0, 8, 3), np.float32))
            b2 = up(np.concatenate(gts) if n_gt else np.zeros((1, 8, 3), np.float32))
            d_off, g_off, p_off = up(dt_off), up(gt_off), up(pair_off)
            iou = torch.empty(max(total, 1), dtype=torch.float32, device=dev)
            nbad = torch.zeros(2, dtype=torch.int32, device=dev)
            ws = _workspace(L.c3d_box3d_overlap_segmented_workspace_bytes(n_dt, max(n_gt, 1), total), dev)
            st = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(L.c3d_box3d_overlap_segmented(b1.data_ptr(), n_dt, b2.data_ptr(), n_gt, d_off.data_ptr(), g_off.data_ptr(),
                                                     p_off.data_ptr(), G, total, eps_coplanar, eps_nonzero, iou.data_ptr(),
                                                     nbad.data_ptr(), ws.data_ptr(), ws.numel(), ctypes.c_void_p(st)), launches=5)
            out = iou[:total].cpu().numpy()
            bad = nbad.tolist()
    if bad[0]:
        print('Warning: skipping {:d} non-coplanar boxes at eval.'.format(int(bad[0])))
    if bad[1]:
        print('Warning: skipping {:d} zero volume boxes at eval.'.format(int(bad[1])))
    res = [out[pair_off[i]:pair_off[i + 1]].reshape(int(nd[i]), int(ng[i])) for i in range(G)]
    return (res, bad) if return_bad_counts else res


def iou2d_xywh(d, g):
    """pycocotools maskUtils.iou(d, g, iscrowd=0) for [x, y, w, h] boxes (omni3d_evaluation.py:1399,1423)."""
    d, g = np.asarray(d, np.float64).reshape(-1, 4), np.asarray(g, np.float64).reshape(-1, 4)
    if len(d) == 0 or len(g) == 0:
        return []
    iw = np.minimum(d[:, None, 0] + d[:, None, 2], g[None, :, 0] + g[None, :, 2]) - np.maximum(d[:, None, 0], g[None, :, 0])
    ih = np.minimum(d[:, None, 1] + d[:, None, 3], g[None, :, 1] + g[None, :, 3]) - np.maximum(d[:, None, 1], g[None, :, 1])
    inter = np.clip(iw, 0, None) * np.clip(ih, 0, None)
    union = (d[:, 2] * d[:, 3])[:, None] + (g[:, 2] * g[:, 3])[None, :] - inter
    return inter / union


def compute_ious_3d(dts, gts, img_ids, cat_ids, max_dets, use_cats=True, eval_prox=False, proximity_thresh=0.3):
    """The reference's `self.ious = {(imgId, catId): self.computeIoU(imgId, catId) ...}` (omni3d_evaluation.py:1339-1343) in
    3D mode.  dts / gts: {(imgId, catId): [ {"score", "bbox3D" (8x3), "bbox" [x,y,w,h], ...}, ... ]} like self._dts / self._gts.
    -> {(imgId, catId): [] | (ious (n,m) ndarray | [], in_prox)}, every 3D IoU coming from ONE segmented launch."""
    cats = list(cat_ids) if use_cats else [-1]
    keys, D, Gs = [], [], []
    for img in img_ids:
        for cat in cats:
            if use_cats:
                gt, dt = gts.get((img, cat), []), dts.get((img, cat), [])
            else:
                gt = [x for c in cat_ids for x in gts.get((img, c), [])]
                dt = [x for c in cat_ids for x in dts.get((img, c), [])]
            inds = np.argsort([-d["score"] for d in dt], kind="mergesort")
            dt = [dt[i] for i in inds][: max_dets]
            keys.append((img, cat)); D.append(dt); Gs.append(gt)
    run = [i for i in range(len(keys)) if len(D[i]) > 0 and len(Gs[i]) > 0]
    mats = box3d_overlap_segmented([[d["bbox3D"] for d in D[i]] for i in run], [[g["bbox3D"] for g in Gs[i]] for i in run]) \
        if run else []
    by = dict(zip(run, mats))
    out = {}
    for i, k in enumerate(keys):
        if len(D[i]) == 0 and len(Gs[i]) == 0:
            out[k] = []
            continue
        ious = by.get(i, [])
        in_prox = None
        if eval_prox:
            i2 = iou2d_xywh([d["bbox"] for d in D[i]], [g["bbox"] for g in Gs[i]])
            in_prox = [] if isinstance(i2, list) else i2 > proximity_thresh
        out[k] = (ious, in_prox)
    return out


# ----------------------------------------------------------------------------------------------------------------------
# Omni3DEval: Omni3Deval (cubercnn/evaluation/omni3d_evaluation.py:1019-1705) with its work on the device.  Matching runs
# in c3d_eval_match, the precision / recall / score tables in c3d_eval_accumulate; detections stay device-resident from
# add_instances through accumulate, and the tables come back in one device-to-host copy.
# ----------------------------------------------------------------------------------------------------------------------
_eval_bound = False


def _bind_eval():
    global _eval_bound
    L = _bind()
    if not _eval_bound:
        vp, i32, i64, f64, sz = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_double, ctypes.c_size_t
        L.c3d_eval_match_workspace_bytes.restype = sz
        L.c3d_eval_match_workspace_bytes.argtypes = [i64, i32, i32]
        L.c3d_eval_match.restype = i32
        L.c3d_eval_match.argtypes = [i32, i32, i32, i32, i32] + [vp] * 10 + [i64, i64, vp, vp, f64, vp, vp, vp, vp, sz, vp]
        L.c3d_eval_accumulate.restype = i32
        L.c3d_eval_accumulate.argtypes = [i32] * 5 + [vp] * 7 + [i64] + [vp] * 6
        _eval_bound = True
    return L


class Omni3DParams:
    """Omni3DParams (omni3d_evaluation.py:1019-1087); thresholds are numpy fp64, passed to the device as computed here."""

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
        self.useCats = 1
        self.iouType = "bbox"
        self.mode = mode
        self.proximity_thresh = 0.3


def _score_key(score):
    """fp64 scores -> int64 keys whose ascending order is numpy's argsort(-score): -0.0 ties +0.0, NaN sorts last."""
    s = -score + 0.0
    b = s.view(torch.int64)
    k = b ^ ((b >> 63) & 0x7FFFFFFFFFFFFFFF)
    return torch.where(torch.isnan(s), torch.full_like(k, torch.iinfo(torch.int64).max), k)


def _dense_rank(key):
    """position of every key among the distinct keys (equal keys share a rank)."""
    sk, perm = torch.sort(key, stable=True)
    r = torch.zeros_like(sk)
    r[1:] = torch.cumsum(sk[1:] != sk[:-1], 0)
    out = torch.empty_like(r)
    out[perm] = r
    return out


def _pairwise_mean8(z):
    """numpy's mean of 8 fp64 values: pairwise_sum's eight-accumulator tree, then / 8."""
    return (((z[:, 0] + z[:, 1]) + (z[:, 2] + z[:, 3])) + ((z[:, 4] + z[:, 5]) + (z[:, 6] + z[:, 7]))) / 8


class _Shared:
    """Ground truths, detections and the (category, image) groups, shared by the 2D and 3D evaluators of one set of
    predictions.  Group g = k * I + i for category index k and image index i."""

    FIELDS = ("score", "img", "cat", "box", "area", "depth", "box3d", "id")

    def __init__(self, gt, img_ids, device):
        self.device = device
        self.all_img = set(int(im["id"]) for im in gt["images"])
        self.img_ids = np.unique(np.asarray(img_ids if img_ids is not None else sorted(self.all_img), np.int64))
        self.cat_ids = np.unique(np.asarray([c["id"] for c in gt["categories"]], np.int64))
        I, K = len(self.img_ids), len(self.cat_ids)
        anns = [a for a in gt["annotations"] if self._index(self.img_ids, a["image_id"]) >= 0
                and self._index(self.cat_ids, a["category_id"]) >= 0]
        grp = np.array([self._index(self.cat_ids, a["category_id"]) * I + self._index(self.img_ids, a["image_id"])
                        for a in anns], np.int64)
        # getAnnIds order: images in imgIds order, annotation order within an image -> stable by group
        o = np.argsort(grp, kind="stable")
        anns = [anns[i] for i in o]
        self.gt_host = {
            "grp": grp[o], "id": np.array([a["id"] for a in anns], np.int64).reshape(-1),
            "box": np.array([a["bbox"] for a in anns], np.float64).reshape(-1, 4),
            "area": np.array([a["area"] for a in anns], np.float64).reshape(-1),
            "depth": np.array([a["depth"] for a in anns], np.float64).reshape(-1),
            "ignore2D": np.array([bool(a.get("ignore2D", 0)) for a in anns], np.uint8).reshape(-1),
            "ignore3D": np.array([bool(a.get("ignore3D", 0)) for a in anns], np.uint8).reshape(-1),
            "box3d": np.array([a["bbox3D"] for a in anns], np.float32).reshape(-1, 8, 3),
        }
        cnt = np.bincount(grp, minlength=K * I)
        self.gt_cnt = cnt
        gt_off = np.zeros(K * I + 1, np.int64)
        gt_off[1:] = np.cumsum(cnt)
        self.gt_host["off"] = gt_off
        self.gt = {k: torch.from_numpy(np.ascontiguousarray(v)).to(device) for k, v in self.gt_host.items()}
        self.gt["off"] = self.gt["off"].int()
        self.chunks = []
        self.n_results = 0
        self._groups = None

    @staticmethod
    def _index(ids, v):
        i = int(np.searchsorted(ids, v))
        return i if i < len(ids) and ids[i] == v else -1

    def add(self, fields):
        self.chunks.append(fields)
        self._groups = None

    def groups(self, max_det):
        """sort detections by (category, image, -score, results order), truncate every group to max_det -> the L list."""
        if self._groups is not None:
            return self._groups
        dev, I, K = self.device, len(self.img_ids), len(self.cat_ids)
        G = K * I
        if self.chunks:
            d = {k: torch.cat([c[k] for c in self.chunks]) for k in self.FIELDS}
        else:
            d = {"score": torch.zeros(0, dtype=torch.float64, device=dev), "img": torch.zeros(0, dtype=torch.int64, device=dev),
                 "cat": torch.zeros(0, dtype=torch.int64, device=dev), "box": torch.zeros(0, 4, dtype=torch.float64, device=dev),
                 "area": torch.zeros(0, dtype=torch.float64, device=dev), "depth": torch.zeros(0, dtype=torch.float64, device=dev),
                 "box3d": torch.zeros(0, 8, 3, dtype=torch.float32, device=dev), "id": torch.zeros(0, dtype=torch.int64, device=dev)}
        N = d["score"].numel()
        srank = _dense_rank(_score_key(d["score"]))
        grp = d["cat"] * I + d["img"]
        gk, order = torch.sort(grp * max(N, 1) + srank, stable=True)
        gs = grp[order]
        cnt = torch.bincount(gs, minlength=G)
        start = torch.cumsum(cnt, 0) - cnt
        rank = torch.arange(N, device=dev) - start[gs]
        keep = rank < max_det
        L = order[keep]
        dt_cnt = cnt.clamp(max=max_det)
        dt_off = torch.zeros(G + 1, dtype=torch.int32, device=dev)
        dt_off[1:] = torch.cumsum(dt_cnt, 0).int()
        g = {k: v[L].contiguous() for k, v in d.items()}
        g["rank"] = rank[keep].int()
        g["grp"] = gs[keep]
        g["dt_cnt"], g["dt_off"] = dt_cnt, dt_off
        # accumulation order: category, then -score, ties in (image, rank) order
        NL = L.numel()
        cat_l = g["cat"]
        _, ent = torch.sort(cat_l * max(NL, 1) + _dense_rank(_score_key(g["score"])), stable=True)
        g["ent_idx"] = ent.int()
        g["ent_rank"] = g["rank"][ent].contiguous()
        g["ent_score"] = g["score"][ent].contiguous()
        ent_off = torch.zeros(K + 1, dtype=torch.int32, device=dev)
        ent_off[1:] = torch.cumsum(torch.bincount(cat_l, minlength=K), 0).int()
        g["ent_off"] = ent_off
        self._groups = g
        return g


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class Omni3DEval:
    """Omni3Deval(cocoGt, cocoDt, mode, eval_prox) on the device, useCats = 1.

    gt: COCO-style dict {"images": [{"id"}], "categories": [{"id"}], "annotations": [...]}, annotations carrying id,
    image_id, category_id, bbox (XYWH), bbox3D (8 x 3), area, depth and optionally ignore2D / ignore3D (as the Omni3D
    dataset API prepares them, cubercnn/data/datasets.py:253-269).  img_ids restricts the evaluated images like
    _evaluate_predictions_on_omni's img_ids.

        e2d = Omni3DEval(gt, "2D"); e2d.add_instances(image_ids, instances, category_map)
        e3d = e2d.for_mode("3D")            # same detections and groups
        for e in (e2d, e3d): e.evaluate(); e.accumulate(); log = e.summarize()
    """

    def __init__(self, gt, mode="2D", eval_prox=False, img_ids=None, device=None, _shared=None):
        if mode not in ("2D", "3D"):
            raise ValueError("mode %s not supported" % mode)
        self.mode, self.eval_prox = mode, bool(eval_prox)
        dev = torch.device(device) if device is not None else _device_of()
        self._s = _shared if _shared is not None else _Shared(gt, img_ids, dev)
        self.params = Omni3DParams(mode)
        self.params.imgIds = [int(i) for i in self._s.img_ids]
        self.params.catIds = [int(c) for c in self._s.cat_ids]
        self.eval, self.stats = {}, []
        self._m = None

    def for_mode(self, mode, eval_prox=None):
        """an evaluator of the same ground truths and detections in another mode (the groups are built once)."""
        return Omni3DEval(None, mode, self.eval_prox if eval_prox is None else eval_prox, _shared=self._s)

    # ------------------------------------------------------------------------------------------------ detections
    def _append(self, img_id, cat_id, score, box, area, depth, box3d, keep_np=None):
        """register results (host or device arrays) with ids continuing the results list, dropping those outside
        imgIds / catIds as getAnnIds does."""
        s = self._s
        dev = s.device
        n = int(score.shape[0])
        ids = torch.arange(s.n_results + 1, s.n_results + n + 1, dtype=torch.int64, device=dev)
        s.n_results += n
        keep = (img_id >= 0) & (cat_id >= 0)
        f = dict(score=score, img=img_id, cat=cat_id, box=box, area=area, depth=depth, box3d=box3d, id=ids)
        s.add({k: v[keep] for k, v in f.items()})

    def add_results(self, results):
        """the reference's COCO-result dicts (image_id, category_id, bbox XYWH, score, depth, bbox3D) -> device arrays,
        ids = position in the results list + 1 and area = w * h as COCO.loadRes assigns them."""
        s = self._s
        if not results:
            return
        bad = {int(r["image_id"]) for r in results} - s.all_img
        if bad:
            raise ValueError(f"Results do not correspond to current coco set: image ids {sorted(bad)[:5]}")
        img = np.array([s._index(s.img_ids, r["image_id"]) for r in results], np.int64)
        cat = np.array([s._index(s.cat_ids, r["category_id"]) for r in results], np.int64)
        box = np.array([r["bbox"] for r in results], np.float64).reshape(-1, 4)
        area = np.array([r["bbox"][2] * r["bbox"][3] for r in results], np.float64)
        b3 = np.array([r["bbox3D"] for r in results], np.float32).reshape(-1, 8, 3)
        depth = np.array([r["depth"] if "depth" in r else np.array(r["bbox3D"])[:, 2].mean() for r in results], np.float64)
        score = np.array([r["score"] for r in results], np.float64)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(s.device)
        self._append(up(img), up(cat), up(score), up(box), up(area), up(depth), up(b3))

    def add_instances(self, image_ids, instances, category_map):
        """RCNN3D inference outputs, kept on the device: instances[j] (pred_boxes XYXY, scores, pred_classes, pred_bbox3D)
        belongs to image image_ids[j]; category_map[c] = dataset category id of contiguous class c, or -1 to drop the
        prediction before ids are assigned (_eval_predictions, omni3d_evaluation.py:856-885).  The result fields are
        computed as instances_to_coco_json + COCO.loadRes compute them: XYWH in float32, area and depth in fp64."""
        s = self._s
        dev = s.device
        counts = [len(x) for x in instances]
        if len(image_ids) != len(instances):
            raise ValueError("image_ids and instances must have the same length")
        bad = {int(i) for i, c in zip(image_ids, counts) if c > 0} - s.all_img
        if bad:
            raise ValueError(f"Results do not correspond to current coco set: image ids {sorted(bad)[:5]}")
        if sum(counts) == 0:
            return
        cmap = np.asarray(category_map, np.int64)
        table = np.array([-1 if c < 0 else (s._index(s.cat_ids, c) if s._index(s.cat_ids, c) >= 0 else -2) for c in cmap],
                         np.int64)
        img_idx = np.repeat(np.array([s._index(s.img_ids, i) for i in image_ids], np.int64), counts)
        cls = torch.cat([x.pred_classes for x in instances]).to(dev).long()
        cat = torch.from_numpy(table).to(dev)[cls]
        present = cat != -1
        xyxy = torch.cat([x.pred_boxes.tensor for x in instances]).to(dev).float()[present]
        box = torch.stack([xyxy[:, 0], xyxy[:, 1], xyxy[:, 2] - xyxy[:, 0], xyxy[:, 3] - xyxy[:, 1]], 1).double()
        b3 = torch.cat([x.pred_bbox3D for x in instances]).to(dev).float()[present].contiguous()
        score = torch.cat([x.scores for x in instances]).to(dev).float()[present].double()
        img = torch.from_numpy(img_idx).to(dev)[present]
        cat = cat[present]
        self._append(img, cat.clamp(min=-1), score, box, box[:, 2] * box[:, 3], _pairwise_mean8(b3[:, :, 2].double()), b3)

    # ------------------------------------------------------------------------------------------------ evaluate
    def evaluate(self):
        """Omni3Deval.evaluate: one c3d_eval_match launch (plus the segmented 3D IoU in 3D mode) over every group."""
        p = self.params
        if p.useCats != 1:
            raise NotImplementedError("Omni3DEval supports useCats = 1 only")
        L = _bind_eval()
        s, dev = self._s, self._s.device
        g = s.groups(p.maxDets[-1])
        A, T = len(p.areaRng), len(p.iouThrs)
        G, NL, NG = len(s.cat_ids) * len(s.img_ids), g["score"].numel(), s.gt["id"].numel()
        is3d = self.mode == "3D"
        st = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            iou3d = pair_off = None
            if is3d:
                pair_off = torch.zeros(G + 1, dtype=torch.int64, device=dev)
                pair_off[1:] = torch.cumsum(g["dt_cnt"] * torch.from_numpy(s.gt_cnt).to(dev), 0)
                total = int(pair_off[-1])
                iou3d = torch.empty(max(total, 1), dtype=torch.float32, device=dev)
                if total > 0:
                    nbad = torch.zeros(2, dtype=torch.int32, device=dev)
                    ws = _workspace(L.c3d_box3d_overlap_segmented_workspace_bytes(NL, max(NG, 1), total), dev)
                    _lib.check(L.c3d_box3d_overlap_segmented(
                        g["box3d"].data_ptr(), NL, s.gt["box3d"].data_ptr(), NG, g["dt_off"].data_ptr(),
                        s.gt["off"].data_ptr(), pair_off.data_ptr(), G, total, 1e-4, 1e-8, iou3d.data_ptr(),
                        nbad.data_ptr(), ws.data_ptr(), ws.numel(), ctypes.c_void_p(st)), launches=5)
            rng = "depth" if is3d else "area"
            match = torch.empty(A * T, max(NL, 1), dtype=torch.int32, device=dev)
            flags = torch.empty(A * T, max(NL, 1), dtype=torch.uint8, device=dev)
            npig = torch.empty(max(G, 1), A, dtype=torch.int32, device=dev)
            ws = torch.empty(max(L.c3d_eval_match_workspace_bytes(NG, A, T), 1), dtype=torch.uint8, device=dev)
            start = np.array([min([t, 1 - 1e-10]) for t in p.iouThrs], np.float64)
            ranges = np.ascontiguousarray(np.asarray(p.areaRng, np.float64))
            empty_b = torch.zeros(1, 4, dtype=torch.float64, device=dev)
            gtf = lambda k: s.gt[k] if NG > 0 else torch.zeros(1, 4, dtype=torch.float64, device=dev)
            _lib.check(L.c3d_eval_match(
                int(is3d), int(self.eval_prox), G, A, T, _ptr(g["dt_off"]), _ptr(s.gt["off"]),
                _ptr(g["box"] if NL else empty_b), _ptr(g[rng] if NL else empty_b), _ptr(gtf("box")), _ptr(gtf(rng)),
                _ptr(gtf("ignore3D" if is3d else "ignore2D")), _ptr(gtf("id")), _ptr(iou3d), _ptr(pair_off), NL, NG,
                start.ctypes.data_as(ctypes.c_void_p), ranges.ctypes.data_as(ctypes.c_void_p), float(p.proximity_thresh),
                _ptr(match), _ptr(flags), _ptr(npig), _ptr(ws), ws.numel(), ctypes.c_void_p(st)))
        self._m = {"match": match, "flags": flags, "npig": npig, "NL": NL, "g": g}
        self._paramsEval = p

    # ------------------------------------------------------------------------------------------------ accumulate
    def accumulate(self):
        """Omni3Deval.accumulate: one c3d_eval_accumulate launch, one device-to-host copy of the three tables."""
        if self._m is None:
            raise RuntimeError("Please run evaluate() first")
        g, I = self._m["g"], len(self._s.img_ids)
        K = len(self._s.cat_ids)
        grp_off = torch.arange(0, K * I + 1, I, dtype=torch.int32, device=self._s.device)
        self.eval = _run_accumulate(self.params, self._s.device, K, grp_off, self._m["npig"], g["ent_off"], g["ent_idx"],
                                    g["ent_rank"], g["ent_score"], self._m["flags"], self._m["NL"])

    def summarize(self):
        """Omni3Deval.summarize: sets .stats (13,) and returns the log string, character for character."""
        if not self.eval:
            raise RuntimeError("Please run accumulate() first")
        self.stats, log = _summarize(self.params, self.mode, self.eval["precision"], self.eval["recall"])
        return log

    def results(self, class_names=None):
        """_derive_omni_results (omni3d_evaluation.py:764-840) without the logging: x100 metrics and AP-<class>."""
        metrics = {"2D": ["AP", "AP50", "AP75", "AP95", "APs", "APm", "APl"],
                   "3D": ["AP", "AP15", "AP25", "AP50", "APn", "APm", "APf"]}[self.mode]
        res = {m: float(self.stats[i] * 100 if self.stats[i] >= 0 else "nan") for i, m in enumerate(metrics)}
        if class_names is None or len(class_names) <= 1:
            return res
        precisions = self.eval["precision"]
        assert len(class_names) == precisions.shape[2]
        for idx, name in enumerate(class_names):
            pr = precisions[:, :, idx, 0, -1]
            pr = pr[pr > -1]
            res["AP-" + "{}".format(name)] = float((np.mean(pr) if pr.size else float("nan")) * 100)
        return res

    def eval_imgs(self):
        """the reference's evalImgs list (category, range, image order; None for empty groups), rebuilt on the host."""
        if self._m is None:
            raise RuntimeError("Please run evaluate() first")
        p, s, g = self.params, self._s, self._m["g"]
        A, T, I, NL = len(p.areaRng), len(p.iouThrs), len(s.img_ids), self._m["NL"]
        match = self._m["match"][:, :NL].cpu().numpy().reshape(A, T, NL)
        flags = self._m["flags"][:, :NL].cpu().numpy().reshape(A, T, NL)
        dt_off = g["dt_off"].cpu().numpy()
        dt_id, dt_score = g["id"].cpu().numpy(), g["score"].cpu().numpy()
        gh = s.gt_host
        ign = gh["ignore3D" if self.mode == "3D" else "ignore2D"]
        rng = gh["depth" if self.mode == "3D" else "area"]
        out = []
        for k, cat in enumerate(s.cat_ids):
            for a, (lo, hi) in enumerate(p.areaRng):
                for i, img in enumerate(s.img_ids):
                    gi = k * I + i
                    d0, d1, g0, g1 = dt_off[gi], dt_off[gi + 1], gh["off"][gi], gh["off"][gi + 1]
                    if d0 == d1 and g0 == g1:
                        out.append(None)
                        continue
                    gig = np.array([int(bool(ign[j]) or rng[j] < lo or rng[j] > hi) for j in range(g0, g1)], np.int64)
                    gtind = np.argsort(gig, kind="mergesort")
                    pos = np.empty(len(gtind), np.int64)
                    pos[gtind] = np.arange(len(gtind))
                    mt = match[a, :, d0:d1]
                    dtm = np.where(mt >= 0, gh["id"][np.maximum(mt, 0)], 0).astype(np.float64)
                    gtm = np.zeros((T, g1 - g0))
                    for t, d in zip(*np.nonzero(mt >= 0)):
                        gtm[t, pos[mt[t, d] - g0]] = dt_id[d0 + d]
                    out.append({"image_id": int(img), "category_id": int(cat), "aRng": p.areaRng[a], "maxDet": p.maxDets[-1],
                                "dtIds": dt_id[d0:d1].tolist(), "gtIds": gh["id"][g0:g1][gtind].tolist(),
                                "dtMatches": dtm, "gtMatches": gtm, "dtScores": dt_score[d0:d1].tolist(),
                                "gtIgnore": gig[gtind], "dtIgnore": (flags[a, :, d0:d1] & 1).astype(bool)})
        return out

    @classmethod
    def concat(cls, evals, cat_ids):
        """summarize_all's re-accumulation (omni3d_evaluation.py:378-447): the evaluated per-dataset evaluators' groups
        concatenated in list order, accumulated over cat_ids.  Returns an evaluator with .eval / .summarize() / .results()."""
        if not evals:
            raise ValueError("concat needs at least one evaluator")
        e0 = evals[0]
        for e in evals:
            if e._m is None:
                raise RuntimeError("Please run evaluate() on every evaluator first")
            if e.mode != e0.mode:
                raise ValueError("cannot concatenate 2D and 3D evaluations")
        dev = e0._s.device
        cat_ids = [int(c) for c in cat_ids]
        K, A = len(cat_ids), len(e0.params.areaRng)
        pos = {c: k for k, c in enumerate(cat_ids)}
        known = set().union(*[set(int(c) for c in e._s.cat_ids) for e in evals])
        missing = [c for c in cat_ids if c not in known]
        if missing:
            raise KeyError(f"categories {missing} are in no evaluation")
        npig = torch.zeros(K, A, dtype=torch.int32, device=dev)
        flags, cats, scores, ranks, cols, off = [], [], [], [], [], 0
        for e in evals:
            s, g = e._s, e._m["g"]
            Ke, Ie = len(s.cat_ids), len(s.img_ids)
            to_out = torch.tensor([pos.get(int(c), -1) for c in s.cat_ids], dtype=torch.int64, device=dev)
            per_cat = e._m["npig"][:Ke * Ie].view(Ke, Ie, A).sum(1, dtype=torch.int32)
            sel = to_out >= 0
            npig.index_add_(0, to_out[sel], per_cat[sel])
            NL = e._m["NL"]
            flags.append(e._m["flags"][:, :NL])
            co = to_out[g["cat"]] if NL else g["cat"]
            keep = co >= 0
            cats.append(co[keep]); scores.append(g["score"][keep]); ranks.append(g["rank"][keep])
            cols.append(torch.nonzero(keep).view(-1) + off)
            off += NL
        flags = torch.cat(flags, 1).contiguous()
        cat_c, score_c, rank_c, col_c = torch.cat(cats), torch.cat(scores), torch.cat(ranks), torch.cat(cols)
        n = cat_c.numel()
        _, ent = torch.sort(cat_c * max(n, 1) + _dense_rank(_score_key(score_c)), stable=True)
        ent_off = torch.zeros(K + 1, dtype=torch.int32, device=dev)
        ent_off[1:] = torch.cumsum(torch.bincount(cat_c, minlength=K), 0).int()
        out = cls.__new__(cls)
        out.mode, out.eval_prox, out._s, out._m, out.stats = e0.mode, e0.eval_prox, None, None, []
        out.params = Omni3DParams(e0.mode)
        out.params.catIds = cat_ids
        out.params.imgIds = sorted(set().union(*[set(e.params.imgIds) for e in evals]))
        out.eval = _run_accumulate(out.params, dev, K, torch.arange(K + 1, dtype=torch.int32, device=dev), npig, ent_off,
                                   col_c[ent].int(), rank_c[ent].contiguous(), score_c[ent].contiguous(), flags, off)
        return out


def _run_accumulate(p, dev, K, grp_off, npig, ent_off, ent_idx, ent_rank, ent_score, flags, n_dt):
    L = _bind_eval()
    T, R, A, M = len(p.iouThrs), len(p.recThrs), len(p.areaRng), len(p.maxDets)
    n_tab = T * R * K * A * M
    with torch.cuda.device(dev):
        buf = torch.empty(2 * n_tab + T * K * A * M, dtype=torch.float64, device=dev)
        rec_thrs = torch.from_numpy(np.ascontiguousarray(p.recThrs, np.float64)).to(dev)
        max_dets = torch.tensor(p.maxDets, dtype=torch.int32, device=dev)
        st = torch.cuda.current_stream(dev).cuda_stream
        if K > 0:
            _lib.check(L.c3d_eval_accumulate(
                K, A, T, M, R, _ptr(grp_off), _ptr(npig), _ptr(ent_off), _ptr(ent_idx), _ptr(ent_rank), _ptr(ent_score),
                _ptr(flags), int(n_dt), _ptr(rec_thrs), _ptr(max_dets), _ptr(buf), _ptr(buf[2 * n_tab:]),
                _ptr(buf[n_tab:]), ctypes.c_void_p(st)))
        host = buf.cpu().numpy()
    return {"params": p, "counts": [T, R, K, A, M], "date": datetime.datetime.now().strftime("%Y-%m-%d %H:%M:%S"),
            "precision": host[:n_tab].reshape(T, R, K, A, M), "recall": host[2 * n_tab:].reshape(T, K, A, M),
            "scores": host[n_tab:2 * n_tab].reshape(T, R, K, A, M)}


def _summarize(p, mode, precision, recall):
    """Omni3Deval.summarize / _summarizeDets (omni3d_evaluation.py:1553-1705) on the host tables."""
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
    lbl, md = p.areaRngLbl, p.maxDets
    calls = [dict(ap=1), dict(ap=1, iouThr=thres[0], maxDets=md[2]), dict(ap=1, iouThr=thres[1], maxDets=md[2]),
             dict(ap=1, iouThr=thres[2], maxDets=md[2])] + \
        [dict(ap=1, areaRng=lbl[i], maxDets=md[2]) for i in (1, 2, 3)] + [dict(ap=0, maxDets=m) for m in md] + \
        [dict(ap=0, areaRng=lbl[i], maxDets=md[2]) for i in (1, 2, 3)]
    stats, log_str = np.zeros((13,)), ""
    for i, kw in enumerate(calls):
        stats[i], log_str = one(log_str=log_str, **kw)
    return stats, log_str
