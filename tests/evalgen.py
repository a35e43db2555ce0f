"""Seeded synthetic Omni3D-style evaluation sets: a COCO-style GT dict and a results list in the reference's
instances_to_coco_json form (float32 boxes / scores widened exactly, depth = mean of the corner z)."""
import numpy as np

import boxgen


def make_set(n_img, n_cat, seed, gt_per_img=4, fp_per_img=6, quirks=True, img0=1, ann0=1):
    rng = np.random.default_rng(seed)
    images = [{"id": img0 + i} for i in range(n_img)]
    cats = [{"id": 10 + 3 * k} for k in range(n_cat)]
    anns, results = [], []
    aid = ann0
    for im in images:
        ng = int(rng.integers(0, 2 * gt_per_img + 1))
        for _ in range(ng):
            c = cats[int(rng.integers(0, max(n_cat - 1, 1)))]["id"]       # the last category never has GTs
            x, y = rng.uniform(0, 600), rng.uniform(0, 400)
            w, h = rng.choice([rng.uniform(2, 200), 32.0, 96.0, 16.0, 64.0]), rng.choice([rng.uniform(2, 200), 32.0, 96.0, 16.0])
            z = float(rng.choice([rng.uniform(1, 60), 10.0, 35.0, rng.uniform(1, 60)]))
            dims = rng.uniform(0.5, 3, 3)
            b3 = boxgen.corners([[rng.uniform(-5, 5), rng.uniform(-2, 2), z]], [dims], boxgen.random_rotations(1, rng))[0]
            bb = [float(np.float32(x)), float(np.float32(y)), float(np.float32(w)), float(np.float32(h))]
            a = {"id": aid, "image_id": im["id"], "category_id": c, "bbox": bb, "bbox3D": b3.tolist(),
                 "area": bb[2] * bb[3], "depth": z}
            if quirks and rng.random() < 0.08:
                a["ignore2D"] = 1
            if quirks and rng.random() < 0.08:
                a["ignore3D"] = 1
            anns.append(a)
            aid += 1
            # detections of this GT: jittered copies, sometimes several
            for _ in range(int(rng.integers(0, 3))):
                j = rng.normal(0, 0.08, 4) * np.array([w, h, w, h])
                xyxy = np.array([x + j[0], y + j[1], x + w + j[2], y + h + j[3]], np.float32)
                b3d = boxgen.corners([b3.mean(0) + rng.normal(0, 0.2, 3)], [dims * rng.uniform(0.8, 1.2, 3)],
                                     boxgen.random_rotations(1, rng))[0]
                results.append(_result(im["id"], c, xyxy, _score(rng, quirks), b3d))
        for _ in range(int(rng.integers(0, 2 * fp_per_img + 1))):
            c = cats[int(rng.integers(0, n_cat))]["id"]
            x, y = rng.uniform(0, 600), rng.uniform(0, 400)
            xyxy = np.array([x, y, x + rng.uniform(2, 150), y + rng.uniform(2, 150)], np.float32)
            b3d = boxgen.corners([[rng.uniform(-5, 5), rng.uniform(-2, 2), rng.uniform(1, 60)]], [rng.uniform(0.5, 3, 3)],
                                 boxgen.random_rotations(1, rng))[0]
            results.append(_result(im["id"], c, xyxy, _score(rng, quirks), b3d))
    if quirks and anns:
        anns[0]["id"] = 0                                     # dtMatches holds GT ids: a match to id 0 reads as unmatched
        im, c = images[0]["id"], cats[0]["id"]               # > 100 detections in one group, tied scores
        for t in range(130):
            x = float(rng.uniform(0, 500))
            xyxy = np.array([x, 50, x + 40, 90], np.float32)
            b3d = boxgen.corners([[rng.uniform(-5, 5), 0, float(rng.choice([10.0, 35.0, 20.0]))]], [[1, 1, 1]])[0]
            results.append(_result(im, c, xyxy, float(np.float32(rng.choice([0.5, 0.25, 0.75]))), b3d))
    perm = rng.permutation(len(results))
    results = [results[i] for i in perm]
    return {"images": images, "categories": cats, "annotations": anns}, results


def _score(rng, quirks):
    if quirks and rng.random() < 0.3:
        return float(rng.choice([0.0, -0.0, 0.5, 0.125]))
    return float(np.float32(rng.random()))


def _result(img, cat, xyxy, score, b3d):
    b = xyxy.astype(np.float32).copy()
    b[2:] -= b[:2]
    b3 = np.asarray(b3d, np.float32).tolist()
    return {"image_id": img, "category_id": cat, "bbox": b.tolist(), "score": score,
            "depth": np.array(b3)[:, 2].mean(), "bbox3D": b3}
