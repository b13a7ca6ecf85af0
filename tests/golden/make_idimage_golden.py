"""Generates tests/golden/idimage_golden.npz by IMPORTING THE REFERENCE's own Python post-processing
(/root/reference/Core/Segmentation/MaskRCNN/helpers.py: generate_id_image, save_id_image) on seeded detections: the id images / class
lists / boxes it returns, and the mask description file it writes.  The reference tree is not available on the GPU box, so the
vectors are committed.  Run:  python tests/golden/make_idimage_golden.py"""
import os, sys, tempfile
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, "/root/reference/Core/Segmentation/MaskRCNN")
import helpers


def detections(seed, H=48, W=64, N=6):
    rng = np.random.default_rng(seed)
    masks = np.zeros((H, W, N), bool); rois = np.zeros((N, 4), np.int32)
    for m in range(N):
        y1, x1 = rng.integers(0, H - 12), rng.integers(0, W - 12); hh, ww = rng.integers(6, 24), rng.integers(6, 24)
        y2, x2 = min(H, y1 + hh), min(W, x1 + ww)
        masks[y1:y2, x1:x2, m] = rng.random((y2 - y1, x2 - x1)) < 0.8
        rois[m] = (y1, x1, y2, x2)
    scores = rng.uniform(0.3, 1.0, N).astype(np.float32)      # (no score exactly at a threshold: float32-vs-Python-float comparison differs between NumPy 1.x and 2.x)
    class_ids = rng.integers(1, 6, N).astype(np.int32)
    return {"masks": masks, "scores": scores, "class_ids": class_ids, "rois": rois}


def random_detections(rng, H=30, W=40):
    """0-8 detections of scattered pixels, any score, class ids 1-4"""
    N = int(rng.integers(0, 9))
    return {"masks": (rng.random((H, W, N)) < 0.2), "scores": rng.uniform(0, 1, N).astype(np.float32),
            "class_ids": rng.integers(1, 5, N).astype(np.int32), "rois": rng.integers(0, 30, (N, 4)).astype(np.int32)}


out = {}
cases = [(detections(0), 0.0, [], []), (detections(1), 0.7, [], []), (detections(2), 0.5, [1, 2, 3], []),
         (detections(3), 0.4, [], [0, 0, 250, 0, 251, 0]), (detections(4), 0.99, [], [])]
rng = np.random.default_rng(99)
for _ in range(20):
    r = random_detections(rng)
    cf = [1, 3] if rng.random() < 0.5 else []
    cases.append((r, float(rng.uniform(0, 1)), cf, []))
for k, (r, min_score, cf, sa) in enumerate(cases):
    img, cls, rois = helpers.generate_id_image(r, min_score, cf, sa)
    out[f"c{k}_masks"] = r["masks"].astype(np.uint8); out[f"c{k}_scores"] = r["scores"]; out[f"c{k}_class_ids"] = r["class_ids"]; out[f"c{k}_rois"] = r["rois"]
    out[f"c{k}_min_score"] = np.float64(min_score); out[f"c{k}_filter"] = np.array(cf, np.int32); out[f"c{k}_special"] = np.array(sa, np.int32)
    out[f"c{k}_img"] = img; out[f"c{k}_out_cls"] = np.array(cls, np.int32); out[f"c{k}_out_rois"] = np.array(rois, np.int32).reshape(-1, 4)
out["ncases"] = len(cases)
# the mask + description files the reference writes for the -maskdir mode (offline_runner.py -> save_id_image)
r = detections(7); img, cls, rois = helpers.generate_id_image(r, 0.0)
with tempfile.TemporaryDirectory() as d:
    helpers.save_id_image(img, d, "Mask0000", cls, True, rois)
    out["saved_png"] = np.frombuffer(open(os.path.join(d, "Mask0000.png"), "rb").read(), np.uint8)
    out["saved_txt"] = np.frombuffer(open(os.path.join(d, "Mask0000.txt"), "rb").read(), np.uint8)
out["saved_img"] = img; out["saved_cls"] = np.array(cls, np.int32); out["saved_rois"] = np.array(rois, np.int32).reshape(-1, 4)
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "idimage_golden.npz"), **out)
print("wrote", len(cases), "cases;", "exported per case:", [len(out[f"c{k}_out_cls"]) for k in range(len(cases))])
