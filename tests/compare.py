"""Keypoint-set comparison (SURVEY.md Appendix B): canonical one-to-one pairing with tolerance."""
import numpy as np


def pair_points(a, b, pos_tol=0.05, scale_rel=0.02, ori_tol=2.0):
    """Greedy one-to-one pairing of records a -> b on (subsampling, x, y, scale, orientation).
    Returns (index pairs, unmatched_a, unmatched_b)."""
    used = np.zeros(len(b), bool)
    pairs = []
    order = np.lexsort((b["xpos"], b["ypos"]))
    by = b["ypos"][order]
    for i in range(len(a)):
        p = a[i]
        tol = pos_tol * max(1.0, p["subsampling"])
        lo, hi = np.searchsorted(by, p["ypos"] - tol), np.searchsorted(by, p["ypos"] + tol)
        best, bestd = -1, 1e9
        for j in order[lo:hi]:
            if used[j]:
                continue
            q = b[j]
            if q["subsampling"] != p["subsampling"]:
                continue
            if abs(q["xpos"] - p["xpos"]) > tol:
                continue
            if abs(q["scale"] - p["scale"]) > scale_rel * p["scale"]:
                continue
            do = abs(q["orientation"] - p["orientation"]) % 360.0
            do = min(do, 360.0 - do)
            if not (do <= ori_tol):
                continue
            d = abs(q["xpos"] - p["xpos"]) + abs(q["ypos"] - p["ypos"]) + do * 0.01
            if d < bestd:
                best, bestd = j, d
        if best >= 0:
            used[best] = True
            pairs.append((i, best))
    ua = sorted(set(range(len(a))) - {i for i, _ in pairs})
    ub = list(np.nonzero(~used)[0])
    return pairs, ua, ub


def compare_sets(a, b, **kw):
    """Summary dict: matched fraction (both ways) and worst relative errors over the pairs."""
    pairs, ua, ub = pair_points(a, b, **kw)
    out = {"na": len(a), "nb": len(b), "pairs": len(pairs), "unmatched_a": len(ua), "unmatched_b": len(ub)}
    if pairs:
        ia = np.array([i for i, _ in pairs]); ib = np.array([j for _, j in pairs])
        pa, pb = a[ia], b[ib]
        out["pos_err"] = float(np.max(np.maximum(np.abs(pa["xpos"] - pb["xpos"]), np.abs(pa["ypos"] - pb["ypos"]))
                                      / np.maximum(1.0, pa["subsampling"])))
        out["scale_rel"] = float(np.max(np.abs(pa["scale"] - pb["scale"]) / pa["scale"]))
        do = np.abs(pa["orientation"] - pb["orientation"]) % 360.0
        out["ori_err"] = float(np.max(np.minimum(do, 360.0 - do)))
        dd = np.abs(pa["data"] - pb["data"])
        finite = np.isfinite(dd).all(axis=1)
        out["desc_max"] = float(dd[finite].max()) if finite.any() else 0.0
        out["desc_med"] = float(np.median(dd[finite].max(axis=1))) if finite.any() else 0.0
        out["desc_bad"] = int((dd[finite].max(axis=1) > 1e-3).sum())
        out["sharp_rel"] = float(np.max(np.abs(pa["sharpness"] - pb["sharpness"]) / np.maximum(1e-3, np.abs(pa["sharpness"]))))
    return out


def reference_summary(r1, r2, seed, sample=32):
    """What is kept of two reference ExtractSift runs on one input (both in canonical order): the counts, sha256 of
    the fields that must match bit for bit, every orientation, the run-to-run noise of orientations and descriptors,
    the rows whose descriptor is not finite, and the descriptors of a seeded sample of rows (sample=None: all rows)."""
    import hashlib
    assert len(r1) == len(r2), (len(r1), len(r2))
    out = {"count1": np.int32(len(r1)), "count2": np.int32(len(r2))}
    for f in ("xpos", "ypos", "scale", "sharpness", "edgeness", "subsampling"):
        out[f + "_sha"] = hashlib.sha256(np.ascontiguousarray(r1[f]).tobytes()).hexdigest()
    do = np.abs(r1["orientation"] - r2["orientation"]) % 360.0
    fin1 = np.isfinite(r1["data"]).all(axis=1)
    fin = fin1 & np.isfinite(r2["data"]).all(axis=1)
    dn = np.abs(r1["data"][fin] - r2["data"][fin]).max(axis=1)
    n = len(r1) if sample is None else min(sample, len(r1))
    rows = np.sort(np.random.default_rng(seed).choice(len(r1), n, replace=False)).astype(np.int32)
    out.update(orientation=r1["orientation"].copy(), ori_noise=float(np.minimum(do, 360.0 - do).max()),
               desc_noise=float(dn.max()), desc_bad_noise=np.int32((dn > 2e-5).sum()),
               nonfinite=np.nonzero(~fin1)[0].astype(np.int32), rows=rows, data=r1["data"][rows].copy())
    return out
