#!/usr/bin/env python3
"""Close the marching-cubes parity pin wherever scikit-image exists (it is absent from this image, the wheelhouse and the
reference tree; `requirements.txt:31` of the reference has it commented out, so no version is pinned either).

    python tools/make_skimage_golden.py            # needs `import skimage`; writes tests/golden/skimage_mc.npz
                                                   # and tests/golden/skimage_mc_face_rule.npz

For a handful of seeded fields — a smooth closed surface, a random field full of ambiguous faces, a sparse-decoder-like
field with NaN — stores what `skimage.measure.marching_cubes(vol, level, method="lewiner")` (the reference call,
hy3dgen/shapegen/models/autoencoders/surface_extractors.py:69-73) returns: vertex / face counts, Euler characteristic,
total area, the vertices (sorted, for a set comparison) and the installed scikit-image version.  `tests/test_mc_skimage.py`
compares the CUDA extractor and the oracle against these vectors when the file exists (Chamfer distance, counts, Euler
characteristic; exact vertex SET equality on fields without ambiguous cubes) and is skipped otherwise.
The fields are regenerated from seeds by the test, only skimage's outputs are stored.

`skimage_mc_face_rule.npz` holds the same statistics for `face_rule_fields()`: fields whose only ambiguous cubes are
MC33 case 3 (two inside corners on one face diagonal), which Lewiner's face test alone decides, so there
`MCSurfaceExtractor(face_rule="asymptotic")` must reproduce skimage's face count and Euler characteristic
(`tests/test_mc_face_rule.py`).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def fields():
    """name -> (volume float32, level).  Deterministic; shared with tests/test_mc_skimage.py."""
    out = {}
    x = np.linspace(-1.01, 1.01, 49, dtype=np.float32)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    out["sphere49"] = (np.tanh(20 * (0.6 - np.sqrt(X * X + Y * Y + Z * Z))).astype(np.float32), 0.0)
    out["two_blobs49"] = ((np.exp(-8 * ((X - 0.3) ** 2 + Y ** 2 + Z ** 2)) + np.exp(-8 * ((X + 0.3) ** 2 + Y ** 2 + Z ** 2))).astype(np.float32), 0.45)
    rng = np.random.default_rng(7)
    out["noise24"] = (rng.standard_normal((24, 25, 26)).astype(np.float32), 0.1)          # ambiguous faces everywhere
    band = np.tanh(20 * (0.6 - np.sqrt(X * X + Y * Y + Z * Z))).astype(np.float32)
    band[np.abs(band) > 0.9995] = np.nan                                                  # unvisited voxels of a sparse decoder
    out["band49_nan"] = (band, 0.0)
    return out


def face_pair_field(n=41, seed=11, spacing=4):
    """Background -1 with isolated pairs of positive voxels on a face diagonal, the face's other two corners negative, the
    face in a random one of the three planes.  Every pair makes the two cubes sharing that face MC33 case 3 and nothing
    else ambiguous; random values make about half of the faces connect (no near-ties: |p q - r s| >= 0.05)."""
    rng = np.random.default_rng(seed)
    vol = np.full((n, n, n), -1.0, np.float32)
    for x in range(1, n - 2, spacing):
        for y in range(1, n - 2, spacing):
            for z in range(1, n - 2, spacing):
                while True:
                    p, q = rng.uniform(0.2, 2.0, 2)
                    r, s = -rng.uniform(0.2, 2.0, 2)
                    if abs(p * q - r * s) >= 0.05:
                        break
                normal = rng.integers(3)
                u, w = [a for a in range(3) if a != normal]                   # the face spans axes u and w
                base = np.array([x, y, z])
                du, dw = np.eye(3, dtype=int)[u], np.eye(3, dtype=int)[w]
                vol[tuple(base)], vol[tuple(base + du + dw)] = p, q
                vol[tuple(base + du)], vol[tuple(base + dw)] = r, s
    return vol


def face_rule_fields():
    """name -> (volume float32, level): fields whose ambiguous cubes are all MC33 case 3.  Deterministic; shared with
    tests/test_mc_face_rule.py."""
    return {"face_pairs41": (face_pair_field(), 0.0), "face_pairs41_level": (face_pair_field(seed=12) + 0.25, 0.25)}


def mesh_stats(v, f):
    e = np.sort(np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]), 1)
    ne = len(np.unique(e, axis=0))
    fin = np.isfinite(v).all(1)
    ok = fin[f].all(1)
    a, b, c = (v[f[ok][:, i]].astype(np.float64) for i in range(3))
    area = float(0.5 * np.linalg.norm(np.cross(b - a, c - a), axis=1).sum())
    return {"V": int(len(v)), "F": int(len(f)), "euler": int(len(v) - ne + len(f)), "area": area}


def main():
    try:
        import skimage
        from skimage import measure
    except ImportError:
        print("scikit-image is not installed here: nothing written (the marching-cubes oracle stays PARITY UNPINNED)")
        return 1
    write(measure, skimage.__version__, fields(), "skimage_mc.npz")
    write(measure, skimage.__version__, face_rule_fields(), "skimage_mc_face_rule.npz")
    return 0


def write(measure, version, flds, fname):
    out = {"skimage_version": np.array(version)}
    for name, (vol, level) in flds.items():
        v, f, _, _ = measure.marching_cubes(vol, level, method="lewiner")
        st = mesh_stats(v, f)
        key = np.lexsort(v.T[::-1])
        out[name + "_verts_sorted"] = v[key].astype(np.float32)
        out[name + "_faces"] = f.astype(np.int32)
        out[name + "_verts"] = v.astype(np.float32)
        for k, val in st.items():
            out[f"{name}_{k}"] = np.array(val)
        print(name, st)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", fname), **out)
    print(f"wrote tests/golden/{fname} (scikit-image", version, ")")


if __name__ == "__main__":
    sys.exit(main())
