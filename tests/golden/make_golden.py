"""Generate golden vectors from the REFERENCE's own code run in the build container.

    python tests/golden/make_golden.py

Needs oracle/_ref/{knn_ref,dq_ref} (built by `make -C oracle ref` from /root/reference: the vendored nanoflann + the
reference's knn_point_cloud.hpp / quaternion.hpp / dual_quaternion.hpp, compiled as they lie).  Writes
tests/golden/knn_ref.json and tests/golden/dq_ref.json; floats are stored as C99 hex strings so they round-trip exactly.
tests/golden/knn_ref_random.npz holds the reference's 8-NN of the random clouds of tests/test_oracle_golden.py.
/root/reference does not exist on the GPU box, so the committed JSON files are what the tests read there."""
import json
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
REF = HERE.parents[1] / "oracle" / "_ref"


def hexf(a):
    return [float(np.float32(v)).hex() for v in np.asarray(a, np.float32).ravel()]


def knn():
    rng = np.random.default_rng(20260923)
    cases = []
    for P, Q, spread in ((8, 5, 0.0), (40, 60, 1.0), (500, 120, 1.0), (2000, 80, 0.3)):
        if P == 8:       # the reference's tests/nanoflann_test.cpp inputs
            pts = np.array([(1, 1, 1), (1, 1, -1), (1, -1, 1), (1, -1, -1), (-1, 1, 1), (-1, 1, -1), (-1, -1, 1), (-1, -1, -1)], np.float32)
            qs = np.array([(-1, -1, -1), (0, 0, 0), (1, 1, 1), (2, 2, 2), (3, 3, 3)], np.float32)
        else:
            pts = rng.uniform(-spread, spread, (P, 3)).astype(np.float32)
            qs = rng.uniform(-1.2 * spread, 1.2 * spread, (Q, 3)).astype(np.float32)
        inp = f"{len(pts)} {len(qs)}\n" + "\n".join(" ".join(repr(float(v)) for v in p) for p in np.vstack([pts, qs]))
        out = subprocess.run([str(REF / "knn_ref")], input=inp, capture_output=True, text=True, check=True).stdout.split()
        cases.append({"points": hexf(pts), "queries": hexf(qs), "idx": [int(v) for v in out[0::2]], "d2": out[1::2]})
    (HERE / "knn_ref.json").write_text(json.dumps({"source": "reference nanoflann + knn_point_cloud.hpp via oracle/ref_shim/knn_ref.cpp", "cases": cases}))


def knn_random():
    """the seeded clouds of tests/test_oracle_golden.py::test_knn_matches_reference_nanoflann_binary"""
    rng = np.random.default_rng(5)
    pts = rng.uniform(-1, 1, (300, 3)).astype(np.float32)
    qs = rng.uniform(-1.2, 1.2, (200, 3)).astype(np.float32)
    inp = f"{len(pts)} {len(qs)}\n" + "\n".join(" ".join(repr(float(v)) for v in p) for p in np.vstack([pts, qs]))
    out = subprocess.run([str(REF / "knn_ref")], input=inp, capture_output=True, text=True, check=True).stdout.split()
    idx = np.array(out[0::2], np.int16).reshape(len(qs), 8)
    d2 = np.array([np.float32(float.fromhex(v)) for v in out[1::2]], np.float32).reshape(len(qs), 8)
    np.savez_compressed(HERE / "knn_ref_random.npz", idx=idx, d2=d2)


def dq():
    rng = np.random.default_rng(7)
    K = 150
    lines, cases = [str(K)], []
    for c in range(K):
        rot = rng.normal(size=(8, 4)).astype(np.float32)
        rot /= np.linalg.norm(rot, axis=1, keepdims=True).astype(np.float32)
        if c % 4 == 0:
            rot[:] = (1, 0, 0, 0)                       # the live pipeline: identity rotations
        else:
            rot[:, 0] = np.abs(rot[:, 0]) + np.float32(0.5)
        t = rng.normal(scale=0.05, size=(8, 3)).astype(np.float32)
        w = rng.uniform(0.0, 1.0, 8).astype(np.float32)
        p = rng.uniform(-1, 1, 3).astype(np.float32)
        for i in range(8):
            lines.append(" ".join(repr(float(v)) for v in (*rot[i], *t[i], w[i])))
        lines.append(" ".join(repr(float(v)) for v in p))
        cases.append({"rot": hexf(rot), "t": hexf(t), "w": hexf(w), "p": hexf(p)})
    out = subprocess.run([str(REF / "dq_ref")], input="\n".join(lines), capture_output=True, text=True, check=True).stdout.split("\n")
    for c, line in zip(cases, out):
        v = line.split()
        c["rot_out"], c["p_out"] = v[:4], v[4:7]
    (HERE / "dq_ref.json").write_text(json.dumps({"source": "reference quaternion.hpp + dual_quaternion.hpp via oracle/ref_shim/dq_ref.cpp", "cases": cases}))


if __name__ == "__main__":
    knn()
    knn_random()
    dq()
    print("wrote", HERE / "knn_ref.json", HERE / "knn_ref_random.npz", HERE / "dq_ref.json")
