#!/usr/bin/env python
"""Fuzz the numpy restatement of the label energy terms (oracle/energy_label_terms.py) against the UNMODIFIED reference:
random small label images (2-D / 3-D / 4-D, random region shapes, sometimes the first voxel pair of an axis on a
region border), random images in float32 / float64 / int16 / uint8 / int32, random alpha / directedness.  Every
set_nweight / set_tweight call must agree bit for bit and in order.

``reference_outputs`` runs the reference (needs the reference tree and `make -C oracle pyshim`); its result is stored in
tests/golden/reference_runs_v1.npz by tests/golden/make_golden_reference_runs.py, and tests/test_oracle_labels.py
replays the same cases through ``check`` against that record.  Run directly, the script compares with the live
reference:

    python tests/golden/fuzz_labels_against_reference.py [cases] [seed]
"""
import hashlib
import os
import sys
import warnings

import numpy

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
import make_golden as base  # noqa: E402
from make_golden_labels import Recorder  # noqa: E402
from oracle import energy_label_terms as elt  # noqa: E402

TERMS = ("stawiaski", "directed", "means", "atlas")


def random_case(rng):
    ndim = int(rng.integers(2, 5))
    shape = tuple(int(rng.integers(2, 7 if ndim < 4 else 4)) for _ in range(ndim))
    k = int(rng.integers(1, max(2, int(numpy.prod(shape)) // 2)))
    lab = rng.integers(1, k + 1, size=shape)
    if rng.random() < 0.5:      # smoother regions
        lab = numpy.sort(lab, axis=int(rng.integers(0, ndim)))
    _, inv = numpy.unique(lab, return_inverse=True)
    lab = (inv + 1).reshape(shape)
    dt = [numpy.float32, numpy.float64, numpy.int16, numpy.uint8, numpy.int32][int(rng.integers(0, 5))]
    if numpy.dtype(dt).kind == "f":
        img = (rng.normal(0, 50, size=shape) * (rng.random() < 0.9)).astype(dt)
    else:
        info = numpy.iinfo(dt)
        img = rng.integers(max(info.min + 1, -300), min(info.max, 300) + 1, size=shape).astype(dt)
    prob = rng.uniform(0, 1, size=shape).astype(numpy.float32 if rng.random() < 0.5 else numpy.float64)
    if rng.random() < 0.3:
        lab = numpy.asfortranarray(lab)
    return lab, img, prob, float(rng.uniform(0.01, 2.0)), -float(rng.uniform(0.0, 0.01))


def digest(rows):
    return numpy.frombuffer(hashlib.sha256(numpy.ascontiguousarray(rows, dtype=numpy.float64).tobytes()).digest(), numpy.uint8)


def reference_outputs(cases, seed):
    """The calls the reference's four label terms issue on each random case, as float64 rows (i, j, w, w_back) for the
    n-weights -- difference_of_means sorted, it walks a Python set -- and (node, source, sink) for regional_atlas;
    per term and case the row count (`<term>_n`) and the SHA-256 of the rows' bits (`<term>_sha256`), which keeps the
    record small and the comparison bit for bit."""
    base.import_reference()
    from medpy.graphcut import energy_label as el
    rng = numpy.random.default_rng(seed)
    rows = {t: [] for t in TERMS}
    for _ in range(cases):
        lab, img, prob, alpha, directedness = random_case(rng)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            r = Recorder(); el.boundary_stawiaski(r, lab, img)
            rows["stawiaski"].append(numpy.asarray(r.n, dtype=numpy.float64).reshape(-1, 4))
            r = Recorder(); el.boundary_stawiaski_directed(r, lab, (img, directedness))
            rows["directed"].append(numpy.asarray(r.n, dtype=numpy.float64).reshape(-1, 4))
            r = Recorder(); el.boundary_difference_of_means(r, lab, img)
            rows["means"].append(numpy.asarray(sorted(r.n), dtype=numpy.float64).reshape(-1, 4))
            r = Recorder(); el.regional_atlas(r, lab, (prob, alpha))
            rows["atlas"].append(numpy.asarray(r.t, dtype=numpy.float64).reshape(-1, 3))
    out = {}
    for t in TERMS:
        out[t + "_n"] = numpy.asarray([len(x) for x in rows[t]], numpy.int64)
        out[t + "_sha256"] = numpy.stack([digest(x) for x in rows[t]])
    return out


def check(cases, seed, ref):
    """The restatement's calls on the same cases equal `ref` (reference_outputs' record) bit for bit and in order."""
    rng = numpy.random.default_rng(seed)
    assert all(len(ref[t + "_n"]) == cases for t in TERMS)

    def same(t, c, got):
        return len(got) == ref[t + "_n"][c] and numpy.array_equal(digest(got), ref[t + "_sha256"][c])

    for c in range(cases):
        lab, img, prob, alpha, directedness = random_case(rng)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            got = numpy.stack([numpy.asarray(x, dtype=numpy.float64) for x in elt.stawiaski_calls(lab, img)], axis=1).reshape(-1, 4)
            assert same("stawiaski", c, got), ("stawiaski", c, lab.shape, img.dtype)
            got = numpy.stack([numpy.asarray(x, dtype=numpy.float64) for x in elt.stawiaski_directed_calls(lab, img, directedness)], axis=1).reshape(-1, 4)
            assert same("directed", c, got), ("directed", c, lab.shape, img.dtype)
            got = numpy.stack([numpy.asarray(x, dtype=numpy.float64) for x in elt.difference_of_means_calls(lab, img)], axis=1).reshape(-1, 4)
            assert same("means", c, got), ("means", c, lab.shape, img.dtype)
            nodes, src, snk = elt.regional_atlas_calls(lab, prob, alpha)
            got = numpy.stack([nodes.astype(numpy.float64), src, snk], axis=1)
            assert same("atlas", c, got), ("atlas", c, lab.shape, prob.dtype)


def main():
    cases = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    check(cases, seed, reference_outputs(cases, seed))
    print("ok", cases)


if __name__ == "__main__":
    main()
