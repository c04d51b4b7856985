#!/usr/bin/env python
"""Fuzz the voxel-path oracle (oracle/energy_terms.py + oracle/bk_lattice.c) against the UNMODIFIED reference: random
small lattices (1-D..4-D), the eight boundary terms, five image dtypes, random sigma / spacing / regional term / marker
overlap.  The n-link weights (get_edge), net t-links (get_trcap), the flow maxflow() returns and the what_segment mask of
the reference's own graph_from_voxels must equal the restatement's, bit for bit.

``reference_outputs`` runs the reference (needs the reference tree and `make -C oracle pyshim`); its result is stored in
tests/golden/reference_runs_v1.npz by tests/golden/make_golden_reference_runs.py, and tests/test_oracle.py replays the
same cases through ``check`` against that record.  Run directly, the script compares with the live reference:

    python tests/golden/fuzz_voxels_against_reference.py [cases] [seed]
"""
import os
import sys
import warnings

import numpy

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
import make_golden as base  # noqa: E402
from oracle import energy_terms as et  # noqa: E402
from oracle import solvers  # noqa: E402


def random_case(rng):
    ndim = int(rng.integers(1, 5))
    shape = tuple(int(rng.integers(2, [0, 12, 7, 5, 4][ndim])) for _ in range(ndim))
    term = base.TERMS[int(rng.integers(0, 8))]
    dt = [numpy.float32, numpy.float64, numpy.int16, numpy.uint8, numpy.int32][int(rng.integers(0, 5))]
    if numpy.dtype(dt).kind == "f":
        img = rng.normal(0, 40, size=shape).astype(dt)
    else:
        info = numpy.iinfo(dt)
        img = rng.integers(max(info.min + 1, -200), min(info.max, 200) + 1, size=shape).astype(dt)
    fn = term.split("_")[1]
    sigma = None if fn == "linear" else float(rng.uniform(0.5, 30.0))
    spacing = tuple(float(x) for x in rng.uniform(0.5, 3.0, size=ndim)) if rng.random() < 0.4 else False
    fg = rng.random(shape) < 0.1
    bg = rng.random(shape) < 0.1
    fg.flat[0] = True
    bg.flat[-1] = True
    c = dict(name="fuzz", fg=fg, bg=bg, boundary=term, image=img, sigma=sigma, spacing=spacing)
    if rng.random() < 0.4:
        c["prob"] = rng.uniform(0, 1, size=shape).astype(numpy.float32 if rng.random() < 0.5 else numpy.float64)
        c["alpha"] = float(rng.uniform(0.05, 3.0))
    return c


def reference_outputs(cases, seed):
    """The reference's graph_from_voxels on the first `cases` random lattices that it accepts, in generation order:
    error[k] = 1 where it raised ValueError (weights <= 0) on the k-th generated lattice; for the others, concatenated,
    the n-link weights (ndim x n each), t-links, flow and mask."""
    gc = base.import_reference()
    rng = numpy.random.default_rng(seed)
    error, w_all, tr_all, flow_all, mask_all = [], [], [], [], []
    while len(flow_all) < cases:
        c = random_case(rng)
        with warnings.catch_warnings(), numpy.errstate(all="ignore"):
            warnings.simplefilter("ignore")
            try:
                w, tr, flow, mask = base.run_case(gc, c)
            except ValueError:
                error.append(1)
                continue
        error.append(0)
        w_all.append(w.ravel())
        tr_all.append(tr)
        flow_all.append(flow)
        mask_all.append(mask.astype(numpy.uint8).ravel())
    return {"error": numpy.asarray(error, numpy.uint8), "w": numpy.concatenate(w_all), "tr": numpy.concatenate(tr_all),
            "flow": numpy.asarray(flow_all, numpy.float64), "mask": numpy.concatenate(mask_all)}


def check(cases, seed, ref):
    """The restatement on the same lattices equals `ref` (reference_outputs' record) bit for bit, and refuses exactly
    the lattices the reference refused.  Returns the number of refused lattices."""
    rng = numpy.random.default_rng(seed)
    done = skipped = 0
    ow = ot = om = 0
    while done < cases:
        c = random_case(rng)
        k = done + skipped
        with warnings.catch_warnings(), numpy.errstate(all="ignore"):
            warnings.simplefilter("ignore")
            boundary = (c["boundary"], c["image"], c["sigma"], c["spacing"])
            regional = (c["prob"], c["alpha"]) if c.get("prob") is not None else None
            try:
                prob = et.build_problem(c["fg"], c["bg"], regional=regional, boundary=boundary)
                our_error = None
            except ValueError as e:
                our_error = e
        assert bool(ref["error"][k]) == (our_error is not None), (k, c["boundary"], c["image"].dtype, our_error)
        if our_error is not None:
            skipped += 1
            continue
        n = c["fg"].size
        nd = c["fg"].ndim
        w = ref["w"][ow:ow + nd * n].reshape(nd, n)
        tr = ref["tr"][ot:ot + n]
        mask = ref["mask"][om:om + n].reshape(c["fg"].shape)
        ow, ot, om = ow + nd * n, ot + n, om + n
        for d in range(len(prob["shape"])):
            assert numpy.array_equal(prob["wf"][d], w[d], equal_nan=True), ("weights", k, c["boundary"], c["image"].dtype, d)
        assert numpy.array_equal(prob["tr"], tr), ("t-links", k, c["boundary"])
        if not numpy.isnan(w).any():
            pflow, pmask, _ = solvers.solve_port(prob)
            assert pflow == ref["flow"][done], ("flow", k, c["boundary"], pflow, ref["flow"][done])
            assert numpy.array_equal(pmask, mask), ("mask", k, c["boundary"])
        done += 1
    assert (ow, ot, om) == (ref["w"].size, ref["tr"].size, ref["mask"].size)
    return skipped


def main():
    cases = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    skipped = check(cases, seed, reference_outputs(cases, seed))
    print("ok", cases, "value-error cases agreed:", skipped)


if __name__ == "__main__":
    main()
