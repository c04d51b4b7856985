#!/usr/bin/env python
"""Generate tests/golden/reference_runs_v1.npz: what the UNMODIFIED reference computed on the seeded inputs of the
oracle tests, so that those tests compare with the reference without it being present.

Needs the reference tree and `make -C oracle ref pyshim`:

    python tests/golden/make_golden_reference_runs.py

Recorded, with the inputs defined here or in the fuzz scripts (the tests regenerate them from the same seeds):

* ``vox/*``      -- fuzz_voxels_against_reference.reference_outputs(VOX_FUZZ)   (tests/test_oracle.py)
* ``lab/*``      -- fuzz_labels_against_reference.reference_outputs(LAB_FUZZ)   (tests/test_oracle_labels.py)
* ``lattice/*``  -- the reference BK (oracle/_ref/libbkref.so) on random_lattices(): flow and mask per lattice
* ``blob32/*``   -- the reference BK on blob32_problem()
* ``sparse/*``   -- the reference BK on sparse_case(seed) for SPARSE_SEEDS
* ``dimacs`` / ``inconsistent`` -- the reference's medpy.graphcut.Graph + graph_to_dimacs on fill_graph(), and
  Graph.inconsistent() on fill_inconsistent() (tests/test_host_labels.py)
"""
import io
import os
import re
import sys

import numpy

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

PATH = os.path.join(HERE, "reference_runs_v1.npz")
VOX_FUZZ = (120, 11)      # (cases, seed)
LAB_FUZZ = (150, 7)
SPARSE_SEEDS = range(40)


def random_lattices():
    """120 random integer-capacity lattices, 1-D..4-D, as build_problem() dicts."""
    rng = numpy.random.default_rng(7)
    for _ in range(120):
        nd = int(rng.integers(1, 5))
        shape = tuple(int(x) for x in rng.integers(1, 7, size=nd))
        n = int(numpy.prod(shape))
        wf = [rng.integers(0, 3, size=n).astype(float) for _ in range(nd)]
        wb = [rng.integers(0, 3, size=n).astype(float) for _ in range(nd)]
        tr = rng.integers(-3, 4, size=n).astype(float)
        yield dict(shape=shape, wf=wf, wb=wb, tr=tr, flow_const=0.0, fg=numpy.zeros(n, numpy.uint8),
                   bg=numpy.zeros(n, numpy.uint8), src=numpy.maximum(tr, 0), snk=numpy.maximum(-tr, 0))


def blob32_problem():
    """The bench workload's generator at 32^3, float64 terms."""
    from medpy_b200 import synthetic
    from oracle import energy_terms as et
    vol = synthetic.two_blob_volume((32, 32, 32), seed=0)
    return et.build_problem(vol["fg"], vol["bg"], regional=(vol["prob"], 0.1),
                            boundary=("difference_exponential", vol["image"], vol["sigma"], False))


def sparse_case(seed):
    """(n, i, j, cap, rev, tw_ops) of a random general graph; even seeds integer capacities, odd seeds real ones with
    negative t-weights."""
    rng = numpy.random.default_rng(1000 + seed)
    n = int(rng.integers(2, 600))
    m = int(rng.integers(1, 8 * n))
    i = rng.integers(0, n, size=m)
    j = rng.integers(0, n, size=m)
    keep = i != j
    i, j = i[keep], j[keep]
    if seed % 2 == 0:
        cap = rng.integers(0, 20, size=i.size).astype(float)      # zero capacities are legal for sum_edge (graph.h:461)
        rev = rng.integers(0, 20, size=i.size).astype(float)
        src = rng.integers(0, 30, size=n).astype(float)
        snk = rng.integers(0, 30, size=n).astype(float)
    else:
        cap = rng.uniform(1e-3, 2.0, size=i.size)
        rev = rng.uniform(1e-3, 2.0, size=i.size)
        src = rng.uniform(0, 3.0, size=n)
        snk = rng.uniform(-0.5, 3.0, size=n)                        # negative t-weights are legal (graph.py:462-498)
    fg = rng.choice(n, size=max(1, n // 20), replace=False)
    bg = rng.choice(n, size=max(1, n // 20), replace=False)
    tw = [(numpy.arange(n), src, snk), (fg, numpy.full(fg.size, 65535.0), numpy.zeros(fg.size)),
          (bg, numpy.zeros(bg.size), numpy.full(bg.size, 65535.0))]
    return n, i, j, cap, rev, tw


def fill_graph(g):
    g.set_nodes(5)
    g.set_nweights({(1, 2): (0.5, 0.25), (2, 3): (1, 0), (4, 5): (0, 2.5)})
    g.add_tweights({3: (0.1, 0.9), 4: (0, 0)})
    g.set_source_nodes([1, 2])
    g.set_sink_nodes([5])
    return g


def fill_inconsistent(g):
    g.set_nodes(2)
    g.set_nweights({(1, 2): (1, 1), (2, 1): (1, 1), (1, 3): (1, 1)})
    g.set_sink_nodes([7])
    return g


def load():
    return numpy.load(PATH)


def text(z, key):
    return bytes(z[key]).decode()


def _reference_graph_module():
    """medpy/graphcut/{graph,write}.py of the reference, without the compiled solver binding they do not need."""
    import make_golden as base
    names = {}
    for mod in ("graph", "write"):
        with open(os.path.join(base.REF, "medpy", "graphcut", mod + ".py")) as fh:
            src = fh.read()
        src = re.sub(r"^from \.maxflow import .*$", "GraphDouble = None", src, flags=re.M)
        ns = {"__name__": "reference_" + mod}
        exec(compile(src, mod, "exec"), ns)
        names[mod] = ns
    return names


def main():
    import fuzz_labels_against_reference as flab
    import fuzz_voxels_against_reference as fvox
    from oracle import solvers
    if not solvers.have_ref():
        raise SystemExit("run `make -C oracle ref pyshim` first")
    out = {}
    for key, mod, (cases, seed) in (("vox", fvox, VOX_FUZZ), ("lab", flab, LAB_FUZZ)):
        rec = mod.reference_outputs(cases, seed)
        mod.check(cases, seed, rec)
        out.update({key + "/" + k: v for k, v in rec.items()})
    flows, masks = [], []
    for prob in random_lattices():
        f, m, _ = solvers.solve_ref(prob)
        flows.append(f)
        masks.append(m.ravel())
    out["lattice/flow"] = numpy.asarray(flows)
    out["lattice/mask"] = numpy.concatenate(masks)
    f, m, _ = solvers.solve_ref(blob32_problem())
    out["blob32/flow"] = numpy.float64(f)
    out["blob32/mask"] = m
    flows, masks = [], []
    for seed in SPARSE_SEEDS:
        f, m, _ = solvers.solve_sparse_ref(*sparse_case(seed))
        flows.append(f)
        masks.append(m)
    out["sparse/flow"] = numpy.asarray(flows)
    out["sparse/mask"] = numpy.concatenate(masks)
    ref = _reference_graph_module()
    buf = io.StringIO()
    ref["write"]["graph_to_dimacs"](fill_graph(ref["graph"]["Graph"]()), buf)
    out["dimacs"] = numpy.frombuffer(buf.getvalue().encode(), numpy.uint8)
    msgs = sorted(fill_inconsistent(ref["graph"]["Graph"]()).inconsistent())
    out["inconsistent"] = numpy.frombuffer("\n".join(msgs).encode(), numpy.uint8)
    numpy.savez_compressed(PATH, **out)
    print("wrote", PATH, "bytes:", os.path.getsize(PATH))


if __name__ == "__main__":
    main()
