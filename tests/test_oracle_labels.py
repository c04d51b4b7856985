"""The numpy restatement of the label-graph energy terms (oracle/energy_label_terms.py) against what the unmodified
reference did on the same inputs (tests/golden/golden_labels_v1.npz, made by tests/golden/make_golden_labels.py):
every set_nweight / set_tweight call, bit for bit and in the reference's order; whole graph_from_labels cuts through
the real BK solver where oracle/_ref is built.  The general-graph BK restatement and the label-term fuzz compare with
the reference's outputs recorded on seeded inputs (tests/golden/reference_runs_v1.npz)."""
import os
import sys

import numpy
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from oracle import energy_label_terms as elt  # noqa: E402
from oracle import solvers  # noqa: E402
import make_golden_reference_runs as reference_runs  # noqa: E402

G = numpy.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_labels_v1.npz"))
NAMES = [str(n) for n in G["names"]]
FULL = [n for n in NAMES if n + "/directed" in G.files]


def _label(nm):
    lab = G[nm + "/label"]
    return numpy.asfortranarray(lab) if bool(G[nm + "/label_forder"]) else lab


def _calls(t):
    return numpy.stack([numpy.asarray(x, dtype=numpy.float64) for x in t], axis=1).reshape(-1, 4)


@pytest.mark.parametrize("nm", NAMES)
def test_stawiaski_calls_bit_exact(nm):
    got = _calls(elt.stawiaski_calls(_label(nm), G[nm + "/image"]))
    want = G[nm + "/stawiaski"]
    assert got.shape == want.shape
    assert numpy.array_equal(got.view(numpy.uint64), want.view(numpy.uint64))


@pytest.mark.parametrize("nm", NAMES)
def test_difference_of_means_calls_bit_exact(nm):
    i, j, w, w2 = elt.difference_of_means_calls(_label(nm), G[nm + "/image"])
    got = _calls((i, j, w, w2))
    want = G[nm + "/means"]          # sorted by (i, j): the reference walks a Python set
    # the reference passes edges as (min, max) already
    assert got.shape == want.shape
    assert numpy.array_equal(got.view(numpy.uint64), want.view(numpy.uint64))


@pytest.mark.parametrize("nm", FULL)
def test_directed_calls_bit_exact(nm):
    got = _calls(elt.stawiaski_directed_calls(_label(nm), G[nm + "/image"], float(G[nm + "/directedness"])))
    want = G[nm + "/directed"]
    assert got.shape == want.shape
    assert numpy.array_equal(got.view(numpy.uint64), want.view(numpy.uint64))


@pytest.mark.parametrize("nm", FULL)
def test_atlas_calls_bit_exact(nm):
    nodes, src, snk = elt.regional_atlas_calls(_label(nm), G[nm + "/prob"], float(G[nm + "/alpha"]))
    got = numpy.stack([nodes.astype(numpy.float64), src, snk], axis=1)
    want = G[nm + "/atlas"]
    assert numpy.array_equal(got.view(numpy.uint64), want.view(numpy.uint64))


def test_check_label_image():
    with pytest.raises(AttributeError):
        elt.check_label_image(numpy.asarray([[1, 4, 8], [1, 3, 10]]))        # tests/graphcut_/energy_label.py:106-113
    with pytest.raises(AttributeError):
        elt.check_label_image(numpy.asarray([[2, 3, 4], [2, 3, 4]]))         # :115-122
    assert elt.check_label_image(numpy.asarray([[1, 2], [3, 3]])) == 3


def label_problem(nm, tag):
    """(n, i, j, cap, rev, tw_ops) of one golden graph_from_labels run, in the reference's call order."""
    lab, img = _label(nm), G[nm + "/image"]
    n = int(lab.max())
    tw = []
    if tag == "cut_stawiaski":
        e = elt.stawiaski_calls(lab, img)
    elif tag == "cut_means":
        e = elt.difference_of_means_calls(lab, img)
    else:
        tw.append(elt.regional_atlas_calls(lab, G[nm + "/prob"], float(G[nm + "/alpha"])))
        e = elt.stawiaski_directed_calls(lab, img, float(G[nm + "/directedness"]))
    fgr = elt.marker_regions(lab, G[nm + "/fg"])
    bgr = elt.marker_regions(lab, G[nm + "/bg"])
    tw.append((fgr, numpy.full(fgr.size, 65535.0), numpy.zeros(fgr.size)))
    tw.append((bgr, numpy.zeros(bgr.size), numpy.full(bgr.size, 65535.0)))
    return n, e[0], e[1], e[2], e[3], tw


@pytest.mark.skipif(not solvers.have_ref(), reason="oracle/_ref not built")
@pytest.mark.parametrize("tag", ["cut_stawiaski", "cut_means", "cut_directed_atlas"])
@pytest.mark.parametrize("nm", FULL)
def test_whole_cut_through_reference_bk(nm, tag):
    n, i, j, cap, rev, tw = label_problem(nm, tag)
    flow, mask, _ = solvers.solve_sparse_ref(n, i, j, cap, rev, tw)
    assert numpy.array_equal(mask, G[nm + "/" + tag + "_mask"])
    want = float(G[nm + "/" + tag + "_flow"])
    if tag == "cut_means":           # arc insertion order of the reference's set walk is not reproducible: value only
        assert flow == pytest.approx(want, rel=1e-12, abs=1e-300)
    else:
        assert flow == want


# ---- the BK restatement for general graphs (oracle/bk_sparse.c) ------------------------------------------------------
@pytest.mark.parametrize("seed", reference_runs.SPARSE_SEEDS)
def test_sparse_port_equals_reference_bk_bit_for_bit(seed):
    z = reference_runs.load()
    n, i, j, cap, rev, tw = reference_runs.sparse_case(seed)
    before = sum(reference_runs.sparse_case(s)[0] for s in range(seed))
    rflow, rmask = z["sparse/flow"][seed], z["sparse/mask"][before:before + n]
    pflow, pmask, _ = solvers.solve_sparse_port(n, i, j, cap, rev, tw)
    assert pflow == rflow                      # same arc order => same augmentations => same float64 flow
    assert numpy.array_equal(pmask, rmask)


@pytest.mark.parametrize("tag", ["cut_stawiaski", "cut_means", "cut_directed_atlas"])
@pytest.mark.parametrize("nm", FULL)
def test_sparse_port_on_golden_region_graphs(nm, tag):
    n, i, j, cap, rev, tw = label_problem(nm, tag)
    flow, mask, _ = solvers.solve_sparse_port(n, i, j, cap, rev, tw)
    assert numpy.array_equal(mask, G[nm + "/" + tag + "_mask"])
    want = float(G[nm + "/" + tag + "_flow"])
    if tag == "cut_means":
        assert flow == pytest.approx(want, rel=1e-12, abs=1e-300)
    else:
        assert flow == want


def test_sparse_port_reference_diamond():
    """lib/maxflow/src/sum_edge_test.py:20-37: flow 2, and 4 once every edge was summed a second time."""
    e = [(0, 1), (0, 2), (1, 3), (2, 3)]
    tw = [(numpy.asarray([0, 3]), numpy.asarray([99.0, 0.0]), numpy.asarray([0.0, 99.0]))]
    i, j = numpy.asarray([a for a, _ in e]), numpy.asarray([b for _, b in e])
    flow, mask, _ = solvers.solve_sparse_port(4, i, j, numpy.ones(4), numpy.zeros(4), tw)
    assert flow == 2.0
    flow, mask, _ = solvers.solve_sparse_port(4, numpy.tile(i, 2), numpy.tile(j, 2), numpy.ones(8), numpy.zeros(8), tw)
    assert flow == 4.0 and mask.tolist() == [1, 1, 1, 0]


def test_label_oracle_fuzzed_against_the_live_reference():
    """150 random label images (2-D..4-D, five image dtypes, F order, random alpha / directedness): every call the
    reference issues equals the restatement's, bit for bit (tests/golden/fuzz_labels_against_reference.py, replayed
    against the reference's recorded calls)."""
    import fuzz_labels_against_reference as fuzz
    z = reference_runs.load()
    cases, seed = reference_runs.LAB_FUZZ
    fuzz.check(cases, seed, {k[4:]: z[k] for k in z.files if k.startswith("lab/")})
