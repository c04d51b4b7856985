"""CPU tests (no GPU) of the host side of the region-graph path: signatures and error conventions of
medpy_b200.graphcut.energy_label / graph_from_labels, the sparse GraphDouble staging, the compat ``medpy.filter``
helpers, and that nothing falls back to a CPU solver."""
import inspect
import os
import sys

import numpy
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _no_gpu():
    import torch
    return not torch.cuda.is_available()


def test_label_terms_keep_reference_signature():
    from medpy_b200.graphcut import energy_label
    assert sorted(energy_label.__all__) == ["boundary_difference_of_means", "boundary_stawiaski",
                                            "boundary_stawiaski_directed", "regional_atlas"]
    for name in energy_label.__all__:   # graph_from_labels checks 3 == len(getargspec(f)[0]) (generate.py:278-289)
        assert len(inspect.getfullargspec(getattr(energy_label, name))[0]) == 3, name


def test_graph_from_labels_arity_errors():
    from medpy_b200.graphcut import graph_from_labels
    lab = numpy.asarray([[1, 2], [1, 2]])
    z = numpy.zeros((2, 2), bool)
    with pytest.raises(AttributeError):
        graph_from_labels(lab, z, z, boundary_term=lambda a, b: None)
    with pytest.raises(AttributeError):
        graph_from_labels(lab, z, z, regional_term=lambda a, b, c, d: None)
    with pytest.raises(AttributeError):
        graph_from_labels(lab, z, z, boundary_term=3)


def test_label_images_that_cannot_be_consecutive_are_rejected_on_the_host():
    from medpy_b200.graphcut.energy_label import LabelContext
    with pytest.raises(AttributeError):
        LabelContext(numpy.asarray([[0, 1], [1, 2]], dtype=numpy.int64))     # ids must start at 1
    with pytest.raises(AttributeError):
        LabelContext(numpy.asarray([[1.5, 1.0]]))
    with pytest.raises(AttributeError):
        LabelContext(numpy.zeros((0, 3), dtype=numpy.int32))


@pytest.mark.skipif(not _no_gpu(), reason="a GPU is present")
def test_no_cpu_fallback_for_region_graphs():
    from medpy_b200.graphcut import GCGraph, energy_label, graph_from_labels
    lab = numpy.asarray([[1, 2], [1, 2]], dtype=numpy.int32)
    z = numpy.zeros((2, 2), bool)
    with pytest.raises(RuntimeError, match="CUDA"):
        graph_from_labels(lab, z, z, boundary_term=energy_label.boundary_stawiaski, boundary_term_args=numpy.zeros((2, 2)))
    g = GCGraph(4, 4, sparse=True)
    g.set_nweight(0, 3, 1.0, 2.0)
    g.set_tweight(0, 5.0, 0.0)
    with pytest.raises(RuntimeError, match="CUDA"):
        g.get_graph().maxflow()


def test_sparse_staging_keeps_call_order_and_validates():
    from medpy_b200.graphcut import GCGraph
    from medpy_b200.graphcut.sparse import SparseGraphDouble
    g = SparseGraphDouble(5, 10)
    g.sum_edge(0, 4, 1.0, 2.0)
    g.add_tweights(1, 3.0, 0.0)
    g.sum_edge(4, 0, 0.5, 0.25)
    g.sum_edges_bulk([1, 2], [3, 4], [1.0, 1.0], [2.0, 2.0])
    g.add_tweights_bulk(None, numpy.arange(5.0), numpy.zeros(5))
    g._close_edges(); g._close_tweights()
    kinds = [op[0] for op in g._ops]
    assert kinds.count("e") == 2 and kinds.count("t") == 2
    first = [op for op in g._ops if op[0] == "e"][0]
    assert first[1].tolist() == [0, 4] and first[2].tolist() == [4, 0]            # the two element-wise calls, in order
    with pytest.raises(ValueError):
        g.sum_edge(0, 0, 1, 1)
    with pytest.raises(ValueError):
        g.sum_edges_bulk([0], [5], [1.0], [1.0])
    with pytest.raises(ValueError):
        g.add_tweights(5, 1, 1)
    gc = GCGraph(4, 4, sparse=True)
    with pytest.raises(ValueError):
        gc.set_nweights_bulk([0, 1], [1, 1], [1.0, 1.0], [1.0, 1.0])             # self loop
    with pytest.raises(ValueError):
        gc.set_nweights_bulk([0], [1], [0.0], [1.0])                             # weight <= 0
    with pytest.raises(ValueError):
        gc.set_nweights_bulk([0], [4], [1.0], [1.0])                             # id out of range
    gc.set_nweights_bulk([0, 2], [1, 3], [1.0, 2.0], [1.0, 2.0])
    with pytest.raises(TypeError):
        gc._add_markers(numpy.zeros(4, bool), numpy.zeros(4, bool))               # lattice-only entry point


def test_chain_graph_moves_to_sparse_backend_with_its_journal():
    from medpy_b200.graphcut.maxflow import GraphDouble
    g = GraphDouble(6, 10)
    g.sum_edge(0, 1, 1.0, 1.5)           # chain neighbours: stays a lattice
    g.add_tweights(0, 9.0, 0.0)
    assert not g.is_sparse
    g.sum_edge(0, 5, 2.0, 2.5)           # arbitrary pair: general graph
    assert g.is_sparse
    sp = g._sp
    sp._close_edges(); sp._close_tweights()
    edges = [op for op in sp._ops if op[0] == "e"][0]
    assert edges[1].tolist() == [0, 0] and edges[2].tolist() == [1, 5] and edges[3].tolist() == [1.0, 2.0]
    tw = [op for op in sp._ops if op[0] == "t"][0]
    assert tw[1].tolist() == [0] and tw[2].tolist() == [9.0]


def test_compat_filter_relabel_and_relabel_map():
    sys.path.insert(0, os.path.join(ROOT, "medpy_b200", "compat"))
    try:
        for m in [k for k in sys.modules if k == "medpy" or k.startswith("medpy.")]:
            del sys.modules[m]
        from medpy import filter as mfilter
        from medpy.core import ArgumentError
        lab = numpy.asarray([[7, 7, 3], [9, 3, 7]])
        assert mfilter.relabel(lab).tolist() == [[1, 1, 2], [3, 2, 1]]          # first appearance order (label.py:95-104)
        assert mfilter.relabel(lab, 5).tolist() == [[5, 5, 6], [7, 6, 5]]
        out = mfilter.relabel_map(numpy.asarray([[1, 2], [3, 1]]), [0, 1, 0, 1])
        assert out.tolist() == [[1, 0], [1, 1]]
        with pytest.raises(ArgumentError):
            mfilter.relabel_map(numpy.asarray([[1, 5]]), [0, 1])
    finally:
        sys.path.pop(0)
        for m in [k for k in sys.modules if k == "medpy" or k.startswith("medpy.")]:
            del sys.modules[m]


def test_graph_record_and_dimacs_writer_match_the_reference():
    """medpy.graphcut.Graph + graph_to_dimacs (graph.py:29-265, write.py:27-76) against what the unmodified reference
    writes and reports for the same graphs (tests/golden/reference_runs_v1.npz)."""
    import io
    from medpy_b200.graphcut import Graph, graph_to_dimacs
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    try:
        import make_golden_reference_runs as reference_runs
    finally:
        sys.path.pop(0)

    ours = reference_runs.fill_graph(Graph())
    buf = io.StringIO()
    graph_to_dimacs(ours, buf)
    assert ours.inconsistent() is False
    assert ours.get_nodes() == [1, 2, 3, 4, 5] and ours.get_edges() == [(1, 2), (2, 3), (4, 5)]
    assert ours.get_tweights()[1] == (Graph.MAX, 0) and ours.get_tweights()[5] == (0, Graph.MAX)
    msgs = reference_runs.fill_inconsistent(Graph()).inconsistent()
    assert msgs and len(msgs) == 5      # node 7 twice (t-weights, t-nodes), node 3 in an edge, two reversed duplicates
    z = reference_runs.load()
    assert buf.getvalue() == reference_runs.text(z, "dimacs")
    assert "\n".join(sorted(msgs)) == reference_runs.text(z, "inconsistent")
