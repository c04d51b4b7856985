"""``medpy_b200.graphcut.maxflow`` -- the object ``graph_from_voxels`` returns.

Mirror of the reference's compiled module ``medpy.graphcut.maxflow`` (Boost.Python,
lib/maxflow/src/wrapper.cpp:59-89): class ``GraphDouble`` with ``add_tweights / sum_edge / add_edge /
maxflow / what_segment / get_edge / get_trcap / get_node_num / get_arc_num / reset`` and the nested enum
``termtype`` (wrapper.cpp:85-88).  Storage is NOT the reference's node/arc lists: the graph is a dense
2*ndim-connected lattice living in B200 HBM behind the C ABI (include/medpy_b200_graphcut.h); whole energy
terms are handed to CUDA kernels, element-wise calls are staged in dense host arrays and uploaded in bulk.

There is no CPU solver here: the first operation that needs the device creates the native graph and
raises ``RuntimeError`` when no CUDA device / built extension is available.
"""
import enum

import numpy

__all__ = ["GraphDouble", "GraphFloat", "GraphInt"]


class _termtype(enum.IntEnum):
    """graph.h:57-61: terminals."""
    SOURCE = 0
    SINK = 1


def _strides_of(shape):
    st = []
    acc = 1
    for s in reversed(shape):
        st.append(acc)
        acc *= int(s)
    return tuple(reversed(st))


class GraphDouble:
    """Lattice max-flow graph with the reference's ``GraphDouble`` method names.

    ``GraphDouble(node_num_max, edge_num_max, shape=None)``: ``shape`` is the logical lattice shape (C-order
    node ids, generate.py:170-172); without it the graph is a 1-D chain of ``node_num_max`` nodes.
    """

    termtype = _termtype

    def __init__(self, node_num_max, edge_num_max=0, shape=None, device=-1, sparse=None):
        # Without a lattice shape the graph starts as a 1-D chain (what element-wise users of the voxel path build) and
        # keeps a journal of its calls; the first edge that does not join chain neighbours -- or sparse=True -- moves
        # it, journal and all, onto the general sparse backend (sparse.py, SURVEY.md §8 row f4).
        self._sp = None
        self._journal = [] if shape is None else None
        if shape is None:
            shape = (int(node_num_max),)
        shape = tuple(int(s) for s in shape)
        if len(shape) < 1 or len(shape) > 4:
            raise ValueError("the lattice path supports 1 to 4 dimensions, got shape {}".format(shape))
        n = 1
        for s in shape:
            n *= s
        if n != int(node_num_max):
            raise ValueError("shape {} does not hold {} nodes".format(shape, node_num_max))
        self._shape = shape
        self._n = n
        self._strides = _strides_of(shape)
        self._edges = int(edge_num_max)
        self._device = device
        self._native = None
        # element-wise staging (dense host arrays, flushed in bulk)
        self._st_src = None
        self._st_snk = None
        self._st_touched = None
        self._st_nw = {}  # axis -> [fwd, bwd] dense arrays
        self._mask = None
        self._offlattice = None
        self._pending = []
        self._defer_weight_check = False
        # whole-lattice terms collected while graph_from_voxels runs (regional, boundary, markers): handed to the device
        # in ONE native call (mgc_build_voxel_graph: single-pass fused build) when the markers arrive or anything else
        # needs the graph.  Only while nothing has reached the device yet (_fresh).
        self._lazy = None
        self._inputs = None
        self._fresh = True
        if sparse:
            if self._journal is None:
                raise ValueError("a lattice shape and sparse=True exclude each other")
            self._to_sparse()

    def _to_sparse(self):
        from .sparse import SparseGraphDouble
        sp = SparseGraphDouble(self._n, self._edges, device=self._device)
        for op in self._journal or []:
            if op[0] == "e":
                sp.sum_edge(op[1], op[2], op[3], op[4])
            elif op[0] == "t":
                sp.add_tweights(op[1], op[2], op[3])
            else:
                sp.add_tweights_bulk(op[1], op[2], op[3])
        self._journal = None
        self._sp = sp
        # drop the chain-lattice staging and device state
        self._st_src = self._st_snk = self._st_touched = None
        self._st_nw = {}
        self._pending = []
        self._native = None
        self._mask = None

    @property
    def is_sparse(self):
        return self._sp is not None

    # ------------------------------------------------------------------ native handle
    @property
    def shape(self):
        return self._shape

    def _nat(self):
        if self._sp is not None:
            raise TypeError("this graph is a general sparse graph: lattice terms (energy_voxel.*) need a graph created "
                            "with a lattice shape")
        if self._native is None:
            from .. import _lib  # raises ImportError loudly when the extension is not built
            self._native = _lib.Graph(list(self._shape), self._device)
            if self._defer_weight_check:
                self._native.set_option(_lib._mgc.OPT_DEFER_WEIGHT_CHECK, 1)
        return self._native

    def defer_weight_check(self, on=True):
        """Let a boundary term return before its kernel has reported non-positive weights; the ValueError is then
        raised by the next call on the graph (graph_from_voxels adds the markers right after the boundary term, so the
        marker upload overlaps the stencil kernel).  ``check_deferred()`` forces the verdict."""
        if not on:
            self._commit()
        self._defer_weight_check = bool(on)
        if self._native is not None:
            from .. import _lib
            self._native.set_option(_lib._mgc.OPT_DEFER_WEIGHT_CHECK, 1 if on else 0)

    def check_deferred(self):
        self._commit()
        if self._native is not None:
            self._native.check_deferred()

    # ------------------------------------------------------------------ collected whole-lattice terms
    def _collect(self, key, value):
        """Record a whole-lattice term instead of launching it; False if it has to run right away (the graph already
        holds terms, element-wise calls are staged, the same kind of term was collected before, or collection is off)."""
        if not self._defer_weight_check or not self._fresh or self._sp is not None:
            return False
        if self._st_src is not None or self._st_nw or self._pending:
            return False
        if self._lazy is not None and key in self._lazy:
            return False
        if self._lazy is None:
            self._lazy = {}
        self._lazy[key] = value
        return True

    def _commit(self):
        """Hand the collected terms to the device: regional term, boundary term, fg / bg markers in the reference's
        order (generate.py:159-172), as one fused pass where the native side can (mgc_build_voxel_graph)."""
        lazy, self._lazy = self._lazy, None
        if not lazy:
            return
        self._fresh = False
        prob, alpha, f32 = lazy.get("reg", (None, 0.0, False))
        kind, image, sigma, spacing, norm = lazy.get("bnd", (-1, None, 0.0, None, float("nan")))
        fg, bg = lazy.get("mark", (None, None))
        self._nat().build_voxel_graph(prob, float(alpha), bool(f32), int(kind), image, float(sigma), spacing, float(norm), fg, bg)

    def _dirty(self):
        self._mask = None

    # ------------------------------------------------------------------ staging of element-wise calls
    # Element-wise calls (add_tweights / sum_edge, i.e. GCGraph.set_tweight / set_nweight / set_source_nodes)
    # never touch the device: they fill dense host batches that are uploaded in call order by _flush().
    def _close_tweight_batch(self):
        if self._st_src is not None:
            self._pending.append(("tw", self._st_src, self._st_snk))
            self._st_src = self._st_snk = self._st_touched = None

    def _open_tweight_batch(self):
        if self._st_src is None:
            self._st_src = numpy.zeros(self._n, dtype=numpy.float64)
            self._st_snk = numpy.zeros(self._n, dtype=numpy.float64)
            self._st_touched = numpy.zeros(self._n, dtype=numpy.bool_)

    def stage_tweights_many(self, ids, cap_source, cap_sink):
        """add_tweights(v, cap_source, cap_sink) for every v in ids, in order (ids already range-checked)."""
        ids = numpy.asarray(ids, dtype=numpy.int64)
        if self._sp is not None:
            return self._sp.stage_tweights_many(ids, cap_source, cap_sink)
        if self._journal is not None:
            self._journal.append(("T", ids.copy(), numpy.full(ids.size, float(cap_source)), numpy.full(ids.size, float(cap_sink))))
        self._dirty()
        self._open_tweight_batch()
        if numpy.unique(ids).size == ids.size:
            if self._st_touched[ids].any():
                self._close_tweight_batch()
                self._open_tweight_batch()
            self._st_src[ids] = float(cap_source)
            self._st_snk[ids] = float(cap_sink)
            self._st_touched[ids] = True
        else:
            for v in ids:
                self._add_tweights_staged(int(v), cap_source, cap_sink)

    def _flush(self):
        self._commit()
        self._close_tweight_batch()
        if self._st_nw:
            for axis in sorted(self._st_nw):
                fwd, bwd = self._st_nw[axis]
                self._pending.append(("nw", axis, fwd, bwd))
            self._st_nw = {}
        pending, self._pending = self._pending, []
        if pending:
            self._fresh = False
        for op in pending:
            if op[0] == "tw":
                self._nat().add_tweights_dense(op[1].reshape(self._shape), op[2].reshape(self._shape))
            else:
                # pairs never set stay 0, which sum_edge semantics allow (graph.h:456-463 asserts cap >= 0)
                self._nat().add_nweights_dense(op[1], op[2].reshape(self._shape), op[3].reshape(self._shape))

    # ------------------------------------------------------------------ bulk term entry points (used by energy_voxel)
    def _lattice_term(self):
        """A whole-lattice term is about to be applied: a shape-less graph that takes one stays the 1-D chain it was
        created as (its journal cannot describe device-side terms, so it can no longer move to the sparse backend)."""
        if self._sp is None:
            self._journal = None

    def add_regional_probability(self, prob, alpha, compute_f32):
        self._lattice_term()
        self._dirty()
        if self._collect("reg", (self._positive_strides(prob), float(alpha), bool(compute_f32))):
            return
        self._flush()
        self._fresh = False
        self._nat().add_regional_probability(self._positive_strides(prob), float(alpha), bool(compute_f32))

    def add_tweights_dense(self, src, snk):
        """add_tweights(v, src[v], snk[v]) for every node (GCGraph.set_tweights_all, graph.py:532-552)."""
        if self._sp is not None:
            return self._sp.add_tweights_bulk(None, numpy.ravel(src), numpy.ravel(snk))
        src = numpy.ascontiguousarray(src, dtype=numpy.float64).reshape(self._shape)
        snk = numpy.ascontiguousarray(snk, dtype=numpy.float64).reshape(self._shape)
        if self._journal is not None:
            # shape-less graph: staged like the element-wise calls (no device needed yet) and journaled node-wise, so a
            # later move to the sparse backend can replay it
            self._journal.append(("T", numpy.arange(self._n), src.ravel().copy(), snk.ravel().copy()))
            self._close_tweight_batch()
            self._pending.append(("tw", src.ravel().copy(), snk.ravel().copy()))
            self._dirty()
            return
        self._flush()
        self._dirty()
        self._fresh = False
        self._nat().add_tweights_dense(src, snk)

    @staticmethod
    def _positive_strides(a):
        """Host arrays with zero / negative strides (broadcast views, reversed slices) are copied once; everything
        else -- including Fortran-ordered arrays as medpy.io.load returns them -- is handed over as is."""
        if a is None or not isinstance(a, numpy.ndarray):
            return a
        if any(st <= 0 and n > 1 for st, n in zip(a.strides, a.shape)):
            return numpy.ascontiguousarray(a)
        return a

    def add_markers(self, fg, bg):
        self._lattice_term()
        self._dirty()
        if self._lazy and "mark" not in self._lazy and self._collect("mark", (self._positive_strides(fg), self._positive_strides(bg))):
            return self._commit()        # the markers are graph_from_voxels' last step: build now
        self._flush()
        self._fresh = False
        self._nat().add_markers(self._positive_strides(fg), self._positive_strides(bg))

    def add_boundary(self, kind, image, sigma, spacing, norm):
        self._lattice_term()
        self._dirty()
        if self._collect("bnd", (int(kind), self._positive_strides(image), float(sigma), spacing, float(norm))):
            return
        self._flush()
        self._fresh = False
        self._nat().add_boundary(int(kind), self._positive_strides(image), float(sigma), spacing, float(norm))

    def add_nweights_dense(self, axis, fwd, bwd):
        self._lattice_term()
        self._flush()
        self._dirty()
        self._fresh = False
        self._nat().add_nweights_dense(int(axis), fwd, bwd)

    # ------------------------------------------------------------------ reference GraphDouble API
    def add_node(self, num=1):
        """graph.h:388-413.  Nodes are implied by the lattice; returns the id the reference would."""
        return 0

    def add_tweights(self, i, cap_source, cap_sink):
        """graph.h:415-425, staged: calls on distinct nodes are batched into one dense device pass."""
        i = int(i)
        if i < 0 or i >= self._n:
            raise ValueError("Invalid node id of {}. Valid values are 0 to {}.".format(i, self._n - 1))
        if self._sp is not None:
            return self._sp.add_tweights(i, cap_source, cap_sink)
        if self._journal is not None:
            self._journal.append(("t", i, float(cap_source), float(cap_sink)))
        self._add_tweights_staged(i, cap_source, cap_sink)

    def _add_tweights_staged(self, i, cap_source, cap_sink):
        self._open_tweight_batch()
        if self._st_touched[i]:
            self._close_tweight_batch()  # add_tweights is order dependent per node: start a new batch
            self._open_tweight_batch()
        self._st_src[i] = float(cap_source)
        self._st_snk[i] = float(cap_sink)
        self._st_touched[i] = True
        self._dirty()

    def _axis_of(self, i, j):
        d = j - i
        for axis, st in enumerate(self._strides):
            if abs(d) == st and self._shape[axis] > 1:
                lo = min(i, j)
                if (lo // st) % self._shape[axis] < self._shape[axis] - 1:
                    return axis
        return None

    def sum_edge(self, i, j, cap, rev_cap):
        """graph.h:456-480 for lattice neighbours (accumulating)."""
        i, j = int(i), int(j)
        if i < 0 or j < 0 or i >= self._n or j >= self._n or i == j:
            raise ValueError("invalid node ids ({}, {})".format(i, j))
        if self._sp is not None:
            return self._sp.sum_edge(i, j, cap, rev_cap)
        axis = self._axis_of(i, j)
        if axis is None:
            if self._journal is not None:
                # not a chain neighbour: this is a general graph (tests/graphcut_/graph.py:47) -> sparse backend
                self._to_sparse()
                return self._sp.sum_edge(i, j, cap, rev_cap)
            # a lattice graph (graph_from_voxels) accepts the call like the reference would, but an edge between
            # non-neighbours can never be solved on the lattice; maxflow() refuses.
            self._offlattice = (i, j)
            return
        if self._journal is not None:
            self._journal.append(("e", i, j, float(cap), float(rev_cap)))
        if axis not in self._st_nw:
            self._st_nw[axis] = [numpy.zeros(self._n, dtype=numpy.float64), numpy.zeros(self._n, dtype=numpy.float64)]
        fwd, bwd = self._st_nw[axis]
        if i < j:
            fwd[i] += float(cap)
            bwd[i] += float(rev_cap)
        else:
            fwd[j] += float(rev_cap)
            bwd[j] += float(cap)
        self._dirty()

    add_edge = sum_edge  # graph.h:427-454: parallel arcs act as summed capacities

    def sum_edges_bulk(self, i, j, cap, rev_cap):
        """One sum_edge call per array entry, in order (general graphs: moves the graph to the sparse backend)."""
        if self._sp is None:
            if self._journal is None:
                raise ValueError("bulk edges between arbitrary nodes need a graph without lattice shape")
            self._to_sparse()
        self._sp.sum_edges_bulk(i, j, cap, rev_cap)

    def add_tweights_bulk(self, nodes, src, snk):
        """One add_tweights call per array entry, in order."""
        if self._sp is not None:
            return self._sp.add_tweights_bulk(nodes, src, snk)
        nodes = numpy.arange(len(src)) if nodes is None else numpy.asarray(nodes)
        for v, a, b in zip(nodes.tolist(), numpy.asarray(src, dtype=float).tolist(), numpy.asarray(snk, dtype=float).tolist()):
            self.add_tweights(v, a, b)

    def maxflow(self):
        """Graph::maxflow (maxflow.cpp:471-604): min-cut energy including the add_tweights constants."""
        if self._sp is not None:
            return self._sp.maxflow()
        if self._offlattice is not None:
            raise NotImplementedError(
                "edge {} does not join lattice neighbours of shape {}: build general graphs with "
                "GraphDouble(nodes, edges) (no shape), which uses the sparse backend".format(self._offlattice, self._shape))
        self._flush()
        return self._nat().maxflow()

    def get_mask(self):
        """Bulk read-out: uint8 array of the lattice shape, 0 where what_segment == SINK else 1
        (what bin/medpy_graphcut_voxel.py:177-181 builds voxel by voxel)."""
        if self._sp is not None:
            return self._sp.get_mask()
        if self._mask is None:
            self.maxflow()
            self._mask = self._nat().get_mask()
        return self._mask

    def what_segment(self, i, default_segm=None):
        """graph.h:560-571."""
        if self._sp is not None:
            return self._sp.what_segment(i)
        m = self.get_mask()
        i = int(i)
        if i < 0 or i >= self._n:
            raise ValueError("Invalid node id of {}. Valid values are 0 to {}.".format(i, self._n - 1))
        return _termtype.SOURCE if m.flat[i] else _termtype.SINK

    def reset(self):
        if self._sp is not None:
            return self._sp.reset()
        if self._journal is not None:
            self._journal = []
        self._st_src = self._st_snk = self._st_touched = None
        self._st_nw = {}
        self._mask = None
        self._offlattice = None
        self._pending = []
        self._lazy = None
        self._fresh = True
        self._inputs = None         # device arrays a lazy build may still read (graph_from_device_arrays)
        if self._native is not None:
            self._native.reset()

    def get_edge(self, i, j):
        if self._sp is not None:
            return self._sp.get_edge(i, j)
        self._flush()
        return self._nat().get_edge(int(i), int(j))

    def get_trcap(self, i):
        if self._sp is not None:
            return self._sp.get_trcap(i)
        self._flush()
        return self._nat().get_trcap(int(i))

    def get_node_num(self):
        return self._n

    def get_arc_num(self):
        if self._sp is not None:
            return self._sp.get_arc_num()
        self._flush()
        return self._nat().get_arc_num()

    def stats(self):
        if self._sp is not None:
            return self._sp.stats()
        return self._nat().stats()


# The reference module exports three instantiations (wrapper.cpp:8-10); only GraphDouble is used by the
# Python layer (graph.py:26,305).  The other names resolve to the same lattice graph.
GraphFloat = GraphDouble
GraphInt = GraphDouble
