"""Device-resident entry point: the same graph ``graph_from_voxels`` builds, from arrays that already live in
HBM (anything exposing ``__cuda_array_interface__``, e.g. torch CUDA tensors).  Used by bench.py's
inputs-resident measurement and by callers that produce the volume on the GPU; the order of operations is the
reference's: regional term, boundary term, foreground markers, background markers (generate.py:159-172).
"""
import math

from .maxflow import GraphDouble

_KINDS = {
    "difference_linear": 0, "difference_exponential": 1, "difference_division": 2, "difference_power": 3,
    "maximum_linear": 4, "maximum_exponential": 5, "maximum_division": 6, "maximum_power": 7,
}


def _as_u8(t):
    """bool tensors do not export __cuda_array_interface__ in every torch version: reinterpret as uint8."""
    try:
        import torch
        if isinstance(t, torch.Tensor) and t.dtype == torch.bool:
            return t.view(torch.uint8)
    except ImportError:  # pragma: no cover
        pass
    return t


def _keep_inputs_option():
    from .. import _lib
    return _lib._mgc.OPT_KEEP_INPUTS


def graph_from_device_arrays(fg_markers, bg_markers, image=None, boundary=None, sigma=None, spacing=False,
                             prob=None, alpha=None, graph=None, stream=None):
    """Build (or rebuild into ``graph``) the lattice graph from device arrays.

    boundary : one of the eight ``energy_voxel.boundary_*`` names without the prefix
    prob/alpha : ``regional_probability_map`` arguments (float32 map * Python float -> float32 products)
    graph : an earlier result to reuse (its device memory is kept, all weights are reset)
    stream : cudaStream_t as int (e.g. ``torch.cuda.current_stream().cuda_stream``) to run on
    """
    shape = tuple(int(s) for s in fg_markers.shape)
    n = 1
    for s in shape:
        n *= s
    if graph is None:
        graph = GraphDouble(n, 0, shape=shape)
    else:
        graph.reset()
    nat = graph._nat()
    if stream is not None:
        nat.set_stream(int(stream))
    graph._fresh = False
    # one native call: single-pass fused build on 1-D..3-D lattices (mgc_build_voxel_graph), the per-term kernels in
    # the reference's order otherwise.  A non-positive n-link weight is reported by maxflow() (ValueError).
    graph.defer_weight_check(True)
    # the inputs stay referenced by the graph until its next build or reset, so the build may run lazily on them
    # (cold blocks are built again from these arrays when the solve reaches them)
    nat.set_option(_keep_inputs_option(), 1)
    graph._inputs = (fg_markers, bg_markers, image, prob)
    compute_f32 = prob is not None and "float32" in str(prob.dtype)
    kind = _KINDS[boundary] if boundary is not None else -1
    sp = [float(s) for s in spacing] if spacing else None
    nat.build_voxel_graph(prob, 0.0 if alpha is None else float(alpha), compute_f32, kind, image,
                          0.0 if sigma is None else float(sigma), sp, math.nan, _as_u8(fg_markers), _as_u8(bg_markers))
    return graph
