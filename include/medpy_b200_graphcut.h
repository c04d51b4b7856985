/* medpy_b200_graphcut.h -- the drop-in boundary of the B200 voxel graph-cut path.
 *
 * C ABI (plain pointers and sizes, no torch / numpy / C++ types) of libmedpy_b200_gc.so.  It replaces,
 * for the voxel path only, what the reference reaches through its Boost.Python extension
 * `medpy.graphcut.maxflow` (lib/maxflow/src/wrapper.cpp:59-89,125-134; class GraphDouble =
 * Pythongraph<double,double,double>, pythongraph.h:15-22) plus the per-edge / per-node Python loops that
 * feed it (medpy/graphcut/energy_voxel.py:611-664, graph.py:310-380,532-552).  Instead of one FFI call per
 * edge, a whole energy term crosses the boundary in one call and is evaluated by a CUDA kernel on the
 * implicit 2*ndim-connected lattice; no edge list is ever materialised.
 *
 * Conventions
 *   - every function returns an int status: MGC_OK (0) or a negative MGC_E_* code; the message for the
 *     last failure on a handle is available from mgc_last_error() (never exit(), unlike graph.cpp:22);
 *   - node id == C-order flat index over the logical shape (generate.py:170-172, energy_voxel.py:650-677);
 *   - arrays are described by (pointer, dtype, byte strides over the logical shape); host pointers are only
 *     borrowed for the duration of the call (copied to the device inside); MGC_MEM_DEVICE pointers must be
 *     valid on the handle's device and are read on the handle's stream;
 *   - all device memory is owned by the library; a handle is not thread-safe, distinct handles are
 *     independent; the GIL can be released around every call;
 *   - there is NO CPU solver behind this ABI: with no usable CUDA device mgc_create fails with
 *     MGC_E_CUDA and nothing else works.
 */
#ifndef MEDPY_B200_GRAPHCUT_H
#define MEDPY_B200_GRAPHCUT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MGC_ABI_VERSION 3
#define MGC_MAX_NDIM 4

/* status codes */
#define MGC_OK 0
#define MGC_E_ARG (-1)     /* malformed argument (mirrors the reference's ValueError cases)     */
#define MGC_E_CUDA (-2)    /* CUDA runtime failure / no device                                  */
#define MGC_E_NOMEM (-3)   /* device allocation failed                                          */
#define MGC_E_STATE (-4)   /* call not valid in the handle's current state                      */
#define MGC_E_WEIGHT (-5)  /* an n-link weight <= 0 was produced (GCGraph.set_nweight, graph.py:436-437) */
#define MGC_E_NOCONV (-6)  /* solver hit its iteration cap without converging                   */
#define MGC_E_LABELS (-7)  /* label image is not numbered 1..K (energy_label.py:444-456 raises AttributeError) */

/* element types of input arrays */
#define MGC_F32 0
#define MGC_F64 1
#define MGC_U8 2
#define MGC_I16 3
#define MGC_I32 4

/* memory space of an input / output pointer */
#define MGC_MEM_HOST 0
#define MGC_MEM_DEVICE 1

/* boundary terms: the eight energy_voxel.boundary_* functions (energy_voxel.py:68-516) */
#define MGC_BOUNDARY_DIFFERENCE_LINEAR 0       /* energy_voxel.py:145-191 */
#define MGC_BOUNDARY_DIFFERENCE_EXPONENTIAL 1  /* :241-302 */
#define MGC_BOUNDARY_DIFFERENCE_DIVISION 2     /* :352-409 */
#define MGC_BOUNDARY_DIFFERENCE_POWER 3        /* :457-516 */
#define MGC_BOUNDARY_MAXIMUM_LINEAR 4          /* :68-116  */
#define MGC_BOUNDARY_MAXIMUM_EXPONENTIAL 5     /* :194-238 */
#define MGC_BOUNDARY_MAXIMUM_DIVISION 6        /* :305-349 (computes the *difference* variant, :347) */
#define MGC_BOUNDARY_MAXIMUM_POWER 7           /* :412-454 */

/* termtype (graph.h:57-61, wrapper.cpp:85-88) */
#define MGC_SOURCE 0
#define MGC_SINK 1

typedef struct mgc_graph mgc_graph; /* opaque; replaces GraphDouble + GCGraph storage */

typedef struct mgc_array {
    const void* data;                    /* first element (logical index 0,...,0) */
    int32_t dtype;                       /* MGC_F32 ... */
    int32_t mem;                         /* MGC_MEM_HOST | MGC_MEM_DEVICE */
    int64_t strides[MGC_MAX_NDIM];       /* BYTE strides over the logical shape (numpy .strides) */
} mgc_array;

typedef struct mgc_stats {
    int64_t n_voxels;
    int64_t push_sweeps;        /* push/relabel sweeps executed                     */
    int64_t global_relabels;    /* exact backward BFS passes                        */
    int64_t relabel_sweeps;     /* relaxation sweeps inside those                   */
    int64_t kernel_launches;    /* every kernel this handle launched                */
    int64_t active_last;        /* active voxels at the last check (0 = converged)  */
    double ms_terms;            /* device ms: boundary + regional + marker kernels  */
    double ms_solve;            /* device ms: init + push-relabel + global relabels */
    double ms_readout;          /* device ms: mask + energy kernels                 */
    double flow_const;          /* sum of the add_tweights minima (graph.h:423)     */
    double energy;              /* value maxflow() returned                         */
    int64_t device_bytes;       /* device memory held by the handle                 */
    double ms_push;             /* device ms inside push/relabel sweeps (CUDA events around each batch)  */
    double ms_relabel;          /* device ms inside global-relabel kernels (init + relaxation sweeps)    */
    double ms_boundary;         /* device ms of the last boundary (n-link) kernel alone                  */
    double ms_init;             /* device ms of the solver-state initialisation kernel (k_init_tile); 0 after a fused build */
} mgc_stats;

/* ---- lifetime ------------------------------------------------------------------------------------- */

/* Replaces GraphDouble(nodes, edges) + add_node(nodes) (graph.py:305-306; graph.cpp:11-31) for a lattice
 * of logical shape `shape[ndim]`, 1 <= ndim <= 4.  `device` = CUDA ordinal (or -1 for the current one). */
int mgc_create(int32_t ndim, const int64_t* shape, int32_t device, mgc_graph** out);
/* Slab variant for the z-slab multi-GPU path: this handle owns planes [z0, z1) of axis 0 of the global
 * lattice `shape` and keeps one ghost plane on each interior side. */
int mgc_create_slab(int32_t ndim, const int64_t* shape, int64_t z0, int64_t z1, int32_t device, mgc_graph** out);
void mgc_destroy(mgc_graph* g); /* ~Graph (graph.cpp:34-43) */
/* Graph::reset (graph.h:133): forget all weights, keep the allocation. */
int mgc_reset(mgc_graph* g);
const char* mgc_last_error(const mgc_graph* g); /* g may be NULL: last create() failure */
int mgc_abi_version(void);
/* Page-locked host buffers from a process-wide pool (the bindings hand the mask back in one: a device->host copy
 * into pinned memory runs at PCIe rate, into fresh pageable memory at a fraction of it).  mgc_host_free returns
 * the block to the pool. */
int mgc_host_alloc(size_t bytes, void** out);
void mgc_host_free(void* p);
/* Device and pinned-host blocks are cached process-wide (a 1024^3 handle holds 84 GB; its blocks stay cached for the next
 * graph after mgc_destroy).  mgc_trim_pools returns every cached block to the driver; live handles keep theirs. */
int mgc_trim_pools(void);
/* Options.  MGC_OPT_DEFER_WEIGHT_CHECK (default 0): mgc_add_boundary on a HOST image does not wait for its kernel to
 * report non-positive weights; the verdict (MGC_E_WEIGHT) is delivered by the next call on the handle instead (terms,
 * markers, maxflow, mgc_check).  graph_from_voxels switches it on because it always adds the markers right after the
 * boundary term, which lets the marker upload overlap the stencil kernel. */
#define MGC_OPT_DEFER_WEIGHT_CHECK 1
/* MGC_OPT_KEEP_INPUTS (default 0): the caller promises that the DEVICE arrays it passes to mgc_build_voxel_graph stay
 * valid and unchanged until the next build or mgc_reset on the handle.  This lets the build run lazily on them: blocks
 * that hold no source excess write only their residual mask and labels, and their capacities are computed again from
 * the inputs when the solve first reaches them.  Host and strided inputs are staged into the handle's own memory and
 * never need the promise; without it, caller-owned device inputs get an eager build. */
#define MGC_OPT_KEEP_INPUTS 2
int mgc_set_option(mgc_graph* g, int32_t option, int64_t value);
/* Deliver a deferred verdict now (MGC_OK / MGC_E_WEIGHT). */
int mgc_check(mgc_graph* g);
/* Use an externally owned cudaStream_t (e.g. torch's current stream) for all work of this handle. */
int mgc_set_stream(mgc_graph* g, void* cuda_stream);
int mgc_synchronize(mgc_graph* g);

/* ---- t-links -------------------------------------------------------------------------------------- */

/* regional_probability_map (energy_voxel.py:33-65) -> set_tweights_all (graph.py:532-552) ->
 * add_tweights(v, p*alpha, (1-p)*alpha) for every voxel (graph.h:415-425).  The products are formed in
 * `compute_dtype` (MGC_F32 or MGC_F64) -- the dtype numpy's promotion gives `probability_map * alpha`
 * (f32 map * Python float stays f32) -- and only then widened to double (graph.py:496-498). */
int mgc_add_regional_probability(mgc_graph* g, const mgc_array* prob, double alpha, int32_t compute_dtype);
/* Generic set_tweights_all: add_tweights(v, src[v], snk[v]); src/snk are arrays of doubles over the
 * logical shape. */
int mgc_add_tweights_dense(mgc_graph* g, const mgc_array* src, const mgc_array* snk);
/* set_source_nodes / set_sink_nodes (graph.py:310-380) as called by graph_from_voxels
 * (generate.py:169-172): add_tweights(v, 65535, 0) where fg != 0, THEN add_tweights(v, 0, 65535) where
 * bg != 0.  Either array may be NULL.  dtype MGC_U8 (numpy bool_). */
int mgc_add_markers(mgc_graph* g, const mgc_array* fg, const mgc_array* bg);

/* ---- n-links -------------------------------------------------------------------------------------- */

/* One of the eight boundary terms evaluated over the whole lattice (replaces the per-edge loop
 * energy_voxel.py:660-664 -> GCGraph.set_nweight -> Graph::sum_edge graph.h:456-480): for every axis d and
 * voxel pair (p, p+e_d):  w = g(|I_p - I_q|) or g(max(|I_p|,|I_q|)), w /= spacing[d] when spacing != NULL,
 * cap(p->q) += w, cap(q->p) += w, all in float64.
 *   sigma : ignored by the two linear terms.
 *   norm  : linear terms only -- the normaliser max|grad| / |max-min| the host computed in the image's own
 *           dtype (energy_voxel.py:99,174); pass NaN to have the device compute it (f32/f64 images).
 * Returns MGC_E_WEIGHT if any produced weight is <= 0 (the reference raises ValueError there). */
int mgc_add_boundary(mgc_graph* g, int32_t kind, const mgc_array* image, double sigma,
                     const double* spacing, double norm);
/* Dense n-links along one axis for user-written boundary terms: fwd/bwd are double arrays over the logical
 * shape; entry p holds cap(p -> p+e_axis) / cap(p+e_axis -> p); entries on the last plane of `axis` are
 * ignored.  Accumulates like sum_edge (graph.h:456-480); 0 leaves a pair untouched, negative values ->
 * MGC_E_WEIGHT (the `<= 0` ValueError of GCGraph.set_nweight is raised by the host layer, graph.py:436-437). */
int mgc_add_nweights_dense(mgc_graph* g, int32_t axis, const mgc_array* fwd, const mgc_array* bwd);

/* ---- the whole graph of graph_from_voxels in one call -------------------------------------------------- */

/* Everything graph_from_voxels puts into the graph (generate.py:159-172: regional term, boundary term, foreground
 * markers, background markers) handed over at once.  On a fresh handle (create / mgc_reset, nothing added yet) of a
 * 1-D..3-D lattice the terms are evaluated by ONE kernel pass (csrc/gc_build.cuh: n-link stencil + t-link replay +
 * solver-state initialisation; the image block of every CTA is staged by a TMA box copy) instead of four passes
 * over the lattice, and for contiguous host arrays the upload of z-chunk c+1 overlaps the build of chunk c.  The
 * result is the graph mgc_add_regional_probability + mgc_add_boundary + mgc_add_markers would leave (same
 * arithmetic per weight; the add_tweights constant is summed in a different, still fixed, order).  Anything else
 * (4-D lattice, no boundary term, terms already present) runs those three calls in that order.
 *   prob / fg / bg may be NULL; boundary_kind -1 = no boundary term; markers either as uint8 arrays (fg, bg) or
 *   bit-packed over the C-order flat voxel index v: bit (v & 31) of word (v >> 5) (fg_bits, bg_bits, bits_mem).
 * Weight verdict: MGC_E_WEIGHT from this call, or -- with MGC_OPT_DEFER_WEIGHT_CHECK -- from the next
 * mgc_check / mgc_maxflow.  Host pointers are borrowed for the duration of the call only. */
typedef struct mgc_voxel_terms {
    const mgc_array* prob;   /* regional_probability_map input (energy_voxel.py:33-65) or NULL */
    double alpha;
    int32_t compute_dtype;   /* MGC_F32 / MGC_F64, see mgc_add_regional_probability */
    int32_t boundary_kind;   /* MGC_BOUNDARY_* or -1 */
    const mgc_array* image;
    double sigma;
    const double* spacing;   /* NULL: no distance weighting */
    double norm;             /* linear terms: normaliser or NaN, see mgc_add_boundary */
    const mgc_array* fg;     /* uint8 marker volumes or NULL */
    const mgc_array* bg;
    const uint32_t* fg_bits; /* bit-packed marker volumes or NULL */
    const uint32_t* bg_bits;
    int32_t bits_mem;        /* MGC_MEM_HOST / MGC_MEM_DEVICE of fg_bits / bg_bits */
    /* Optional (host bit planes only): the number of leading 32-bit WORDS of BOTH planes that have been written so far,
     * advanced by a producer thread while this call runs (the binding packs the marker bytes on worker threads while the
     * image is already on its way to the device).  The call waits for it before it enqueues the upload of a chunk.
     * NULL: the planes are complete. */
    const volatile int64_t* bits_ready_words;
} mgc_voxel_terms;
int mgc_build_voxel_graph(mgc_graph* g, const mgc_voxel_terms* terms);
/* 1 if mgc_build_voxel_graph would take the single-pass path on a fresh state of this handle. */
int mgc_can_fuse(const mgc_graph* g);

/* ---- solve / read-out ----------------------------------------------------------------------------- */

/* Graph::maxflow() (maxflow.cpp:471-604; wrapper.cpp:68): runs the lattice push-relabel to a maximum
 * preflow and returns the min-cut energy INCLUDING the add_tweights constants, like the reference's `flow`.
 * Idempotent after convergence. */
int mgc_maxflow(mgc_graph* g, double* energy);
/* Bulk form of the what_segment loop (bin/medpy_graphcut_voxel.py:177-181): out[v] = 0 if the voxel is in
 * the SINK set else 1, C-order over the logical shape.  `mem` selects host or device destination. */
int mgc_get_mask(mgc_graph* g, uint8_t* out, int32_t mem);
/* Graph::what_segment(i) (graph.h:560-571): MGC_SINK or MGC_SOURCE (free nodes -> SOURCE). */
int mgc_what_segment(mgc_graph* g, int64_t node, int32_t* segment);
/* Graph::get_edge(i, j) (graph.h:482-497): current residual capacity of arc i->j, 0 if not lattice neighbours. */
int mgc_get_edge(mgc_graph* g, int64_t i, int64_t j, double* cap);
/* Graph::get_trcap(i) (graph.h:535-540): current residual terminal capacity (>0 source, <0 sink). */
int mgc_get_trcap(mgc_graph* g, int64_t node, double* trcap);
int mgc_get_node_num(const mgc_graph* g, int64_t* n);
int mgc_get_arc_num(const mgc_graph* g, int64_t* n);
int mgc_get_stats(const mgc_graph* g, mgc_stats* out);
/* Lazy build (MGC_OPT_KEEP_INPUTS, MEDPY_GC_LAZY): build blocks (8 x 8 x 32 voxels) of the last build if it ran lazily, else
 * 0, and how many of them held their capacity planes at the last maxflow (built hot or materialised on demand). */
int mgc_get_lazy_stats(const mgc_graph* g, int64_t* build_blocks, int64_t* materialised);

/* ---- pre-step of the boundary_maximum_* terms (SURVEY.md §8 row f1) ----------------------------------- */

/* bin/medpy_gradient.py:79-85: scipy.ndimage.generic_gradient_magnitude(image, prewitt, output=float32), mode 'reflect',
 * reproduced bit for bit.  `image`: f32/f64/u8/i16/i32 array over `shape[ndim]` (1 <= ndim <= 4, any positive strides);
 * `out`: C-contiguous float32 array of the same shape in host (MGC_MEM_HOST) or device memory. */
int mgc_gradient_magnitude_prewitt(int32_t ndim, const int64_t* shape, const mgc_array* image, float* out,
                                   int32_t out_mem, int32_t device);

/* ---- z-slab multi-GPU stepping (driven by the host over NCCL; see INTEGRATION.md) ------------------- */

/* Number of elements of one border-plane message: the product of the extents of axes 1..ndim-1. */
int mgc_slab_plane_elems(const mgc_graph* g, int64_t* n);
/* Initialise the solver state (source-excess clamp, sink capacities) once all terms are in. */
int mgc_slab_begin(mgc_graph* g);
/* `n` local push/relabel passes (tile solver: two-colour passes; per-voxel solver: sweeps). */
int mgc_slab_push(mgc_graph* g, int32_t n);
/* Pack the messages for the lower / upper neighbour into device buffers of plane_elems elements each:
 * heights (int32) of my border plane and the flow (double) pushed across the border since the last pack.
 * Pass NULL for a side without neighbour. */
int mgc_slab_pack(mgc_graph* g, int32_t* h_lo, double* f_lo, int32_t* h_hi, double* f_hi);
/* Apply the neighbours' messages: ghost-plane heights, and received flow added to excess and to the reverse
 * residual of my border plane.  `changed_dev` (DEVICE pointer or NULL) is set to 1 by the kernel if any ghost label
 * differs from before; the caller zeroes it and typically all-reduces it over the ranks.  No host synchronisation. */
int mgc_slab_unpack(mgc_graph* g, const int32_t* h_lo, const double* f_lo, const int32_t* h_hi, const double* f_hi,
                    int32_t* changed_dev);
/* Global relabel, distributed: (re)start a backward BFS from the sink ... */
int mgc_slab_relabel_begin(mgc_graph* g);
/* ... relax locally until nothing changes (given the current ghost labels).  changed_out may be NULL (then the call
 * does not synchronise with the host); otherwise *changed_out = 1 if any tile was visited in this call. */
int mgc_slab_relabel_relax(mgc_graph* g, int32_t* changed_out);
/* Voxels with excess > 0 and a finite label (owned planes only). */
int mgc_slab_count_active(mgc_graph* g, int64_t* active_out);
/* Same, written to a DEVICE counter (uint64) without synchronising with the host. */
int mgc_slab_count_active_dev(mgc_graph* g, unsigned long long* count_dev);
/* Finish: build the mask of the owned planes and this slab's share of the energy
 * (flow absorbed by the owned sink links + owned add_tweights constants). */
int mgc_slab_finish(mgc_graph* g, double* energy_part);

/* ---- z-slab solve inside the library (NCCL over NVLink on the handle's stream) ------------------------------ */

/* The stepping calls above let a host drive the slabs; these three run the WHOLE distributed solve natively: border
 * messages go out with ncclSend / ncclRecv (grouped, on the handle's stream), the stop test is one ncclAllReduce and
 * one host synchronisation per relabel round, the energy is all-reduced (float64).  libnccl.so.2 is bound at run time
 * (the copy already loaded in the process, e.g. torch's); asynchronous NCCL errors are polled at every host decision
 * and returned as MGC_E_CUDA instead of hanging.
 *   mgc_slab_comm_unique_id : 128-byte ncclUniqueId made by ONE rank; the host distributes it (any transport);
 *   mgc_slab_comm_init      : collective over the `world` slab ranks (rank r owns the r-th slab);
 *   mgc_slab_solve          : collective; *energy_total = the global min-cut energy on every rank.  mgc_get_mask then
 *                             returns the rank's owned planes. */
int mgc_slab_comm_unique_id(void* out128);
int mgc_slab_comm_init(mgc_graph* g, int32_t rank, int32_t world, const void* unique_id128);
int mgc_slab_solve(mgc_graph* g, double* energy_total);
int mgc_slab_solve_stats(const mgc_graph* g, int64_t* exchanges, int64_t* relabel_rounds, int64_t* push_passes,
                         int64_t* global_relabels);
/* Device milliseconds of the last mgc_slab_solve per phase (CUDA events on the handle's stream): out6[0] local BFS,
 * [1] border exchanges (pack + ncclSend/ncclRecv + unpack), [2] stop test (count + all-reduce), [3] push passes,
 * [4] read-out + energy all-reduce, and out6[5] = HOST milliseconds spent blocked in the per-round synchronisations. */
int mgc_slab_solve_phase_ms(const mgc_graph* g, double* out6);

/* ---- general sparse graphs (SURVEY.md §8 rows f3/f4) ----------------------------------------------------- */

/* The graphs of the reference that are NOT voxel lattices: the region adjacency graph graph_from_labels builds
 * (generate.py:177-338) and graphs assembled call by call through GCGraph / GraphDouble (graph.py:382-498,
 * wrapper.cpp:63-83; e.g. tests/graphcut_/graph.py:47).  The handle replaces GraphDouble(nodes, edges) + add_node:
 * edges and terminal weights arrive in bulk (arrays of what would have been one call each, applied in array order with
 * the reference's accumulation semantics), the max-flow runs on the device as a CSR push-relabel (gc_sparse.cuh). */
typedef struct mgc_sparse mgc_sparse;
int mgc_sparse_create(int64_t n_nodes, int32_t device, mgc_sparse** out);
void mgc_sparse_destroy(mgc_sparse* g);
int mgc_sparse_reset(mgc_sparse* g);                           /* Graph::reset (graph.h:133) */
const char* mgc_sparse_last_error(const mgc_sparse* g);        /* g may be NULL: last create() failure */
/* count x Graph::sum_edge(i[k], j[k], cap[k], rev_cap[k]) (graph.h:456-480) in order: the first call for a node pair
 * creates its arc pair, later calls -- in either orientation -- accumulate with +=.  Host arrays.  MGC_E_ARG for ids
 * outside [0, n) or i == j (the ValueErrors of GCGraph.set_nweight, graph.py:418-435). */
int mgc_sparse_sum_edges(mgc_sparse* g, int64_t count, const int32_t* i, const int32_t* j, const double* cap,
                         const double* rev_cap);
/* count x Graph::add_tweights(nodes[k], src[k], snk[k]) (graph.h:415-425) in order; nodes == NULL means 0..count-1. */
int mgc_sparse_add_tweights(mgc_sparse* g, int64_t count, const int32_t* nodes, const double* src, const double* snk);
/* Graph::maxflow(): min-cut energy including the add_tweights constants.  Idempotent until the graph changes. */
int mgc_sparse_maxflow(mgc_sparse* g, double* energy);
/* out[v] = 0 if what_segment(v) == SINK else 1, for all n nodes (host buffer). */
int mgc_sparse_get_mask(mgc_sparse* g, uint8_t* out);
int mgc_sparse_what_segment(mgc_sparse* g, int64_t node, int32_t* segment);
/* Capacity of arc i->j / net terminal capacity as assembled so far (the values the reference's getters return before
 * maxflow(); 0 for unconnected pairs). */
int mgc_sparse_get_edge(const mgc_sparse* g, int64_t i, int64_t j, double* cap);
int mgc_sparse_get_trcap(const mgc_sparse* g, int64_t node, double* trcap);
int mgc_sparse_get_node_num(const mgc_sparse* g, int64_t* n);
int mgc_sparse_get_arc_num(const mgc_sparse* g, int64_t* n);    /* 2 per connected node pair */
int mgc_sparse_get_stats(const mgc_sparse* g, mgc_stats* out);

/* ---- label images: the region adjacency graph built on the device (row f3) ------------------------------------ */

/* A label image resident in device memory.  Replaces what every energy_label term recomputes from the numpy array
 * (energy_label.py:78-86,181-189): mgc_labels_create stages `labels` (MGC_I32, any positive strides, logical shape
 * `shape[ndim]`, 1 <= ndim <= 4) once and runs __check_label_image (:444-456): MGC_E_LABELS unless the ids are
 * exactly 1..K.  Region r of the image is node r-1 of the graph (generate.py:334-337). */
typedef struct mgc_labels mgc_labels;
int mgc_labels_create(int32_t ndim, const int64_t* shape, const mgc_array* labels, int32_t device, mgc_labels** out);
void mgc_labels_destroy(mgc_labels* l);
const char* mgc_labels_last_error(const mgc_labels* l);       /* l may be NULL: last create() failure */
int mgc_labels_region_count(const mgc_labels* l, int64_t* k);
/* Boundary terms over all border voxel pairs (2*ndim-connectivity), reduced per region pair in the reference's own
 * accumulation order (axis by axis, C order inside an axis), so the sums equal what the chain of set_nweight ->
 * sum_edge calls leaves in the reference's arcs:
 *   MGC_LABELS_ADJACENCY  : __compute_edges_nd (energy_label.py:411-441): the pairs only (`values` ignored);
 *   MGC_LABELS_STAWIASKI  : boundary_stawiaski (:123-214): w = (1/(1+max(|g_p|,|g_q|)))^2, both directions;
 *   MGC_LABELS_STAWIASKI_DIRECTED : boundary_stawiaski_directed (:217-342) with `directedness` (incl. the double
 *                                   count of every axis' first pair that numpy.vectorize causes there).
 * `values` = gradient image (f32/f64/u8/i16/i32) over the same shape.  The result stays in the handle:
 * *n_edges region pairs, fetched with mgc_labels_fetch_edges into host arrays of that length, sorted by (i, j), i < j:
 * w_ij = capacity i->j, w_ji = capacity j->i. */
#define MGC_LABELS_ADJACENCY 0
#define MGC_LABELS_STAWIASKI 1
#define MGC_LABELS_STAWIASKI_DIRECTED 2
int mgc_labels_boundary(mgc_labels* l, int32_t kind, const mgc_array* values, double directedness, int64_t* n_edges);
int mgc_labels_fetch_edges(const mgc_labels* l, int32_t* i, int32_t* j, double* w_ij, double* w_ji);
/* Per-region sums of `values` and voxel counts (host arrays of K entries).
 *   MGC_SUM_BINCOUNT : numpy.bincount(labels, weights) as used by scipy.ndimage.mean (energy_label.py:92): float64,
 *                      front to back in C order;
 *   MGC_SUM_PAIRWISE : numpy.sum over the region's voxels in the array's own float type (regional_atlas,
 *                      energy_label.py:384-386): numpy's pairwise summation, reproduced exactly (integer arrays are
 *                      summed exactly either way). */
#define MGC_SUM_BINCOUNT 0
#define MGC_SUM_PAIRWISE 1
int mgc_labels_region_sums(mgc_labels* l, const mgc_array* values, int32_t mode, double* sums, int64_t* counts);
/* flags[r] = 1 if any voxel of region r+1 is marked (numpy.unique(label_image[markers] - 1), generate.py:334-337);
 * `markers` MGC_U8 over the same shape, flags = host array of K bytes. */
int mgc_labels_region_flags(mgc_labels* l, const mgc_array* markers, uint8_t* flags);
/* out[p] = per_region[label[p] - 1]: maps the cut back onto the voxels (bin/medpy_graphcut_label.py:139-148).
 * per_region = host array of K bytes; out = C-contiguous uint8 over the shape in host or device memory. */
int mgc_labels_apply(mgc_labels* l, const uint8_t* per_region, uint8_t* out, int32_t out_mem);

#ifdef __cplusplus
}
#endif
#endif /* MEDPY_B200_GRAPHCUT_H */
