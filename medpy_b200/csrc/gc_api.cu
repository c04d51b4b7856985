// gc_api.cu -- C-ABI of libmedpy_b200_gc.so (include/medpy_b200_graphcut.h) and the host driver of the
// lattice push-relabel solver.  sm_100a only; there is no CPU path: without a CUDA device every entry
// point fails with MGC_E_CUDA.
#include "../../include/medpy_b200_graphcut.h"
#include "gc_common.cuh"
#include "gc_terms.cuh"
#include "gc_solver.cuh"
#include "gc_tiles.cuh"
#include "gc_persist.cuh"
#include "gc_tma.cuh"
#include "gc_tiles4.cuh"
#include "gc_sweep.cuh"
#include "gc_build.cuh"
#include "gc_gradient.cuh"

#include <dlfcn.h>
#include <nccl.h>
#include <nvtx3/nvToolsExt.h>

#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

// ---------------------------------------------------------------------------------------------------
// device memory pool: graph_from_voxels creates a new graph per call (generate.py:120); handing freed
// blocks to the next handle keeps cudaMalloc (milliseconds per GB) out of the steady state.
// ---------------------------------------------------------------------------------------------------
namespace {
std::mutex g_pool_mu;
std::map<std::pair<int, size_t>, std::vector<void*>> g_pool;
thread_local std::string g_create_error;

size_t round_up(size_t b) { const size_t g = size_t(1) << 21; return (b + g - 1) / g * g; }

cudaError_t pool_alloc(int dev, size_t bytes, void** out)
{
    bytes = round_up(bytes);
    {
        std::lock_guard<std::mutex> lk(g_pool_mu);
        auto it = g_pool.find({dev, bytes});
        if (it != g_pool.end() && !it->second.empty()) {
            *out = it->second.back();
            it->second.pop_back();
            return cudaSuccess;
        }
    }
    cudaError_t e = cudaMalloc(out, bytes);
    if (e != cudaSuccess) {
        // release cached blocks and retry once
        std::lock_guard<std::mutex> lk(g_pool_mu);
        for (auto& kv : g_pool) if (kv.first.first == dev) { for (void* p : kv.second) cudaFree(p); kv.second.clear(); }
        cudaGetLastError();
        e = cudaMalloc(out, bytes);
    }
    return e;
}

void pool_free(int dev, size_t bytes, void* p)
{
    if (!p) return;
    std::lock_guard<std::mutex> lk(g_pool_mu);
    g_pool[{dev, round_up(bytes)}].push_back(p);
}

// pinned host blocks (mask read-back buffers handed to the binding): same pooling idea as device memory
std::map<size_t, std::vector<void*>> g_host_pool;
std::map<void*, size_t> g_host_live;

int cached_sm_count(int dev)
{
    static std::mutex mu;
    static std::map<int, int> cache;
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(dev);
    if (it != cache.end()) return it->second;
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cache[dev] = n;
    return n;
}

struct Buf {
    void* p = nullptr;
    size_t bytes = 0;
};

size_t dtype_size(int dt)
{
    switch (dt) {
        case MGC_F32: return 4;
        case MGC_F64: return 8;
        case MGC_U8: return 1;
        case MGC_I16: return 2;
        case MGC_I32: return 4;
        default: return 0;
    }
}
}  // namespace

struct mgc_graph {
    int device = 0;
    int user_ndim = 0;
    int nd = 3;             // canonical axes
    int shift = 0;          // canonical axis = user axis + shift
    int64_t user_shape[4] = {1, 1, 1, 1};
    Lattice L{};
    bool slab = false;
    bool ghost_lo = false, ghost_hi = false;
    int64_t global_dim0 = 0, z0 = 0, z1 = 0;

    State<double> S{};
    std::vector<Buf> owned_bufs;       // everything allocated from the pool
    Buf scratch[5];                    // staged (contiguous) copies of input arrays: 0 prob/src, 1 fg/snk, 2 image, 4 bg
    Buf raw;                           // raw span of a strided host array
    uint8_t* mask_dev = nullptr;
    double* partials = nullptr;        // per-block partial sums
    unsigned n_partials = 0;
    void* minmax_buf = nullptr;        // 3 x 1024 partial min/max/absmax
    double* d_scalars = nullptr;       // [0] flow_const, [1] absorbed, [2..3] minmax out
    int* d_flags = nullptr;            // [0] bad weight, [1] changed, [2] work
    unsigned long long* d_count = nullptr;
    int64_t device_bytes = 0;

    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaEvent_t ev[6] = {};
    // host -> device staging runs on its own stream so that the copy of the next term overlaps the kernel of the
    // previous one; the host only waits for the COPY (its pointer is borrowed for the call), never for the kernel
    cudaStream_t up_stream = nullptr;
    cudaEvent_t ev_up = nullptr;
    cudaEvent_t ev_slot[5] = {};       // main-stream point after which a staging slot may be overwritten (3 = raw span)
    bool slot_used[5] = {false, false, false, false, false};
    cudaEvent_t ev_chunk[2] = {};      // chunked fused build: upload stream -> main stream hand-over (alternating)
    cudaEvent_t ev_terms[2] = {};      // span of the term kernels since the last reset
    bool terms_open = false;
    // deferred weight verdict (MGC_OPT_DEFER_WEIGHT_CHECK)
    bool defer_check = false;
    bool bad_pending = false;
    int* h_bad = nullptr;              // pinned
    cudaEvent_t ev_bad = nullptr;
    cudaEvent_t ev_b[2] = {};          // the boundary kernel alone

    bool init_timed = false;           // ev[4..5] bracket the last k_init_tile
    bool boundary_timed = false;       // ev[2..3]... the boundary kernel's own events (ev_b) await reading
    bool caps_fresh = true;            // capacity arrays not written yet since create/reset (hold garbage)
    bool tr_fresh = true;              // same for tr[]
    bool state_init = false;
    bool flow_started = false;         // push kernels have run since the last reset: cap[] holds residuals, not the terms
    bool debug_checks = false;         // MEDPY_GC_DEBUG=1: device-side invariant + flow-conservation checks around every solve
    double debug_excess0 = 0.0;        // clamped source excess the solve started from
    bool fuse_build = true;            // mgc_build_voxel_graph uses the single-pass k_build_tile (MEDPY_GC_FUSE=0: four passes)
    // lazy build (gc_build.cuh, MODE 1): cold 8 x 8 x 32 blocks leave cap / tr / excess unwritten until the push passes
    // reach them.  bflag[block] = 1 once a block's planes are valid; d_lazy[0] counts such blocks.  The build's inputs,
    // tensor maps and parameters are kept until every block is materialised, the handle is reset or rebuilt.
    bool lazy_build = true;            // MEDPY_GC_LAZY=0: always eager
    bool keep_inputs = false;          // MGC_OPT_KEEP_INPUTS: caller-owned device inputs stay valid until the next build / reset
    bool lazy = false;                 // the current build left cold blocks behind
    int* bflag = nullptr;
    int* d_lazy = nullptr;
    BuildMaps lazy_maps{};
    BuildArgs lazy_args{};
    BoundaryParams lazy_P{};
    int64_t lazy_blocks = 0;           // build blocks of the last lazy build (0: eager)
    int64_t lazy_materialised = 0;     // ... of which hold their planes at the last read-out
    int build_chunks = 8;              // host inputs: z-chunks whose upload overlaps the build of the previous chunk
    bool solved = false;
    bool has_nlinks = false;
    double energy = 0.0;
    std::vector<uint8_t> host_mask;
    bool host_mask_valid = false;

    // tile solver (3-D lattices)
    Tiles TL{};
    Tiles4 TL4{};                      // 4-D lattices: 4x4x8x4 tiles (gc_tiles4.cuh)
    uint8_t* smask = nullptr;          // 4-D: residual sink link flag (the 8 arc bits fill rmask)
    bool use_tiles = false;
    int* pflag = nullptr;              // push: tile is already on the list its colour consumes next
    int* rflag = nullptr;              // relabel: tile is already on the next relabel list
    int* rl_items[2] = {nullptr, nullptr};     // relabel worklists (double buffered)
    int* pl_items[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // push worklists [colour][buffer]
    int* d_tcount = nullptr;           // [0..1] relabel counts, [2..5] push counts [colour*2+buffer], [8] cursor
    int pl_sel[2] = {0, 0};            // buffer each colour consumes next
    int rl_cur = 0;                    // relabel list consumed next
    bool labels_fresh = false;         // labels + relabel list 0 come straight from k_init_tile
    int n_ctas = 296;                  // persistent CTAs per tile-kernel launch
    bool use_coop = false;             // whole solve as one cooperative launch (gc_persist.cuh); opt-in, MEDPY_GC_COOP=1
    int coop_bfs_grid = 0;             // co-resident CTAs of k_bfs_coop (0: per-pass host loop)
    bool use_tma = false;              // push kernel stages its tile planes with TMA (gc_tma.cuh)
    PushMaps maps{};                   // tensor maps of cap[0..5] and excess
    int coop_grid = 0;                 // co-resident CTAs of k_solve_coop
    int tile_iters = 8;                // synchronous push/relabel rounds per tile visit
    int tile_iters_first = 4;          // ... in the first round after init (mostly stranded excess: measured best at 512^3)
    int iters_now = 8;
    int passes0 = 1, passes_max = 32;  // two-colour passes per round: starts at passes0, at most doubles per round
    // directional line sweeps in front of the worklist BFS (gc_sweep.cuh): used when more than 1/sweep_frac of the
    // tiles are waiting for labels (hard instances: the sink is far from most of the lattice)
    bool skip_first_test = true;       // MEDPY_GC_FIRST_TEST=1 restores the stop test of the first round
    int sweep_mode = -1;               // decided at the first relabel of a solve: 1 = hard instance (sweep at every relabel), 0 = worklist BFS only
    bool use_sweeps = true;
    int sweep_frac = 8;                // sweep when pending tiles > ntiles / sweep_frac
    int sweep_rounds_min = 1;          // rounds before the first fixed-point check (MEDPY_GC_SWEEP_MIN_ROUNDS); measured: 2 is slower
                                       // (one round + check + worklist BFS is the usual sequence; config 5 1.45 s vs 1.70 s)
    int sweep_rounds_max = 4;
    int sweep_done_frac = 16;          // hand over to the worklist BFS when violating tiles <= ntiles / sweep_done_frac (measured best on configs 2 / 4)

    // tuning
    int sweeps_per_round = 32;
    int relax_batch = 4;
    int64_t max_rounds = 100000;

    // z-slab solve inside the library (mgc_slab_comm_init / mgc_slab_solve): NCCL communicator of the slab ranks, border
    // message buffers [labels int32 | pad | flow float64] per neighbour and direction, stop-test scalars
    ncclComm_t comm = nullptr;
    int comm_rank = 0, comm_world = 1;
    char* msg[4] = {nullptr, nullptr, nullptr, nullptr};   // send_lo, send_hi, recv_lo, recv_hi (device)
    size_t msg_h_bytes = 0, msg_bytes = 0;
    long long* d_stat = nullptr;       // [changed in round A, changed in round B, active voxels] (device, all-reduced in place)
    long long* h_stat = nullptr;       // pinned mirror
    double* d_esum = nullptr;          // energy all-reduce
    int64_t slab_exchanges = 0, slab_relabel_rounds = 0, slab_push_passes = 0, slab_global_relabels = 0;
    // per-phase device time of the last mgc_slab_solve (CUDA events on the stream, resolved at the end of the solve):
    // [0] local BFS (reset + relax), [1] border exchanges (pack + NCCL send/recv + unpack), [2] stop test (count + all-reduce),
    // [3] push passes, [4] read-out + energy all-reduce; [5] = host time blocked in stream synchronisations (ms)
    std::vector<cudaEvent_t> ph_events;
    std::vector<int> ph_kind;
    size_t ph_used = 0;
    double slab_phase_ms[6] = {0, 0, 0, 0, 0, 0};

    mgc_stats st{};
    std::string err;
};

namespace {

void slab_comm_release(mgc_graph* g);

// NVTX range per phase (build / relabel / push / readout / exchange): visible in nsys / ncu timelines, a no-op without a
// profiler attached (SURVEY.md §5.1)
struct Nvtx {
    explicit Nvtx(const char* name) { nvtxRangePushA(name); }
    ~Nvtx() { nvtxRangePop(); }
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            g->err = std::string(#call) + ": " + cudaGetErrorString(_e);                           \
            return MGC_E_CUDA;                                                                     \
        }                                                                                          \
    } while (0)

#define FAIL(code, msg)                                                                            \
    do {                                                                                           \
        g->err = (msg);                                                                            \
        return (code);                                                                             \
    } while (0)

inline unsigned nblocks(const mgc_graph* g) { return (g->L.n + 255u) / 256u; }
// grid of the grid-stride reduction kernels (partials per launch)
inline unsigned rblocks(const mgc_graph* g) { const unsigned nb = nblocks(g); return nb < REDUCE_BLOCKS ? nb : REDUCE_BLOCKS; }

int alloc_buf(mgc_graph* g, size_t bytes, void** out)
{
    void* p = nullptr;
    cudaError_t e = pool_alloc(g->device, bytes, &p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        g->err = std::string("device allocation of ") + std::to_string(bytes) + " bytes failed: " + cudaGetErrorString(e);
        return MGC_E_NOMEM;
    }
    g->owned_bufs.push_back({p, bytes});
    g->device_bytes += (int64_t)round_up(bytes);
    *out = p;
    return MGC_OK;
}

int ensure_scratch(mgc_graph* g, Buf& b, size_t bytes)
{
    if (b.bytes >= bytes) return MGC_OK;
    if (b.p) {
        // a kernel or copy that is still in flight may be using the old block: drain before it goes back to the pool
        if (g->stream) cudaStreamSynchronize(g->stream);
        if (g->up_stream) cudaStreamSynchronize(g->up_stream);
        pool_free(g->device, b.bytes, b.p);
        g->device_bytes -= (int64_t)round_up(b.bytes);
    }
    b.p = nullptr; b.bytes = 0;
    void* p = nullptr;
    cudaError_t e = pool_alloc(g->device, bytes, &p);
    if (e != cudaSuccess) { cudaGetLastError(); g->err = "scratch allocation failed"; return MGC_E_NOMEM; }
    b.p = p; b.bytes = bytes;
    g->device_bytes += (int64_t)round_up(bytes);
    return MGC_OK;
}

// Bring an input array into a C-contiguous device buffer over the local lattice.  Returns a device pointer
// valid until the next stage_input on the same slot.
template <typename E>
int gather_launch(mgc_graph* g, const char* src, const Strides4& st, E* dst)
{
    // exact Fortran order over a 3-D lattice (the layout medpy.io.load hands out): coalesced tiled transpose
    const int Z = g->L.dim[0], Y = g->L.dim[1], X = g->L.dim[2];
    if (g->nd == 3 && Z > 1 && X > 1 && Y <= 65535 && (Z + 31) / 32 <= 65535 &&
        st.s[0] == (long long)sizeof(E) && (Y == 1 || st.s[1] == (long long)sizeof(E) * Z) && st.s[2] == (long long)sizeof(E) * Z * Y) {
        const dim3 grid((unsigned)((X + 31) / 32), (unsigned)Y, (unsigned)((Z + 31) / 32));
        k_gather_fortran3<E><<<grid, 256, 0, g->stream>>>(Z, Y, X, reinterpret_cast<const E*>(src), dst);
        g->st.kernel_launches++;
        return MGC_OK;
    }
    if (g->nd == 3) k_gather<E, 3><<<nblocks(g), 256, 0, g->stream>>>(g->L, src, st, dst);
    else            k_gather<E, 4><<<nblocks(g), 256, 0, g->stream>>>(g->L, src, st, dst);
    g->st.kernel_launches++;
    return MGC_OK;
}

// host -> device copy on the upload stream: waits until the staging slot's previous reader is done, makes the
// main stream wait for the copy, and blocks the HOST only until the copy itself has finished.
int upload(mgc_graph* g, void* dst, const void* src, size_t bytes, int slot)
{
    if (g->slot_used[slot]) CK(cudaStreamWaitEvent(g->up_stream, g->ev_slot[slot], 0));
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, g->up_stream));
    CK(cudaEventRecord(g->ev_up, g->up_stream));
    CK(cudaStreamWaitEvent(g->stream, g->ev_up, 0));
    CK(cudaEventSynchronize(g->ev_up));
    return MGC_OK;
}

// call after the kernel(s) that read the staging slots have been launched
void slots_release(mgc_graph* g, unsigned mask)
{
    // only the slots this call's kernels actually read: marking the others would make the NEXT call's upload wait for
    // this call's kernel although it targets a different buffer
    for (int i = 0; i < 5; ++i)
        if (mask & (1u << i)) { cudaEventRecord(g->ev_slot[i], g->stream); g->slot_used[i] = true; }
}

int stage_input(mgc_graph* g, const mgc_array* a, int slot, const void** out)
{
    const size_t es = dtype_size(a->dtype);
    if (!es) FAIL(MGC_E_ARG, "unsupported dtype");
    if (!a->data) FAIL(MGC_E_ARG, "null array");
    // canonical strides
    Strides4 st{};
    bool contiguous = true;
    long long span = (long long)es;
    long long expect = (long long)es;
    for (int d = g->nd - 1; d >= 0; --d) {
        long long s = 0;
        int ud = d - g->shift;
        if (ud >= 0) s = (long long)a->strides[ud];
        if (g->L.dim[d] > 1) {
            if (s <= 0) FAIL(MGC_E_ARG, "array strides must be positive (pass a contiguous copy)");
            if (s != expect) contiguous = false;
            span += (long long)(g->L.dim[d] - 1) * s;
        } else {
            s = 0;
        }
        st.s[d] = s;
        expect *= g->L.dim[d];
    }
    const size_t bytes = (size_t)g->L.n * es;
    if (contiguous && a->mem == MGC_MEM_DEVICE) { *out = a->data; return MGC_OK; }
    int rc = ensure_scratch(g, g->scratch[slot], bytes);
    if (rc) return rc;
    if (contiguous) {
        rc = upload(g, g->scratch[slot].p, a->data, bytes, slot);
        if (rc) return rc;
        *out = g->scratch[slot].p;
        return MGC_OK;
    }
    const char* src = (const char*)a->data;
    if (a->mem == MGC_MEM_HOST) {
        rc = ensure_scratch(g, g->raw, (size_t)span);
        if (rc) return rc;
        rc = upload(g, g->raw.p, a->data, (size_t)span, 3);
        if (rc) return rc;
        src = (const char*)g->raw.p;
    }
    else if (g->slot_used[slot]) CK(cudaStreamWaitEvent(g->stream, g->ev_slot[slot], 0));
    switch (a->dtype) {
        case MGC_F32: gather_launch<float>(g, src, st, (float*)g->scratch[slot].p); break;
        case MGC_F64: gather_launch<double>(g, src, st, (double*)g->scratch[slot].p); break;
        case MGC_U8: gather_launch<uint8_t>(g, src, st, (uint8_t*)g->scratch[slot].p); break;
        case MGC_I16: gather_launch<int16_t>(g, src, st, (int16_t*)g->scratch[slot].p); break;
        case MGC_I32: gather_launch<int32_t>(g, src, st, (int32_t*)g->scratch[slot].p); break;
    }
    CK(cudaGetLastError());
    // the gather is the last reader of the raw span: the next upload into it (same call, e.g. bg after fg) must wait
    if (a->mem == MGC_MEM_HOST) { CK(cudaEventRecord(g->ev_slot[3], g->stream)); g->slot_used[3] = true; }
    *out = g->scratch[slot].p;
    return MGC_OK;
}

int finish_flow_const(mgc_graph* g)
{
    k_sum_partials<<<1, 256, 0, g->stream>>>(g->partials, rblocks(g), g->d_scalars);
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    return MGC_OK;
}

void invalidate(mgc_graph* g)
{
    g->state_init = false;
    g->solved = false;
    g->host_mask_valid = false;
}

struct Timer {
    mgc_graph* g;
    double* acc;
    Timer(mgc_graph* g_, double* acc_) : g(g_), acc(acc_) { cudaEventRecord(g->ev[0], g->stream); }
    void stop_sync()
    {
        cudaEventRecord(g->ev[1], g->stream);
        cudaEventSynchronize(g->ev[1]);
        float ms = 0;
        cudaEventElapsedTime(&ms, g->ev[0], g->ev[1]);
        *acc += ms;
    }
};

// term kernels are not synchronised one by one: their span on the stream is measured between the first term after a
// reset and the last term before the solve, and read when the solve synchronises anyway
struct TermSpan {
    mgc_graph* g;
    explicit TermSpan(mgc_graph* g_) : g(g_)
    {
        if (!g->terms_open) { cudaEventRecord(g->ev_terms[0], g->stream); g->terms_open = true; }
    }
    void stop(unsigned slot_mask) { slots_release(g, slot_mask); cudaEventRecord(g->ev_terms[1], g->stream); }
};

void resolve_term_span(mgc_graph* g)
{
    if (!g->terms_open) return;
    if (cudaEventSynchronize(g->ev_terms[1]) == cudaSuccess) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, g->ev_terms[0], g->ev_terms[1]) == cudaSuccess) g->st.ms_terms += ms;
        if (g->boundary_timed && cudaEventElapsedTime(&ms, g->ev_b[0], g->ev_b[1]) == cudaSuccess) g->st.ms_boundary = ms;
        g->boundary_timed = false;
    }
    g->terms_open = false;
}

// deliver a deferred weight verdict: waits for the boundary kernel that produced it
int check_pending(mgc_graph* g)
{
    if (!g->bad_pending) return MGC_OK;
    g->bad_pending = false;
    CK(cudaEventSynchronize(g->ev_bad));
    if (*g->h_bad) FAIL(MGC_E_WEIGHT, "Negative or zero weights are not allowed.");
    return MGC_OK;
}

// rank-3 float64 tensor maps with an 8x8x8 box over the local lattice (x fastest); driver entry point resolved at run
// time so the library does not link libcuda
typedef CUresult (*tmap_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
tmap_encode_fn tensor_map_encoder()
{
    static tmap_encode_fn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) {
            cudaGetLastError();
            return nullptr;
        }
        encode = (tmap_encode_fn)fn;
    }
    return encode;
}

bool make_push_maps(mgc_graph* g)
{
    tmap_encode_fn encode = tensor_map_encoder();
    if (!encode) return false;
    const cuuint64_t X = (cuuint64_t)g->L.dim[2], Y = (cuuint64_t)g->L.dim[1], Z = (cuuint64_t)g->L.dim[0];
    if (X % 2) return false;                                   // global strides must be multiples of 16 B
    const cuuint64_t dims[3] = {X, Y, Z};
    const cuuint64_t strides[2] = {X * 8, X * Y * 8};
    const cuuint32_t box[3] = {TILE, TILE, TILE};
    const cuuint32_t estr[3] = {1, 1, 1};
    for (int p = 0; p < TMA_PLANES; ++p) {
        void* base = p < 6 ? (void*)g->S.cap[p] : (void*)g->S.excess;
        if (((uintptr_t)base) & 15) return false;
        if (encode(&g->maps.m[p], CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return false;
    }
    return true;
}

int create_impl(int32_t ndim, const int64_t* shape, int64_t z0, int64_t z1, bool slab, int32_t device, mgc_graph** out)
{
    if (!out) return MGC_E_ARG;
    *out = nullptr;
    if (ndim < 1 || ndim > MGC_MAX_NDIM || !shape) { g_create_error = "ndim must be 1..4"; return MGC_E_ARG; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        g_create_error = std::string("no usable CUDA device (this library has no CPU path): ") + cudaGetErrorString(e);
        return MGC_E_CUDA;
    }
    if (device < 0) cudaGetDevice(&device);
    if (device >= ndev) { g_create_error = "bad device ordinal"; return MGC_E_ARG; }
    e = cudaSetDevice(device);
    if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); return MGC_E_CUDA; }

    mgc_graph* g = new mgc_graph();
    g->device = device;
    g->user_ndim = ndim;
    g->nd = ndim == 4 ? 4 : 3;
    g->shift = g->nd - ndim;
    for (int d = 0; d < ndim; ++d) {
        if (shape[d] < 1) { g_create_error = "extents must be >= 1"; delete g; return MGC_E_ARG; }
        g->user_shape[d] = shape[d];
    }
    int64_t dims[4] = {1, 1, 1, 1};
    for (int d = 0; d < ndim; ++d) dims[d + g->shift] = shape[d];
    g->slab = slab;
    int own0 = 0, own1 = (int)dims[0];
    if (slab) {
        if (g->shift != 0 || z0 < 0 || z1 > shape[0] || z0 >= z1) { g_create_error = "bad slab"; delete g; return MGC_E_ARG; }
        g->global_dim0 = shape[0]; g->z0 = z0; g->z1 = z1;
        g->ghost_lo = z0 > 0; g->ghost_hi = z1 < shape[0];
        dims[0] = (z1 - z0) + (g->ghost_lo ? 1 : 0) + (g->ghost_hi ? 1 : 0);
        own0 = g->ghost_lo ? 1 : 0;
        own1 = own0 + (int)(z1 - z0);
    }
    int64_t n = 1;
    for (int d = 0; d < g->nd; ++d) n *= dims[d];
    if (n >= (int64_t(1) << 31)) { g_create_error = "lattice too large for one device handle (>= 2^31 voxels)"; delete g; return MGC_E_ARG; }
    g->L.nd = g->nd;
    unsigned s = (unsigned)n;
    for (int d = 0; d < 4; ++d) { g->L.dim[d] = 1; g->L.stride[d] = 1; }
    for (int d = 0; d < g->nd; ++d) { g->L.dim[d] = (int)dims[d]; s /= (unsigned)dims[d]; g->L.stride[d] = s; }
    for (int d = 0; d < 4; ++d) {
        const unsigned long long st = g->L.stride[d];
        // ceil(2^64 / st) = floor((2^64 - 1) / st) + 1 for st > 1 that does not divide 2^64 ... and also when it does
        g->L.magic[d] = st <= 1 ? 0ull : (~0ull / st) + 1ull;
    }
    g->L.n = (unsigned)n;
    g->L.plane = g->L.stride[0];
    g->L.own0 = own0; g->L.own1 = own1;

    int rc = MGC_OK;
    const size_t nb = (size_t)n;
    void* p = nullptr;
    for (int k = 0; k < 2 * g->nd && !rc; ++k) { rc = alloc_buf(g, nb * sizeof(double), &p); g->S.cap[k] = (double*)p; }
    if (!rc) { rc = alloc_buf(g, nb * sizeof(double), &p); g->S.excess = (double*)p; }
    if (!rc) { rc = alloc_buf(g, nb * sizeof(double), &p); g->S.sink = (double*)p; }
    if (!rc) { rc = alloc_buf(g, nb * sizeof(double), &p); g->S.tr = (double*)p; }
    if (!rc) { rc = alloc_buf(g, nb * sizeof(int), &p); g->S.height = (int*)p; }
    if (!rc) { rc = alloc_buf(g, nb, &p); g->S.rmask = (uint8_t*)p; }
    if (!rc) { rc = alloc_buf(g, nb, &p); g->mask_dev = (uint8_t*)p; }
    g->n_partials = nblocks(g);
    if (g->nd == 3) {   // k_build_tile writes one partial per 8 x 8 x 32 block
        const unsigned nbuild = (unsigned)((g->L.dim[0] + 7) / 8) * (unsigned)((g->L.dim[1] + 7) / 8) * (unsigned)((g->L.dim[2] + 31) / 32);
        if (nbuild > g->n_partials) g->n_partials = nbuild;
    }
    if (!rc) { rc = alloc_buf(g, (size_t)g->n_partials * sizeof(double), &p); g->partials = (double*)p; }
    if (!rc) { rc = alloc_buf(g, 3 * 1024 * sizeof(double), &p); g->minmax_buf = p; }
    if (!rc) { rc = alloc_buf(g, 64, &p); g->d_scalars = (double*)p; }
    if (!rc) { rc = alloc_buf(g, 64, &p); g->d_flags = (int*)p; }
    if (!rc) { rc = alloc_buf(g, 64, &p); g->d_count = (unsigned long long*)p; }
    if (!rc && g->nd == 3) {
        for (int d = 0; d < 3; ++d) g->TL.nt[d] = (g->L.dim[d] + TILE - 1) / TILE;
        g->TL.ntiles = g->TL.nt[0] * g->TL.nt[1] * g->TL.nt[2];
        const size_t tb = (size_t)g->TL.ntiles * sizeof(int);
        if (!rc) { rc = alloc_buf(g, tb, &p); g->pflag = (int*)p; }
        if (!rc) { rc = alloc_buf(g, tb, &p); g->rflag = (int*)p; }
        for (int i = 0; i < 2 && !rc; ++i) { rc = alloc_buf(g, tb, &p); g->rl_items[i] = (int*)p; }
        for (int i = 0; i < 4 && !rc; ++i) { rc = alloc_buf(g, tb, &p); g->pl_items[i >> 1][i & 1] = (int*)p; }
        if (!rc) { rc = alloc_buf(g, 256, &p); g->d_tcount = (int*)p; }
        if (!rc && !slab) {
            const size_t nbuild = (size_t)((g->L.dim[0] + 7) / 8) * ((g->L.dim[1] + 7) / 8) * ((g->L.dim[2] + 31) / 32);
            rc = alloc_buf(g, nbuild * sizeof(int), &p); g->bflag = (int*)p;
            if (!rc) { rc = alloc_buf(g, 64, &p); g->d_lazy = (int*)p; }
        }
        {   // dirty-tile tracking for the partial relabel reset (MEDPY_GC_PARTIAL_RESET=0: off)
            const char* ed = getenv("MEDPY_GC_PARTIAL_RESET");
            g->TL.dflag = nullptr; g->TL.ditems = nullptr; g->TL.dcount = nullptr;
            g->TL.schg = nullptr; g->TL.sweep_stamp = 0;
            {   // MEDPY_GC_SWEEP_CHECK=0: tile marks + k_sweep_list instead of the exhaustive fixed-point check.  Measured SLOWER
                // (1024^3: 1.66 s vs 1.45 s): "changed in the last round, or next to it" is a much larger worklist than "still
                // violating", and the finishing BFS pays per listed tile -- so the check pass stays the default.
                const char* es = getenv("MEDPY_GC_SWEEP_CHECK");
                if (!rc && es && atoi(es) == 0) {
                    rc = alloc_buf(g, tb, &p); g->TL.schg = (int*)p;
                    if (!rc && cudaMemset(p, 0, tb) != cudaSuccess) { cudaGetLastError(); g->TL.schg = nullptr; }
                }
            }
            if (!rc && (!ed || atoi(ed) != 0)) {
                rc = alloc_buf(g, tb, &p); g->TL.dflag = (int*)p;
                if (!rc) { rc = alloc_buf(g, tb, &p); g->TL.ditems = (int*)p; }
                if (!rc) { rc = alloc_buf(g, 64, &p); g->TL.dcount = (int*)p; }
            }
        }
        g->n_ctas = 2 * cached_sm_count(device);   // k_push_tile is built for 2 CTAs per SM
        g->use_tiles = true;
        if (const char* sv = getenv("MEDPY_GC_SOLVER")) if (!strcmp(sv, "v0")) g->use_tiles = false;
        if (const char* e1 = getenv("MEDPY_GC_ITERS")) if (atoi(e1) > 0) g->tile_iters = g->tile_iters_first = atoi(e1);
        if (const char* e2 = getenv("MEDPY_GC_PASSES0")) if (atoi(e2) > 0) g->passes0 = atoi(e2);
        if (const char* e3 = getenv("MEDPY_GC_PASSES_MAX")) if (atoi(e3) > 0) g->passes_max = atoi(e3);
        if (const char* e4 = getenv("MEDPY_GC_COOP")) g->use_coop = atoi(e4) != 0;
        if (const char* e7 = getenv("MEDPY_GC_SWEEP")) g->use_sweeps = atoi(e7) != 0;
        if (const char* e8 = getenv("MEDPY_GC_SWEEP_FRAC")) if (atoi(e8) > 0) g->sweep_frac = atoi(e8);
        if (const char* e9 = getenv("MEDPY_GC_SWEEP_ROUNDS")) if (atoi(e9) > 0) g->sweep_rounds_max = atoi(e9);
        if (const char* e11 = getenv("MEDPY_GC_SWEEP_MIN_ROUNDS")) if (atoi(e11) > 0) g->sweep_rounds_min = atoi(e11);
        if (const char* e10 = getenv("MEDPY_GC_SWEEP_DONE_FRAC")) if (atoi(e10) > 0) g->sweep_done_frac = atoi(e10);
        {
            const char* e6 = getenv("MEDPY_GC_TMA");
            const size_t smem = 2 * TMA_STAGE_BYTES + 6 * TILE_VOX * sizeof(double) + 1024 * sizeof(int) + 64;
            if ((!e6 || atoi(e6) != 0) && make_push_maps(g) &&
                cudaFuncSetAttribute(k_push_tile_tma<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess)
                g->use_tma = true;
            else
                cudaGetLastError();
        }
        {
            int coop = 0, nb = 0;
            const char* e5 = getenv("MEDPY_GC_BFS");
            cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
            if ((!e5 || strcmp(e5, "host") != 0) && coop &&
                cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_bfs_coop, TILE_VOX, 0) == cudaSuccess && nb >= 1)
                g->coop_bfs_grid = nb * cached_sm_count(device);
            else
                cudaGetLastError();
        }
        {
            int coop = 0, nb = 0;
            cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
            if (!g->use_coop) { /* not requested */ }
            else if (!coop || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_solve_coop<double>, TILE_VOX, 0) != cudaSuccess || nb < 1) {
                cudaGetLastError();
                g->use_coop = false;
            } else {
                g->coop_grid = nb * cached_sm_count(device);
            }
        }
    }
    if (!rc && g->nd == 4 && !slab) {
        const int ext[4] = {4, 4, 8, 4};
        g->TL4.ntiles = 1;
        for (int d = 0; d < 4; ++d) { g->TL4.nt[d] = (g->L.dim[d] + ext[d] - 1) / ext[d]; g->TL4.ntiles *= g->TL4.nt[d]; }
        g->TL.ntiles = g->TL4.ntiles;   // list sizes / shared helpers
        const size_t tb = (size_t)g->TL4.ntiles * sizeof(int);
        if (!rc) { rc = alloc_buf(g, tb, &p); g->pflag = (int*)p; }
        if (!rc) { rc = alloc_buf(g, tb, &p); g->rflag = (int*)p; }
        for (int i = 0; i < 2 && !rc; ++i) { rc = alloc_buf(g, tb, &p); g->rl_items[i] = (int*)p; }
        for (int i = 0; i < 4 && !rc; ++i) { rc = alloc_buf(g, tb, &p); g->pl_items[i >> 1][i & 1] = (int*)p; }
        if (!rc) { rc = alloc_buf(g, 256, &p); g->d_tcount = (int*)p; }
        if (!rc) { rc = alloc_buf(g, nb, &p); g->smask = (uint8_t*)p; }
        g->n_ctas = 2 * cached_sm_count(device);
        g->use_tiles = true;
        if (const char* sv = getenv("MEDPY_GC_SOLVER")) if (!strcmp(sv, "v0")) g->use_tiles = false;
        {
            int coop = 0, nbk = 0;
            const char* e5 = getenv("MEDPY_GC_BFS");
            cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
            if ((!e5 || strcmp(e5, "host") != 0) && coop &&
                cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nbk, k_bfs_coop4, T4_VOX, 0) == cudaSuccess && nbk >= 1)
                g->coop_bfs_grid = nbk * cached_sm_count(device);
            else
                cudaGetLastError();
        }
        if (const char* e1 = getenv("MEDPY_GC_ITERS")) if (atoi(e1) > 0) g->tile_iters = atoi(e1);
        if (const char* e2 = getenv("MEDPY_GC_PASSES0")) if (atoi(e2) > 0) g->passes0 = atoi(e2);
        if (const char* e3 = getenv("MEDPY_GC_PASSES_MAX")) if (atoi(e3) > 0) g->passes_max = atoi(e3);
        if (const char* e7 = getenv("MEDPY_GC_SWEEP")) g->use_sweeps = atoi(e7) != 0;
        if (const char* e8 = getenv("MEDPY_GC_SWEEP_FRAC")) if (atoi(e8) > 0) g->sweep_frac = atoi(e8);
        if (const char* e9 = getenv("MEDPY_GC_SWEEP_ROUNDS")) if (atoi(e9) > 0) g->sweep_rounds_max = atoi(e9);
        if (const char* e10 = getenv("MEDPY_GC_SWEEP_DONE_FRAC")) if (atoi(e10) > 0) g->sweep_done_frac = atoi(e10);
    }
    if (rc) { g_create_error = g->err; mgc_destroy(g); return rc; }
    if (cudaStreamCreate(&g->stream) != cudaSuccess) { g_create_error = "cudaStreamCreate failed"; mgc_destroy(g); return MGC_E_CUDA; }
    g->own_stream = true;
    for (auto& ev : g->ev) cudaEventCreate(&ev);
    cudaStreamCreateWithFlags(&g->up_stream, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&g->ev_up, cudaEventDisableTiming);
    for (auto& ev : g->ev_slot) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    for (auto& ev : g->ev_chunk) cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    for (auto& ev : g->ev_terms) cudaEventCreate(&ev);
    if (const char* f0 = getenv("MEDPY_GC_DEBUG")) g->debug_checks = atoi(f0) != 0;
    if (const char* f3 = getenv("MEDPY_GC_FIRST_TEST")) g->skip_first_test = atoi(f3) == 0;
    if (const char* f1 = getenv("MEDPY_GC_FUSE")) g->fuse_build = atoi(f1) != 0;
    if (const char* f4 = getenv("MEDPY_GC_LAZY")) g->lazy_build = atoi(f4) != 0;
    if (const char* f2 = getenv("MEDPY_GC_CHUNKS")) if (atoi(f2) > 0) g->build_chunks = atoi(f2);
    cudaEventCreateWithFlags(&g->ev_bad, cudaEventDisableTiming);
    for (auto& ev : g->ev_b) cudaEventCreate(&ev);
    // [0] weight verdict, [2..3] active count.  From the pinned pool: cudaHostAlloc / cudaFreeHost per handle (one handle per
    // graph_from_voxels call) are heavyweight driver calls that synchronise the device
    { void* hp = nullptr; g->h_bad = (mgc_host_alloc(64, &hp) == MGC_OK) ? (int*)hp : nullptr; }
    if (const char* s1 = getenv("MEDPY_GC_SWEEPS")) g->sweeps_per_round = atoi(s1) > 0 ? atoi(s1) : g->sweeps_per_round;
    if (const char* s2 = getenv("MEDPY_GC_RELAX_BATCH")) g->relax_batch = atoi(s2) > 0 ? atoi(s2) : g->relax_batch;
    g->st.n_voxels = (int64_t)n;
    rc = mgc_reset(g);
    if (rc) { g_create_error = g->err; mgc_destroy(g); return rc; }
    *out = g;
    return MGC_OK;
}

template <typename E, int ND, bool FRESH>
void boundary_launch_nd(mgc_graph* g, const E* img, const BoundaryParams& P)
{
    const dim3 grid(nblocks(g)), block(256);
    // specialised instances: exponential term, no spacing, float32 / float64 images (every BASELINE configuration)
    if (P.fn == 1 && P.inv_spacing_on == 0.0 && (sizeof(E) == 4 || sizeof(E) == 8) && !std::is_integral<E>::value) {
        if (P.use_max) k_boundary<E, ND, double, FRESH, 1, 1, 0><<<grid, block, 0, g->stream>>>(g->L, g->S, img, P, g->d_flags);
        else           k_boundary<E, ND, double, FRESH, 1, 0, 0><<<grid, block, 0, g->stream>>>(g->L, g->S, img, P, g->d_flags);
        return;
    }
    k_boundary<E, ND, double, FRESH><<<grid, block, 0, g->stream>>>(g->L, g->S, img, P, g->d_flags);
}

template <typename E>
int boundary_launch(mgc_graph* g, const E* img, const BoundaryParams& P)
{
    if (g->caps_fresh) {
        if (g->nd == 3) boundary_launch_nd<E, 3, true>(g, img, P);
        else            boundary_launch_nd<E, 4, true>(g, img, P);
    } else {
        if (g->nd == 3) boundary_launch_nd<E, 3, false>(g, img, P);
        else            boundary_launch_nd<E, 4, false>(g, img, P);
    }
    g->caps_fresh = false;
    g->st.kernel_launches++;
    return MGC_OK;
}

template <typename E>
int minmax_launch(mgc_graph* g, const E* img)
{
    unsigned nb = g->n_partials < 1024u ? g->n_partials : 1024u;
    E* pm = (E*)g->minmax_buf;
    E* px = pm + 1024;
    E* pa = px + 1024;
    k_minmax_partial<E><<<nb, 256, 0, g->stream>>>(img, g->L.n, pm, px, pa);
    k_minmax_final<E><<<1, 32, 0, g->stream>>>(pm, px, pa, nb, g->d_scalars + 2);
    g->st.kernel_launches += 2;
    return MGC_OK;
}

// parameters of one of the eight boundary terms; the linear normaliser is computed on the device (K0) when `norm` is NaN
int boundary_params(mgc_graph* g, int kind, int dtype, const void* img, double sigma, const double* spacing, double norm, BoundaryParams* out)
{
    BoundaryParams P{};
    P.fn = kind & 3;
    // boundary_maximum_division computes the difference variant (energy_voxel.py:347)
    P.use_max = (kind >= 4 && kind != MGC_BOUNDARY_MAXIMUM_DIVISION) ? 1 : 0;
    P.sigma = (P.fn == 1) ? pow(sigma, 2) : sigma;   // math.pow(sigma, 2), energy_voxel.py:231
    P.inv_sigma2 = (P.fn == 1 && P.sigma != 0.0) ? 1.0 / P.sigma : 0.0;
    P.inv_spacing_on = spacing ? 1.0 : 0.0;
    for (int d = 0; d < 4; ++d) P.spacing[d] = 1.0;
    if (spacing) for (int d = 0; d < g->user_ndim; ++d) P.spacing[d + g->shift] = spacing[d];
    P.norm = norm;
    if (P.fn == 0 && std::isnan(norm)) {
        if (g->slab) FAIL(MGC_E_ARG, "z-slab handles need the global normaliser of the linear terms");
        int rc = MGC_OK;
        switch (dtype) {
            case MGC_F32: rc = minmax_launch<float>(g, (const float*)img); break;
            case MGC_F64: rc = minmax_launch<double>(g, (const double*)img); break;
            case MGC_U8: rc = minmax_launch<uint8_t>(g, (const uint8_t*)img); break;
            case MGC_I16: rc = minmax_launch<int16_t>(g, (const int16_t*)img); break;
            case MGC_I32: rc = minmax_launch<int32_t>(g, (const int32_t*)img); break;
        }
        if (rc) return rc;
        double mm[2];
        CK(cudaMemcpyAsync(mm, g->d_scalars + 2, sizeof(mm), cudaMemcpyDeviceToHost, g->stream));
        CK(cudaStreamSynchronize(g->stream));
        P.norm = (kind == MGC_BOUNDARY_MAXIMUM_LINEAR) ? mm[1] : mm[0];
    }
    *out = P;
    return MGC_OK;
}

// terms that were never given leave their arrays unwritten: zero them before anything reads them
int materialise_zeros(mgc_graph* g)
{
    const size_t nb = (size_t)g->L.n;
    if (g->caps_fresh) {
        for (int k = 0; k < 2 * g->nd; ++k) CK(cudaMemsetAsync(g->S.cap[k], 0, nb * sizeof(double), g->stream));
        g->caps_fresh = false;
    }
    if (g->tr_fresh) {
        CK(cudaMemsetAsync(g->S.tr, 0, nb * sizeof(double), g->stream));
        g->tr_fresh = false;
    }
    return MGC_OK;
}

int ensure_state(mgc_graph* g)
{
    if (g->state_init) return MGC_OK;
    { int rc0 = materialise_zeros(g); if (rc0) return rc0; }
    if (g->nd == 3) k_init_state<3, double><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S);
    else            k_init_state<4, double><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S);
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    g->state_init = true;
    return MGC_OK;
}

int relabel_init(mgc_graph* g)
{
    if (g->nd == 3) k_relabel_init<3, double><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S);
    else            k_relabel_init<4, double><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S);
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    return MGC_OK;
}

// relax until a whole batch changes nothing; *any = 1 if anything changed at all
int relabel_relax(mgc_graph* g, int* any)
{
    *any = 0;
    for (;;) {
        CK(cudaMemsetAsync(g->d_flags + 1, 0, sizeof(int), g->stream));
        cudaEventRecord(g->ev[2], g->stream);
        for (int i = 0; i < g->relax_batch; ++i) {
            if (g->nd == 3) k_relabel_relax<3><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S.rmask, g->S.height, g->d_flags + 1);
            else            k_relabel_relax<4><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S.rmask, g->S.height, g->d_flags + 1);
        }
        g->st.kernel_launches += g->relax_batch;
        g->st.relabel_sweeps += g->relax_batch;
        cudaEventRecord(g->ev[3], g->stream);
        int changed = 0;
        CK(cudaMemcpyAsync(&changed, g->d_flags + 1, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
        CK(cudaStreamSynchronize(g->stream));
        { float ms = 0; cudaEventElapsedTime(&ms, g->ev[2], g->ev[3]); g->st.ms_relabel += ms; }
        if (!changed) break;
        *any = 1;
    }
    return MGC_OK;
}

int count_active(mgc_graph* g, int64_t* out)
{
    CK(cudaMemsetAsync(g->d_count, 0, sizeof(unsigned long long), g->stream));
    k_count_active<double><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S, g->d_count);
    g->st.kernel_launches++;
    unsigned long long c = 0;
    CK(cudaMemcpyAsync(&c, g->d_count, sizeof(c), cudaMemcpyDeviceToHost, g->stream));
    CK(cudaStreamSynchronize(g->stream));
    *out = (int64_t)c;
    g->st.active_last = (int64_t)c;
    return MGC_OK;
}

// n push sweeps; *work_last = whether the last sweep still found an active voxel
int push_sweeps(mgc_graph* g, int n, int* work_last)
{
    g->flow_started = true;
    if (work_last) cudaEventRecord(g->ev[2], g->stream);
    for (int i = 0; i < n; ++i) {
        if (i == n - 1) CK(cudaMemsetAsync(g->d_flags + 2, 0, sizeof(int), g->stream));
        if (g->nd == 3) k_push<3, double><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S, g->d_flags + 2);
        else            k_push<4, double><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S, g->d_flags + 2);
    }
    g->st.kernel_launches += n;
    g->st.push_sweeps += n;
    CK(cudaGetLastError());
    if (work_last) {
        cudaEventRecord(g->ev[3], g->stream);
        CK(cudaMemcpyAsync(work_last, g->d_flags + 2, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
        CK(cudaStreamSynchronize(g->stream));
        float ms = 0;
        cudaEventElapsedTime(&ms, g->ev[2], g->ev[3]);
        g->st.ms_push += ms;
    }
    return MGC_OK;
}

// ---- tile solver driver --------------------------------------------------------------------------------
WorkList rl(mgc_graph* g, int i) { return WorkList{g->rl_items[i], g->d_tcount + i}; }
WorkList pl(mgc_graph* g, int color, int buf) { return WorkList{g->pl_items[color][buf], g->d_tcount + 2 + color * 2 + buf}; }
int* cursor(mgc_graph* g) { return g->d_tcount + 8; }

int read_tcount(mgc_graph* g, int idx, int* out)
{
    CK(cudaMemcpyAsync(out, g->d_tcount + idx, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
    CK(cudaStreamSynchronize(g->stream));
    return MGC_OK;
}

// forget the dirty tiles (everything is in the reset state: fresh build / init, or a full reset just ran)
int dirty_clear(mgc_graph* g)
{
    if (g->nd == 3 && g->TL.dflag) {
        CK(cudaMemsetAsync(g->TL.dflag, 0, (size_t)g->TL.ntiles * sizeof(int), g->stream));
        CK(cudaMemsetAsync(g->TL.dcount, 0, sizeof(int), g->stream));
    }
    return MGC_OK;
}

// first call: solver state + first labels + first worklists in one pass (k_init_tile)
int init_tiles(mgc_graph* g)
{
    Nvtx range("mgc:init_state");
    CK(cudaMemsetAsync(g->d_tcount, 0, 256, g->stream));
    g->pl_sel[0] = g->pl_sel[1] = 0;
    cudaEventRecord(g->ev[4], g->stream);
    if (g->nd == 4)
        k_init_tile4<double><<<g->TL4.ntiles, T4_VOX, 0, g->stream>>>(g->L, g->TL4, g->S, g->smask, g->rflag, rl(g, 0), g->pflag,
                                                                      pl(g, 0, 0), pl(g, 1, 0));
    else
    k_init_tile<double><<<g->TL.ntiles, TILE_VOX, 0, g->stream>>>(g->L, g->TL, g->S, g->rflag, rl(g, 0), g->pflag,
                                                                  pl(g, 0, 0), pl(g, 1, 0));
    cudaEventRecord(g->ev[5], g->stream);
    g->init_timed = true;
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    g->state_init = true;
    g->labels_fresh = true;
    g->rl_cur = 0;
    g->sweep_mode = -1;
    return dirty_clear(g);
}

// exact global relabel by tile-wise relaxation; work is proportional to the tiles whose labels still move.
// begin: labels from the residual mask + a fresh worklist (skipped when k_init_tile just produced both)
int relabel_tiles_begin(mgc_graph* g)
{
    if (g->labels_fresh) {
        g->labels_fresh = false;
        g->rl_cur = 0;
        CK(cudaMemsetAsync(g->d_tcount + CTL_RLCUR, 0, sizeof(int), g->stream));
        return MGC_OK;
    }
    CK(cudaMemsetAsync(g->d_tcount, 0, 2 * sizeof(int), g->stream));
    CK(cudaMemsetAsync(g->rflag, 0, (size_t)g->TL.ntiles * sizeof(int), g->stream));
    if (g->nd == 4) {
        k_relabel_reset4<<<g->TL4.ntiles, T4_VOX, 0, g->stream>>>(g->L, g->TL4, g->S.rmask, g->smask, g->S.height, g->rflag, rl(g, 0));
    } else {
        if (g->TL.dflag && g->sweep_mode == 0) {
            // easy instance: only the tiles written since the last reset (labels / sink-link bits) are not in the reset state
            k_relabel_reset_list<<<g->n_ctas * 2, TILE_VOX, 0, g->stream>>>(g->L, g->TL, g->S.rmask, g->S.height, g->rflag, rl(g, 0));
            CK(cudaMemsetAsync(g->TL.dcount, 0, sizeof(int), g->stream));
        } else {
            const unsigned nruns = (unsigned)g->L.dim[0] * (unsigned)g->L.dim[1] * (unsigned)g->TL.nt[2];
            unsigned grid = (nruns + 255u) / 256u;
            if (grid > (unsigned)g->n_ctas * 8u) grid = (unsigned)g->n_ctas * 8u;
            k_relabel_reset<<<grid, 256, 0, g->stream>>>(g->L, g->TL, g->S.rmask, g->S.height, g->rflag, rl(g, 0));
            int rcd = dirty_clear(g);
            if (rcd) return rcd;
        }
    }
    g->st.kernel_launches++;
    g->rl_cur = 0;
    CK(cudaMemsetAsync(g->d_tcount + CTL_RLCUR, 0, sizeof(int), g->stream));
    CK(cudaGetLastError());
    return MGC_OK;
}

// run passes until the current worklist is empty; *any = 1 if any tile was visited
// one round of directional sweeps (both directions of every axis), then the list of tiles that are not at the fixed
// point yet (gc_sweep.cuh); *pending = number of such tiles (host synchronisation)
int relabel_sweep_round(mgc_graph* g, int* pending, bool with_check)
{
    const int last = g->nd - 1;
    if (g->nd == 3 && g->TL.schg) g->TL.sweep_stamp++;        // marks of this round (the array is never cleared)
    for (int a = 0; a < last; ++a) {
        if (g->L.dim[a] < 2) continue;
        const unsigned nlines = g->L.n / (unsigned)g->L.dim[a];
        k_sweep_axis<<<(nlines + 255u) / 256u, 256, 0, g->stream>>>(g->L, g->TL, g->S.rmask, g->S.height, a);
        g->st.kernel_launches++;
    }
    const bool marks = g->nd == 3 && g->TL.schg;      // the short-row kernel does not mark tiles: 3-D lattices use the general one
    if (g->L.dim[last] >= 2 && g->L.dim[last] <= SWEEP_SHORT && !marks) {
        const unsigned nrows = g->L.n / (unsigned)g->L.dim[last];
        k_sweep_rows_short<<<(nrows + 255u) / 256u, 256, 0, g->stream>>>(g->L, g->S.rmask, g->S.height);
        g->st.kernel_launches++;
    } else if (g->L.dim[last] >= 2) {
        const unsigned nrows = g->L.n / (unsigned)g->L.dim[last];
        unsigned grid = (nrows + SWEEP_WARPS - 1) / SWEEP_WARPS;
        const unsigned cap = (unsigned)cached_sm_count(g->device) * 16u;
        if (grid > cap) grid = cap;
        k_sweep_rows<<<grid, 32 * SWEEP_WARPS, 0, g->stream>>>(g->L, g->TL, g->S.rmask, g->S.height);
        g->st.kernel_launches++;
    }
    g->st.relabel_sweeps++;
    if (!with_check) { CK(cudaGetLastError()); return MGC_OK; }     // an early round: the next one follows without a verdict
    CK(cudaMemsetAsync(g->d_tcount, 0, 2 * sizeof(int), g->stream));
    CK(cudaMemsetAsync(g->rflag, 0, (size_t)g->TL.ntiles * sizeof(int), g->stream));
    if (g->nd == 4) k_relabel_check4<<<nblocks(g), 256, 0, g->stream>>>(g->L, g->TL4, g->S.rmask, g->S.height, g->rflag, rl(g, 0));
    else if (g->TL.schg) k_sweep_list<<<(g->TL.ntiles + 255) / 256, 256, 0, g->stream>>>(g->TL, g->rflag, rl(g, 0));
    else            k_relabel_check<<<nblocks(g), 256, 0, g->stream>>>(g->L, g->TL, g->S.rmask, g->S.height, g->rflag, rl(g, 0));
    g->st.kernel_launches++;
    g->rl_cur = 0;
    CK(cudaMemsetAsync(g->d_tcount + CTL_RLCUR, 0, sizeof(int), g->stream));
    CK(cudaGetLastError());
    return read_tcount(g, 0, pending);
}

int relabel_tiles_run(mgc_graph* g, int* any, bool want_any = true)
{
    *any = 0;
    if (g->use_sweeps && g->use_tiles && g->TL.ntiles >= 64 && g->sweep_mode != 0) {
        int pending = 0;
        int rc = read_tcount(g, g->rl_cur, &pending);
        if (rc) return rc;
        // one decision per solve (one host synchronisation): an instance whose first relabel has to label most of the
        // lattice is a hard one at every later relabel too, an easy one (regional term: most voxels own a sink link) never is
        if (g->sweep_mode < 0) g->sweep_mode = pending > g->TL.ntiles / g->sweep_frac ? 1 : 0;
        if (pending > g->TL.ntiles / g->sweep_frac) {
            *any = 1;
            int prev = g->TL.ntiles + 1;
            const int rmin = g->sweep_rounds_min < g->sweep_rounds_max ? g->sweep_rounds_min : g->sweep_rounds_max;
            for (int r = 0; r < g->sweep_rounds_max; ++r) {
                // the first rounds run without the 5 B/voxel fixed-point check: nobody would act on its verdict
                const bool check = r + 1 >= rmin;
                rc = relabel_sweep_round(g, &pending, check);
                if (rc) return rc;
                if (!check) continue;
                if (pending <= g->TL.ntiles / g->sweep_done_frac) break;
                if ((long long)pending * 4 > (long long)prev * 3) break;      // a round that clears < 25 %: the rest is local detail
                prev = pending;
            }
        }
    }
    if (g->coop_bfs_grid > 0 && g->use_tiles) {
        // all passes in one cooperative launch; the list selector lives in the control block (device side), so the
        // host does not have to synchronise unless the caller wants to know whether anything moved
        CK(cudaMemsetAsync(g->d_tcount + CTL_CURSOR, 0, sizeof(int), g->stream));
        int* it0 = g->rl_items[0]; int* it1 = g->rl_items[1];
        if (g->nd == 4) {
            void* args4[] = {&g->L, &g->TL4, &g->S.rmask, &g->S.height, &g->rflag, &it0, &it1, &g->d_tcount};
            CK(cudaLaunchCooperativeKernel((void*)k_bfs_coop4, dim3(g->coop_bfs_grid), dim3(T4_VOX), args4, 0, g->stream));
        } else {
            void* args[] = {&g->L, &g->TL, &g->S.rmask, &g->S.height, &g->rflag, &it0, &it1, &g->d_tcount};
            CK(cudaLaunchCooperativeKernel((void*)k_bfs_coop, dim3(g->coop_bfs_grid), dim3(TILE_VOX), args, 0, g->stream));
        }
        g->st.kernel_launches++;
        g->st.relabel_sweeps++;     // passes are counted on the device (ctl[CTL_RELP]); one launch here
        if (want_any) {
            int relp = 0;
            CK(cudaMemcpyAsync(&relp, g->d_tcount + CTL_RELP, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
            CK(cudaStreamSynchronize(g->stream));
            if (relp != 0) *any = 1;
        }
        return MGC_OK;
    }
    for (;;) {
        const int cur = g->rl_cur;
        int pending = 0;
        int rc = read_tcount(g, cur, &pending);
        if (rc) return rc;
        if (!pending) break;
        *any = 1;
        CK(cudaMemsetAsync(g->d_tcount + (1 - cur), 0, sizeof(int), g->stream));
        CK(cudaMemsetAsync(cursor(g), 0, sizeof(int), g->stream));
        const int grid = pending < g->n_ctas * 2 ? pending : g->n_ctas * 2;   // 4 KB smem: more CTAs per SM fit
        if (g->nd == 4)
            k_relabel_tile4<<<grid, T4_VOX, 0, g->stream>>>(g->L, g->TL4, g->S.rmask, g->S.height, g->rflag, rl(g, cur),
                                                            cursor(g), rl(g, 1 - cur));
        else
        k_relabel_tile<<<grid, TILE_VOX, 0, g->stream>>>(g->L, g->TL, g->S.rmask, g->S.height, g->rflag, rl(g, cur),
                                                         cursor(g), rl(g, 1 - cur));
        g->rl_cur = 1 - cur;
        g->st.kernel_launches++;
        g->st.relabel_sweeps++;
    }
    CK(cudaGetLastError());
    return MGC_OK;
}

int lazy_materialise_list(mgc_graph* g, const WorkList& tiles);

// one colour: consume its current list; still-active tiles go to its alternate list, receivers of cross-face flow
// to the list the other colour consumes next
int push_color(mgc_graph* g, int color)
{
    g->flow_started = true;
    const int a = g->pl_sel[color], oa = g->pl_sel[1 - color];
    if (g->lazy && g->nd == 3) {          // every block the listed tiles can write into holds its capacity planes
        int rc = lazy_materialise_list(g, pl(g, color, a));
        if (rc) return rc;
    }
    CK(cudaMemsetAsync(cursor(g), 0, sizeof(int), g->stream));
    if (g->nd == 4) {
        k_push_tile4<double><<<g->n_ctas, T4_VOX, 0, g->stream>>>(g->L, g->TL4, g->S, g->smask, g->iters_now, g->pflag, pl(g, color, a),
                                                                  cursor(g), pl(g, color, 1 - a), pl(g, 1 - color, oa));
    } else if (g->use_tma) {
        const size_t smem = 2 * TMA_STAGE_BYTES + 6 * TILE_VOX * sizeof(double) + 1024 * sizeof(int) + 64;
        k_push_tile_tma<double><<<g->n_ctas, TILE_VOX, smem, g->stream>>>(g->L, g->TL, g->S, g->maps, g->iters_now, g->pflag,
                                                                          pl(g, color, a), cursor(g), pl(g, color, 1 - a),
                                                                          pl(g, 1 - color, oa));
    } else
    k_push_tile<double><<<g->n_ctas, TILE_VOX, 0, g->stream>>>(g->L, g->TL, g->S, g->iters_now, g->pflag, pl(g, color, a),
                                                               cursor(g), pl(g, color, 1 - a), pl(g, 1 - color, oa));
    CK(cudaMemsetAsync(g->d_tcount + 2 + color * 2 + a, 0, sizeof(int), g->stream));   // consumed list is empty again
    g->pl_sel[color] = 1 - a;
    g->st.kernel_launches++;
    return MGC_OK;
}

int push_tiles(mgc_graph* g, int passes)
{
    Nvtx range("mgc:push_passes");
    cudaEventRecord(g->ev[2], g->stream);
    for (int p = 0; p < passes; ++p) {
        int rc = push_color(g, 0);
        if (rc) return rc;
        rc = push_color(g, 1);
        if (rc) return rc;
    }
    g->st.push_sweeps += passes;
    CK(cudaGetLastError());
    if (g->slab) return MGC_OK;      // slabs are stepped asynchronously: no per-call timing synchronisation
    cudaEventRecord(g->ev[3], g->stream);
    CK(cudaEventSynchronize(g->ev[3]));
    { float ms = 0; cudaEventElapsedTime(&ms, g->ev[2], g->ev[3]); g->st.ms_push += ms; }
    return MGC_OK;
}

// active voxels, counted exactly over the two pending push lists (a superset of the tiles that can hold one)
int count_active_tiles_enqueue(mgc_graph* g, unsigned long long* dst)
{
    CK(cudaMemsetAsync(dst, 0, sizeof(unsigned long long), g->stream));
    if (g->nd == 4) {
        for (int color = 0; color < 2; ++color)
            k_count_active_tiles4<double><<<g->n_ctas * 2, T4_VOX, 0, g->stream>>>(g->L, g->TL4, g->S, pl(g, color, g->pl_sel[color]), dst);
        g->st.kernel_launches += 2;
    } else {
        k_count_active_tiles2<double><<<g->n_ctas * 2, TILE_VOX, 0, g->stream>>>(g->L, g->TL, g->S, pl(g, 0, g->pl_sel[0]), pl(g, 1, g->pl_sel[1]), dst);
        g->st.kernel_launches++;
    }
    CK(cudaGetLastError());
    return MGC_OK;
}

int count_active_tiles(mgc_graph* g, int64_t* out)
{
    int rc = count_active_tiles_enqueue(g, g->d_count);
    if (rc) return rc;
    unsigned long long c = 0;
    CK(cudaMemcpyAsync(&c, g->d_count, sizeof(c), cudaMemcpyDeviceToHost, g->stream));
    CK(cudaStreamSynchronize(g->stream));
    *out = (int64_t)c;
    g->st.active_last = (int64_t)c;
    return MGC_OK;
}

// One cooperative launch running the phases selected by `flags` (gc_persist.cuh); the host mirrors of the list
// selectors and the statistics are refreshed from the control block afterwards.
int solve_coop(mgc_graph* g, int flags, int passes, int64_t* active_out)
{
    if (flags & (SOLVE_F_PUSH | SOLVE_F_LOOP)) g->flow_started = true;
    int hdr[4] = {0, g->pl_sel[0], g->pl_sel[1], g->rl_cur};     // cursor, list selectors
    CK(cudaMemcpyAsync(g->d_tcount + CTL_CURSOR, hdr, sizeof(hdr), cudaMemcpyHostToDevice, g->stream));
    SolveLists SL;
    SL.rl_items[0] = g->rl_items[0]; SL.rl_items[1] = g->rl_items[1];
    for (int c = 0; c < 2; ++c) for (int b = 0; b < 2; ++b) SL.pl_items[c][b] = g->pl_items[c][b];
    unsigned long long* active = g->d_count;
    unsigned long long* timers = g->d_count + 1;
    int iters = g->tile_iters, pmax = g->passes_max, mr = (int)(g->max_rounds > 0x7fffffff ? 0x7fffffff : g->max_rounds);
    void* args[] = {&g->L, &g->TL, &g->S, &SL, &g->rflag, &g->pflag, &g->d_tcount, &active, &timers,
                    &flags, &iters, &passes, &pmax, &mr};
    CK(cudaLaunchCooperativeKernel((void*)k_solve_coop<double>, dim3(g->coop_grid), dim3(TILE_VOX), args, 0, g->stream));
    g->st.kernel_launches++;
    int ctl[20];
    unsigned long long cnt[3];
    CK(cudaMemcpyAsync(ctl, g->d_tcount, sizeof(ctl), cudaMemcpyDeviceToHost, g->stream));
    CK(cudaMemcpyAsync(cnt, g->d_count, sizeof(cnt), cudaMemcpyDeviceToHost, g->stream));
    CK(cudaStreamSynchronize(g->stream));
    g->pl_sel[0] = ctl[CTL_SEL0]; g->pl_sel[1] = ctl[CTL_SEL0 + 1]; g->rl_cur = ctl[CTL_RLCUR];
    g->st.push_sweeps += ctl[CTL_PUSHP];
    g->st.relabel_sweeps += ctl[CTL_RELP];
    g->st.global_relabels += ctl[CTL_GREL];
    g->st.ms_relabel += 1e-6 * (double)cnt[1];
    g->st.ms_push += 1e-6 * (double)cnt[2];
    if (flags & (SOLVE_F_COUNT | SOLVE_F_LOOP)) { g->st.active_last = (int64_t)cnt[0]; if (active_out) *active_out = (int64_t)cnt[0]; }
    if (ctl[CTL_STATUS] != 0) FAIL(MGC_E_NOCONV, "push-relabel did not converge within the round cap");
    return MGC_OK;
}

// MEDPY_GC_DEBUG=1: device-side invariants; `after` = compare flow conservation with the excess recorded before the solve
int debug_invariants(mgc_graph* g, bool after)
{
    if (!g->debug_checks) return MGC_OK;
    double* d = g->d_scalars + 4;        // [4] excess, [5] absorbed, [6] violations
    CK(cudaMemsetAsync(d, 0, 3 * sizeof(double), g->stream));
    const bool tiles3 = g->use_tiles && g->nd == 3;
    if (g->nd == 3) {
        if (tiles3) k_debug_invariants<3, double, true><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S, d);
        else        k_debug_invariants<3, double, false><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S, d);
    } else {
        k_debug_invariants<4, double, false><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S, d);
    }
    double h[3] = {0, 0, 0};
    CK(cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, g->stream));
    CK(cudaStreamSynchronize(g->stream));
    if (h[2] != 0.0) {
        g->err = "debug check: " + std::to_string((long long)h[2]) + " invariant violation(s) (negative capacity / excess, absorbed flow out of range or stale residual mask)";
        return MGC_E_STATE;
    }
    if (!after) { g->debug_excess0 = h[0] + h[1]; return MGC_OK; }
    const double scale = fabs(g->debug_excess0) > 1.0 ? fabs(g->debug_excess0) : 1.0;
    if (!g->slab && !(fabs(h[0] + h[1] - g->debug_excess0) <= 1e-9 * scale)) {
        char buf[200];
        snprintf(buf, sizeof(buf), "debug check: flow not conserved: excess %.17g + absorbed %.17g != initial %.17g", h[0], h[1], g->debug_excess0);
        g->err = buf;
        return MGC_E_STATE;
    }
    return MGC_OK;
}

int solve_tiles(mgc_graph* g)
{
    int rc = materialise_zeros(g);
    if (rc) return rc;
    if (!g->state_init) {
        rc = init_tiles(g);
        if (rc) return rc;
    }
    if (g->use_coop && g->nd == 3) {
        const int flags = SOLVE_F_LOOP | (g->labels_fresh ? 0 : SOLVE_F_RESET);
        g->labels_fresh = false;
        return solve_coop(g, flags, g->passes0, nullptr);
    }
    // One host synchronisation per round: relabel (reset + BFS), stop test and the previous round's push passes are all
    // enqueued back to back; the host waits once, reads the active count and the CUDA-event times of both phases and
    // decides.  The stop test of the FIRST round is skipped (a graph that was just built almost always has active
    // voxels; if it has none the push pass is a no-op and the next round's test ends the solve).
    int passes = g->passes0;
    int64_t rounds = 0;
    bool push_open = false;
    int passes_done = 0;
    unsigned long long active_fallback = 0;
    unsigned long long* h_active = g->h_bad ? (unsigned long long*)g->h_bad + 1 : &active_fallback;      // pinned
    for (;;) {
        cudaEventRecord(g->ev[2], g->stream);
        {
            Nvtx range("mgc:global_relabel");
            rc = relabel_tiles_begin(g);
            if (rc) return rc;
            int any = 0;
            rc = relabel_tiles_run(g, &any, false);
            if (rc) return rc;
        }
        cudaEventRecord(g->ev[3], g->stream);
        g->st.global_relabels++;
        const bool test = rounds > 0 || !g->skip_first_test;
        if (test) {
            rc = count_active_tiles_enqueue(g, g->d_count);
            if (rc) return rc;
            CK(cudaMemcpyAsync(h_active, g->d_count, sizeof(unsigned long long), cudaMemcpyDeviceToHost, g->stream));
        }
        CK(cudaEventSynchronize(g->ev[3]));
        if (test) CK(cudaStreamSynchronize(g->stream));
        float ms = 0;
        if (g->init_timed) {          // k_init_tile of the per-term path: its events are reused for the push spans below
            if (cudaEventElapsedTime(&ms, g->ev[4], g->ev[5]) == cudaSuccess) g->st.ms_init = ms;
            g->init_timed = false;
        }
        cudaEventElapsedTime(&ms, g->ev[2], g->ev[3]);
        const double t_rel = ms;
        g->st.ms_relabel += ms;
        double t_pass = 0.0;
        if (push_open) {
            cudaEventElapsedTime(&ms, g->ev[4], g->ev[5]);
            g->st.ms_push += ms;
            t_pass = ms / (passes_done > 0 ? passes_done : 1);
            push_open = false;
            // next round: at most double, and no more push time than one global relabel costs (measured, not guessed):
            // easy instances keep relabelling often, hard ones (long BFS, cheap passes) push longer between relabels
            int want = t_pass > 1e-4 ? (int)(t_rel / t_pass + 0.999) : passes * 2;
            if (want < 1) want = 1;
            if (want > passes * 2) want = passes * 2;
            passes = want > g->passes_max ? g->passes_max : want;
        }
        if (test) {
            g->st.active_last = (int64_t)*h_active;
            if (*h_active == 0ull) break;
        }
        if (++rounds > g->max_rounds) FAIL(MGC_E_NOCONV, "push-relabel did not converge within the round cap");
        g->iters_now = rounds == 1 ? g->tile_iters_first : g->tile_iters;
        {
            Nvtx range("mgc:push_passes");
            cudaEventRecord(g->ev[4], g->stream);
            for (int p = 0; p < passes; ++p) {
                rc = push_color(g, 0);
                if (rc) return rc;
                rc = push_color(g, 1);
                if (rc) return rc;
            }
            cudaEventRecord(g->ev[5], g->stream);
            g->st.push_sweeps += passes;
            passes_done = passes;
            push_open = true;
            CK(cudaGetLastError());
        }
    }
    g->init_timed = false;       // ev[4..5] were reused for the push spans
    return MGC_OK;
}

int readout(mgc_graph* g, double* energy_part)
{
    Nvtx range("mgc:readout");
    if (g->use_tiles && g->nd == 3) k_readout<double, true><<<rblocks(g), 256, 0, g->stream>>>(g->L, g->S, g->mask_dev, g->partials);
    else                            k_readout<double, false><<<rblocks(g), 256, 0, g->stream>>>(g->L, g->S, g->mask_dev, g->partials);
    CK(cudaMemsetAsync(g->d_scalars + 1, 0, sizeof(double), g->stream));
    k_sum_partials<<<1, 256, 0, g->stream>>>(g->partials, rblocks(g), g->d_scalars + 1);
    g->st.kernel_launches += 2;
    double sc[2] = {0, 0};
    CK(cudaMemcpyAsync(sc, g->d_scalars, sizeof(sc), cudaMemcpyDeviceToHost, g->stream));
    int mat = 0;
    if (g->lazy_blocks) CK(cudaMemcpyAsync(&mat, g->d_lazy, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
    CK(cudaStreamSynchronize(g->stream));
    g->lazy_materialised = mat;
    g->st.flow_const = sc[0];
    *energy_part = sc[0] + sc[1];
    if (g->init_timed) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, g->ev[4], g->ev[5]) == cudaSuccess) g->st.ms_init = ms;
        g->init_timed = false;
    }
    return MGC_OK;
}

// ---- NCCL, bound at run time ------------------------------------------------------------------------------
// The library does not link libnccl: the first mgc_slab_comm_* call binds the copy that is already loaded in the
// process (torch's, when the host side is Python) or opens libnccl.so.2 itself.
struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*CommAbort)(ncclComm_t) = nullptr;
    ncclResult_t (*CommGetAsyncError)(ncclComm_t, ncclResult_t*) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    bool ok = false;
};

NcclApi& nccl_api()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return;
        bool all = true;
        auto bind = [&](auto& fn, const char* name) { fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(h, name)); if (!fn) all = false; };
        bind(api.GetUniqueId, "ncclGetUniqueId"); bind(api.CommInitRank, "ncclCommInitRank"); bind(api.CommDestroy, "ncclCommDestroy");
        bind(api.CommAbort, "ncclCommAbort"); bind(api.CommGetAsyncError, "ncclCommGetAsyncError"); bind(api.GetErrorString, "ncclGetErrorString");
        bind(api.AllReduce, "ncclAllReduce"); bind(api.Send, "ncclSend"); bind(api.Recv, "ncclRecv");
        bind(api.GroupStart, "ncclGroupStart"); bind(api.GroupEnd, "ncclGroupEnd");
        api.ok = all;
    });
    return api;
}

#define NK(call)                                                                                   \
    do {                                                                                           \
        ncclResult_t _r = (call);                                                                  \
        if (_r != ncclSuccess) {                                                                   \
            g->err = std::string(#call) + ": " + nccl_api().GetErrorString(_r);                    \
            return MGC_E_CUDA;                                                                     \
        }                                                                                          \
    } while (0)

void slab_comm_release(mgc_graph* g)
{
    if (g->comm && nccl_api().ok) nccl_api().CommDestroy(g->comm);
    g->comm = nullptr;
}

// asynchronous NCCL errors (a peer that died, a network fault) surface here instead of as a hang: polled at every
// host-visible decision of the slab solve (SURVEY.md §5.3)
int slab_comm_poll(mgc_graph* g)
{
    if (!g->comm) return MGC_OK;
    ncclResult_t async = ncclSuccess;
    NK(nccl_api().CommGetAsyncError(g->comm, &async));
    if (async != ncclSuccess && async != ncclInProgress) {
        g->err = std::string("NCCL asynchronous error: ") + nccl_api().GetErrorString(async);
        nccl_api().CommAbort(g->comm);
        g->comm = nullptr;
        return MGC_E_CUDA;
    }
    return MGC_OK;
}

// phase spans of the slab solve: begin / end record an event pair on the stream; resolved once the solve is over
void phase_begin(mgc_graph* g, int kind)
{
    if (g->ph_used + 2 > g->ph_events.size()) { g->ph_events.resize(g->ph_used + 2, nullptr); }
    for (int i = 0; i < 2; ++i) if (!g->ph_events[g->ph_used + i]) cudaEventCreate(&g->ph_events[g->ph_used + i]);
    cudaEventRecord(g->ph_events[g->ph_used], g->stream);
    g->ph_kind.push_back(kind);
}
void phase_end(mgc_graph* g)
{
    cudaEventRecord(g->ph_events[g->ph_used + 1], g->stream);
    g->ph_used += 2;
}
void phase_resolve(mgc_graph* g)
{
    for (size_t i = 0; i + 1 < g->ph_used; i += 2) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, g->ph_events[i], g->ph_events[i + 1]) == cudaSuccess) g->slab_phase_ms[g->ph_kind[i / 2]] += ms;
    }
    g->ph_used = 0;
    g->ph_kind.clear();
}

// one border exchange: pack -> grouped send/recv with both neighbours -> unpack, all enqueued on the handle's stream
int slab_exchange(mgc_graph* g, long long* changed_dev, bool labels_only)
{
    Nvtx range("mgc:slab_exchange");
    phase_begin(g, 1);
    NcclApi& N = nccl_api();
    const unsigned P = g->L.plane;
    const unsigned nb = (P + 255u) / 256u;
    int32_t* h_send[2] = {(int32_t*)g->msg[0], (int32_t*)g->msg[1]};
    double* f_send[2] = {(double*)(g->msg[0] + g->msg_h_bytes), (double*)(g->msg[1] + g->msg_h_bytes)};
    const bool have[2] = {g->ghost_lo, g->ghost_hi};
    for (int side = 0; side < 2; ++side) {
        if (!have[side]) continue;
        const size_t border = side == 0 ? (size_t)g->L.own0 * P : (size_t)(g->L.own1 - 1) * P;
        const size_t ghost = side == 0 ? border - P : border + P;
        k_slab_pack<double><<<nb, 256, 0, g->stream>>>(P, g->S.height + border, g->S.excess + ghost, h_send[side], labels_only ? nullptr : f_send[side]);
        g->st.kernel_launches++;
    }
    CK(cudaGetLastError());
    // relabel rounds exchange labels only (4 B per border voxel); push exchanges add the parked flow (12 B per border voxel)
    const size_t bytes = labels_only ? g->msg_h_bytes : g->msg_bytes;
    if (g->comm_world > 1) {
        NK(N.GroupStart());
        if (have[0]) { NK(N.Send(g->msg[0], bytes, ncclUint8, g->comm_rank - 1, g->comm, g->stream)); NK(N.Recv(g->msg[2], bytes, ncclUint8, g->comm_rank - 1, g->comm, g->stream)); }
        if (have[1]) { NK(N.Send(g->msg[1], bytes, ncclUint8, g->comm_rank + 1, g->comm, g->stream)); NK(N.Recv(g->msg[3], bytes, ncclUint8, g->comm_rank + 1, g->comm, g->stream)); }
        NK(N.GroupEnd());
    }
    const int32_t* h_lo = have[0] ? (const int32_t*)g->msg[2] : nullptr;
    const double* f_lo = (have[0] && !labels_only) ? (const double*)(g->msg[2] + g->msg_h_bytes) : nullptr;
    const int32_t* h_hi = have[1] ? (const int32_t*)g->msg[3] : nullptr;
    const double* f_hi = (have[1] && !labels_only) ? (const double*)(g->msg[3] + g->msg_h_bytes) : nullptr;
    g->slab_exchanges++;
    const int rc_unpack = mgc_slab_unpack(g, h_lo, f_lo, h_hi, f_hi, (int32_t*)changed_dev);
    phase_end(g);
    return rc_unpack;
}

// ---- fused graph build (gc_build.cuh) ------------------------------------------------------------------
// rank-3 tensor map of the image with the 10 x 10 x BUILD_BX halo box; false when the 16-byte rules are not met
bool make_image_map(mgc_graph* g, const void* img, int dtype, CUtensorMap* out)
{
    tmap_encode_fn encode = tensor_map_encoder();
    if (!encode) return false;
    const size_t es = dtype_size(dtype);
    const cuuint64_t X = (cuuint64_t)g->L.dim[2], Y = (cuuint64_t)g->L.dim[1], Z = (cuuint64_t)g->L.dim[0];
    if ((X * es) % 16 || ((uintptr_t)img & 15)) return false;
    CUtensorMapDataType dt;
    switch (dtype) {
        case MGC_F32: dt = CU_TENSOR_MAP_DATA_TYPE_FLOAT32; break;
        case MGC_F64: dt = CU_TENSOR_MAP_DATA_TYPE_FLOAT64; break;
        case MGC_U8: dt = CU_TENSOR_MAP_DATA_TYPE_UINT8; break;
        case MGC_I16: dt = CU_TENSOR_MAP_DATA_TYPE_UINT16; break;     // moved as raw 2-byte words
        default: dt = CU_TENSOR_MAP_DATA_TYPE_INT32; break;
    }
    const cuuint64_t dims[3] = {X, Y, Z};
    const cuuint64_t strides[2] = {X * es, X * Y * es};
    cuuint32_t bx = 0;
    switch (dtype) {
        case MGC_F32: bx = BuildBox<float>::BX; break;
        case MGC_F64: bx = BuildBox<double>::BX; break;
        case MGC_U8: bx = BuildBox<uint8_t>::BX; break;
        case MGC_I16: bx = BuildBox<int16_t>::BX; break;
        default: bx = BuildBox<int32_t>::BX; break;
    }
    const cuuint32_t box[3] = {bx, BUILD_HY, BUILD_HZ};
    const cuuint32_t estr[3] = {1, 1, 1};
    return encode(out, dt, 3, const_cast<void*>(img), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// rank-3 tensor map of a C-contiguous array over the local lattice with an 8 x 8 x 32 box (probability map, marker bytes)
bool make_block_map(mgc_graph* g, const void* ptr, int dtype, CUtensorMap* out)
{
    tmap_encode_fn encode = tensor_map_encoder();
    if (!encode || !ptr) return false;
    const size_t es = dtype_size(dtype);
    const cuuint64_t X = (cuuint64_t)g->L.dim[2], Y = (cuuint64_t)g->L.dim[1], Z = (cuuint64_t)g->L.dim[0];
    if ((X * es) % 16 || ((uintptr_t)ptr & 15)) return false;
    const CUtensorMapDataType dt = dtype == MGC_F64 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : (dtype == MGC_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT8);
    const cuuint64_t dims[3] = {X, Y, Z};
    const cuuint64_t strides[2] = {X * es, X * Y * es};
    const cuuint32_t box[3] = {BUILD_TX, BUILD_TY, BUILD_TZ};
    const cuuint32_t estr[3] = {1, 1, 1};
    return encode(out, dt, 3, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <typename E, int FN, int USE_MAX, int SPACING, int TIN = 0, int MODE = 0>
int build_launch_inst(mgc_graph* g, const BuildMaps& imap, const BuildArgs& A, const BoundaryParams& P, int nz_layers)
{
    auto kern = k_build_tile<E, double, FN, USE_MAX, SPACING, TIN, MODE>;
    const size_t smem = build_smem_bytes<E>();
    static bool attr_done = false;       // per instantiation
    if (!attr_done) { cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr_done = true; }
    const dim3 grid((unsigned)((g->L.dim[2] + BUILD_TX - 1) / BUILD_TX), (unsigned)((g->L.dim[1] + BUILD_TY - 1) / BUILD_TY), (unsigned)nz_layers);
    kern<<<grid, BUILD_THREADS, smem, g->stream>>>(g->L, g->TL, g->S, imap, A, P, g->d_flags, g->partials, g->rflag, rl(g, 0), g->pflag,
                                                     pl(g, 0, 0), pl(g, 1, 0), g->bflag, g->d_lazy);
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    return MGC_OK;
}

template <typename E>
int build_launch(mgc_graph* g, const BuildMaps& imap, const BuildArgs& A, const BoundaryParams& P, int nz_layers)
{
    if constexpr (!std::is_integral<E>::value) {
        if (P.fn == 1 && P.inv_spacing_on == 0.0) {
            if constexpr (std::is_same<E, float>::value) {
                // float32 image + float32 probability map + byte markers, everything staged by TMA: the compile-time variant
                const bool fast = A.use_tma && A.prob && !A.prob_f64 && A.compute_f32 && A.tma_prob && A.tma_mark == 3 &&
                                  !A.fg_bits && !A.bg_bits && A.dbg == 0;
                if (fast && g->lazy) {
                    if (P.use_max) return build_launch_inst<E, 1, 1, 0, 1, 1>(g, imap, A, P, nz_layers);
                    return build_launch_inst<E, 1, 0, 0, 1, 1>(g, imap, A, P, nz_layers);
                }
                if (fast) {
                    if (P.use_max) return build_launch_inst<E, 1, 1, 0, 1>(g, imap, A, P, nz_layers);
                    return build_launch_inst<E, 1, 0, 0, 1>(g, imap, A, P, nz_layers);
                }
            }
            if (g->lazy) FAIL(MGC_E_STATE, "internal: lazy build without its kernel variant");
            if (P.use_max) return build_launch_inst<E, 1, 1, 0>(g, imap, A, P, nz_layers);
            return build_launch_inst<E, 1, 0, 0>(g, imap, A, P, nz_layers);
        }
    }
    if (g->lazy) FAIL(MGC_E_STATE, "internal: lazy build without its kernel variant");
    return build_launch_inst<E, -1, -1, -1>(g, imap, A, P, nz_layers);
}

// the variant a lazy build runs (build_launch: float32 image, exponential term without spacing, staged t-link inputs)
bool lazy_variant(const BuildArgs& A, const BoundaryParams& P, int img_dtype)
{
    return img_dtype == MGC_F32 && P.fn == 1 && P.inv_spacing_on == 0.0 && A.use_tma && A.prob && !A.prob_f64 &&
           A.compute_f32 && A.tma_prob && A.tma_mark == 3 && !A.fg_bits && !A.bg_bits && A.dbg == 0;
}

template <int USE_MAX>
int lazy_list_inst(mgc_graph* g, const WorkList& tiles)
{
    auto kern = k_build_materialise<float, double, 1, USE_MAX, 0>;
    const size_t smem = build_smem_bytes<float>();
    static bool attr_done = false;
    if (!attr_done) { cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr_done = true; }
    kern<<<g->n_ctas * 2, BUILD_THREADS, smem, g->stream>>>(g->L, g->TL, g->S, g->lazy_maps, g->lazy_args, g->lazy_P, tiles,
                                                           g->bflag, g->d_lazy);
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    return MGC_OK;
}

int lazy_materialise_list(mgc_graph* g, const WorkList& tiles)
{
    return g->lazy_P.use_max ? lazy_list_inst<1>(g, tiles) : lazy_list_inst<0>(g, tiles);
}

template <int USE_MAX>
int lazy_all_inst(mgc_graph* g)
{
    auto kern = k_build_materialise_all<float, double, 1, USE_MAX, 0>;
    const size_t smem = build_smem_bytes<float>();
    static bool attr_done = false;
    if (!attr_done) { cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr_done = true; }
    const dim3 grid((unsigned)((g->L.dim[2] + BUILD_TX - 1) / BUILD_TX), (unsigned)((g->L.dim[1] + BUILD_TY - 1) / BUILD_TY),
                    (unsigned)((g->L.dim[0] + BUILD_TZ - 1) / BUILD_TZ));
    kern<<<grid, BUILD_THREADS, smem, g->stream>>>(g->L, g->TL, g->S, g->lazy_maps, g->lazy_args, g->lazy_P, g->bflag, g->d_lazy);
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    return MGC_OK;
}

// Every reader of cap / tr / excess outside the tile push passes (get_edge / get_trcap, further terms, the debug
// checks, the cooperative and per-voxel solvers) sees the whole lattice: materialise what is still cold, stream-ordered,
// and let the next upload into a staging slot wait for it.
int lazy_materialise_all(mgc_graph* g)
{
    if (!g->lazy) return MGC_OK;
    const int rc = g->lazy_P.use_max ? lazy_all_inst<1>(g) : lazy_all_inst<0>(g);
    if (rc) return rc;
    slots_release(g, 0x17u);
    g->lazy = false;
    return MGC_OK;
}

int build_launch_dtype(mgc_graph* g, int dtype, const BuildMaps& imap, const BuildArgs& A, const BoundaryParams& P, int nz_layers)
{
    switch (dtype) {
        case MGC_F32: return build_launch<float>(g, imap, A, P, nz_layers);
        case MGC_F64: return build_launch<double>(g, imap, A, P, nz_layers);
        case MGC_U8: return build_launch<uint8_t>(g, imap, A, P, nz_layers);
        case MGC_I16: return build_launch<int16_t>(g, imap, A, P, nz_layers);
        default: return build_launch<int32_t>(g, imap, A, P, nz_layers);
    }
}

// C-contiguous over the local lattice?
bool c_contiguous(const mgc_graph* g, const mgc_array* a)
{
    long long expect = (long long)dtype_size(a->dtype);
    for (int d = g->nd - 1; d >= 0; --d) {
        const int ud = d - g->shift;
        if (g->L.dim[d] > 1) {
            if (ud < 0 || (long long)a->strides[ud] != expect) return false;
        }
        expect *= g->L.dim[d];
    }
    return true;
}

bool can_fuse(const mgc_graph* g) { return g->use_tiles && g->nd == 3 && g->fuse_build; }

}  // namespace

template <typename E, int ND>
static cudaError_t gradient_launch(const int64_t* shape, const E* img, float* out, long long n)
{
    GradCtx<ND> G;
    long long st = 1;
    for (int d = ND - 1; d >= 0; --d) { G.dim[d] = (int)shape[d]; G.stride[d] = st; st *= shape[d]; }
    k_gradient_magnitude<E, ND><<<(unsigned)((n + 255) / 256), 256>>>(G, n, img, out);
    return cudaGetLastError();
}

template <typename E>
static cudaError_t gradient_dispatch(int nd, const int64_t* shape, const E* img, float* out, long long n)
{
    switch (nd) {
        case 1: return gradient_launch<E, 1>(shape, img, out, n);
        case 2: return gradient_launch<E, 2>(shape, img, out, n);
        case 3: return gradient_launch<E, 3>(shape, img, out, n);
        default: return gradient_launch<E, 4>(shape, img, out, n);
    }
}


// =====================================================================================================
// C ABI
// =====================================================================================================
extern "C" {

int mgc_abi_version(void) { return MGC_ABI_VERSION; }

const char* mgc_last_error(const mgc_graph* g) { return g ? g->err.c_str() : g_create_error.c_str(); }

int mgc_create(int32_t ndim, const int64_t* shape, int32_t device, mgc_graph** out)
{
    return create_impl(ndim, shape, 0, 0, false, device, out);
}

int mgc_create_slab(int32_t ndim, const int64_t* shape, int64_t z0, int64_t z1, int32_t device, mgc_graph** out)
{
    if (ndim < 3) { g_create_error = "z-slab handles need ndim >= 3"; return MGC_E_ARG; }
    return create_impl(ndim, shape, z0, z1, true, device, out);
}

void mgc_destroy(mgc_graph* g)
{
    if (!g) return;
    cudaSetDevice(g->device);
    if (g->stream) cudaStreamSynchronize(g->stream);
    for (auto& b : g->owned_bufs) pool_free(g->device, b.bytes, b.p);
    for (auto& b : g->scratch) if (b.p) pool_free(g->device, b.bytes, b.p);
    if (g->raw.p) pool_free(g->device, g->raw.bytes, g->raw.p);
    for (auto& ev : g->ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : g->ev_slot) if (ev) cudaEventDestroy(ev);
    for (auto& ev : g->ev_terms) if (ev) cudaEventDestroy(ev);
    for (auto& ev : g->ev_chunk) if (ev) cudaEventDestroy(ev);
    if (g->ev_up) cudaEventDestroy(g->ev_up);
    if (g->ev_bad) cudaEventDestroy(g->ev_bad);
    for (auto& ev : g->ev_b) if (ev) cudaEventDestroy(ev);
    for (auto& ev : g->ph_events) if (ev) cudaEventDestroy(ev);
    if (g->h_bad) mgc_host_free(g->h_bad);
    if (g->h_stat) mgc_host_free(g->h_stat);
    slab_comm_release(g);
    if (g->up_stream) { cudaStreamSynchronize(g->up_stream); cudaStreamDestroy(g->up_stream); }
    if (g->own_stream && g->stream) cudaStreamDestroy(g->stream);
    delete g;
}

int mgc_reset(mgc_graph* g)
{
    if (!g) return MGC_E_ARG;
    CK(cudaSetDevice(g->device));
    // no memset of the big arrays: the first n-link / t-link term overwrites them (FRESH kernels)
    g->caps_fresh = true;
    g->tr_fresh = true;
    CK(cudaMemsetAsync(g->d_scalars, 0, 64, g->stream));
    CK(cudaMemsetAsync(g->d_flags, 0, 64, g->stream));
    invalidate(g);
    g->flow_started = false;
    g->has_nlinks = false;
    g->energy = 0.0;
    int64_t n = g->st.n_voxels;
    g->st = mgc_stats{};
    g->st.n_voxels = n;
    g->terms_open = false;
    g->bad_pending = false;
    g->lazy = false;
    g->lazy_blocks = g->lazy_materialised = 0;
    return MGC_OK;
}

int mgc_gradient_magnitude_prewitt(int32_t ndim, const int64_t* shape, const mgc_array* image, float* out,
                                   int32_t out_mem, int32_t device)
{
    if (ndim < 1 || ndim > 4 || !shape || !image || !image->data || !out) { g_create_error = "bad arguments"; return MGC_E_ARG; }
    const size_t es = dtype_size(image->dtype);
    if (!es) { g_create_error = "unsupported dtype"; return MGC_E_ARG; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        g_create_error = "no usable CUDA device (this library has no CPU path)";
        return MGC_E_CUDA;
    }
    if (device < 0) cudaGetDevice(&device);
    cudaSetDevice(device);
    long long n = 1;
    bool contiguous = true;
    long long expect = (long long)es;
    for (int d = ndim - 1; d >= 0; --d) {
        if (shape[d] < 1) { g_create_error = "extents must be >= 1"; return MGC_E_ARG; }
        if (shape[d] > 1 && image->strides[d] != expect) contiguous = false;
        expect *= shape[d];
        n *= shape[d];
    }
    if (!contiguous) { g_create_error = "gradient input must be C-contiguous (the host layer copies otherwise)"; return MGC_E_ARG; }
    void* d_in = nullptr;
    void* d_out = nullptr;
    const size_t in_bytes = (size_t)n * es, out_bytes = (size_t)n * sizeof(float);
    cudaError_t e = cudaSuccess;
    if (image->mem == MGC_MEM_HOST) {
        if ((e = pool_alloc(device, in_bytes, &d_in)) != cudaSuccess) { cudaGetLastError(); g_create_error = "device allocation failed"; return MGC_E_NOMEM; }
        e = cudaMemcpy(d_in, image->data, in_bytes, cudaMemcpyHostToDevice);
    }
    const void* src = image->mem == MGC_MEM_HOST ? d_in : image->data;
    float* dst = out;
    if (e == cudaSuccess && out_mem == MGC_MEM_HOST) {
        if ((e = pool_alloc(device, out_bytes, &d_out)) == cudaSuccess) dst = (float*)d_out;
    }
    if (e == cudaSuccess) {
        switch (image->dtype) {
            case MGC_F32: e = gradient_dispatch<float>(ndim, shape, (const float*)src, dst, n); break;
            case MGC_F64: e = gradient_dispatch<double>(ndim, shape, (const double*)src, dst, n); break;
            case MGC_U8: e = gradient_dispatch<uint8_t>(ndim, shape, (const uint8_t*)src, dst, n); break;
            case MGC_I16: e = gradient_dispatch<int16_t>(ndim, shape, (const int16_t*)src, dst, n); break;
            default: e = gradient_dispatch<int32_t>(ndim, shape, (const int32_t*)src, dst, n); break;
        }
    }
    if (e == cudaSuccess && out_mem == MGC_MEM_HOST) e = cudaMemcpy(out, d_out, out_bytes, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (d_in) pool_free(device, in_bytes, d_in);
    if (d_out) pool_free(device, out_bytes, d_out);
    if (e != cudaSuccess) { cudaGetLastError(); g_create_error = std::string("gradient kernel failed: ") + cudaGetErrorString(e); return MGC_E_CUDA; }
    return MGC_OK;
}

int mgc_host_alloc(size_t bytes, void** out)
{
    if (!out || !bytes) return MGC_E_ARG;
    const size_t rb = round_up(bytes);
    std::lock_guard<std::mutex> lk(g_pool_mu);
    auto it = g_host_pool.find(rb);
    void* p = nullptr;
    if (it != g_host_pool.end() && !it->second.empty()) { p = it->second.back(); it->second.pop_back(); }
    else if (cudaHostAlloc(&p, rb, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); g_create_error = "pinned host allocation failed"; return MGC_E_NOMEM; }
    g_host_live[p] = rb;
    *out = p;
    return MGC_OK;
}

void mgc_host_free(void* p)
{
    if (!p) return;
    std::lock_guard<std::mutex> lk(g_pool_mu);
    auto it = g_host_live.find(p);
    if (it == g_host_live.end()) return;
    g_host_pool[it->second].push_back(p);
    g_host_live.erase(it);
}

// Give cached blocks back to the driver: every device block of the size-keyed pool (all devices) and every pinned host block
// that is not handed out.  Handles that are alive keep what they hold.
int mgc_trim_pools(void)
{
    std::lock_guard<std::mutex> lk(g_pool_mu);
    int cur = 0;
    cudaGetDevice(&cur);
    for (auto& kv : g_pool) {
        if (kv.second.empty()) continue;
        cudaSetDevice(kv.first.first);
        for (void* p : kv.second) cudaFree(p);
        kv.second.clear();
    }
    cudaSetDevice(cur);
    for (auto& kv : g_host_pool) { for (void* p : kv.second) cudaFreeHost(p); kv.second.clear(); }
    cudaGetLastError();
    return MGC_OK;
}

int mgc_set_option(mgc_graph* g, int32_t option, int64_t value)
{
    if (!g) return MGC_E_ARG;
    if (option == MGC_OPT_DEFER_WEIGHT_CHECK) { g->defer_check = value != 0; return MGC_OK; }
    if (option == MGC_OPT_KEEP_INPUTS) { g->keep_inputs = value != 0; return MGC_OK; }
    FAIL(MGC_E_ARG, "unknown option");
}

int mgc_check(mgc_graph* g)
{
    if (!g) return MGC_E_ARG;
    return check_pending(g);
}

int mgc_set_stream(mgc_graph* g, void* cuda_stream)
{
    if (!g) return MGC_E_ARG;
    CK(cudaStreamSynchronize(g->stream));
    if (g->own_stream) { cudaStreamDestroy(g->stream); g->own_stream = false; }
    g->stream = (cudaStream_t)cuda_stream;
    return MGC_OK;
}

int mgc_synchronize(mgc_graph* g)
{
    if (!g) return MGC_E_ARG;
    CK(cudaStreamSynchronize(g->stream));
    return MGC_OK;
}

int mgc_add_regional_probability(mgc_graph* g, const mgc_array* prob, double alpha, int32_t compute_dtype)
{
    if (!g || !prob) return MGC_E_ARG;
    if (g->flow_started) FAIL(MGC_E_STATE, "the graph has been solved (its capacities hold residuals): reset() it before adding terms");
    if (prob->dtype != MGC_F32 && prob->dtype != MGC_F64) FAIL(MGC_E_ARG, "probability map must be float32 or float64");
    if (compute_dtype != MGC_F32 && compute_dtype != MGC_F64) FAIL(MGC_E_ARG, "compute dtype must be float32 or float64");
    CK(cudaSetDevice(g->device));
    { int rcl = lazy_materialise_all(g); if (rcl) return rcl; }
    TermSpan t(g);
    const void* p = nullptr;
    int rc = stage_input(g, prob, 0, &p);
    if (rc) return rc;
    rc = check_pending(g);
    if (rc) return rc;
    if (prob->dtype == MGC_F32 && (g->L.n % 4u) == 0u && ((uintptr_t)p % 16u) == 0u)
        k_regional_f32x4<double><<<rblocks(g), 256, 0, g->stream>>>(g->L, g->S, (const float4*)p, alpha, compute_dtype == MGC_F32, g->tr_fresh ? 1 : 0, g->partials);
    else if (prob->dtype == MGC_F32)
        k_regional<float, double><<<rblocks(g), 256, 0, g->stream>>>(g->L, g->S, (const float*)p, alpha, compute_dtype == MGC_F32, g->tr_fresh ? 1 : 0, g->partials);
    else
        k_regional<double, double><<<rblocks(g), 256, 0, g->stream>>>(g->L, g->S, (const double*)p, alpha, 0, g->tr_fresh ? 1 : 0, g->partials);
    g->tr_fresh = false;
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    rc = finish_flow_const(g);
    if (rc) return rc;
    invalidate(g);
    t.stop(1u);
    return MGC_OK;
}

int mgc_add_tweights_dense(mgc_graph* g, const mgc_array* src, const mgc_array* snk)
{
    if (!g || !src || !snk) return MGC_E_ARG;
    if (g->flow_started) FAIL(MGC_E_STATE, "the graph has been solved (its capacities hold residuals): reset() it before adding terms");
    if (src->dtype != MGC_F64 || snk->dtype != MGC_F64) FAIL(MGC_E_ARG, "dense t-weights must be float64");
    CK(cudaSetDevice(g->device));
    { int rcl = lazy_materialise_all(g); if (rcl) return rcl; }
    TermSpan t(g);
    const void *ps = nullptr, *pk = nullptr;
    int rc = stage_input(g, src, 0, &ps);
    if (rc) return rc;
    rc = stage_input(g, snk, 1, &pk);
    if (rc) return rc;
    rc = check_pending(g);
    if (rc) return rc;
    k_tweights_dense<double><<<rblocks(g), 256, 0, g->stream>>>(g->L, g->S, (const double*)ps, (const double*)pk, g->tr_fresh ? 1 : 0, g->partials);
    g->tr_fresh = false;
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    rc = finish_flow_const(g);
    if (rc) return rc;
    invalidate(g);
    t.stop(3u);
    return MGC_OK;
}

int mgc_add_markers(mgc_graph* g, const mgc_array* fg, const mgc_array* bg)
{
    if (!g) return MGC_E_ARG;
    if (!fg && !bg) return MGC_OK;
    if (g->flow_started) FAIL(MGC_E_STATE, "the graph has been solved (its capacities hold residuals): reset() it before adding terms");
    if ((fg && fg->dtype != MGC_U8) || (bg && bg->dtype != MGC_U8)) FAIL(MGC_E_ARG, "markers must be uint8 / bool");
    CK(cudaSetDevice(g->device));
    { int rcl = lazy_materialise_all(g); if (rcl) return rcl; }
    TermSpan t(g);
    const void *pf = nullptr, *pb = nullptr;
    int rc = MGC_OK;
    if (fg) { rc = stage_input(g, fg, 1, &pf); if (rc) return rc; }
    if (bg) { rc = stage_input(g, bg, 4, &pb); if (rc) return rc; }
    rc = check_pending(g);      // after the uploads: they overlapped the boundary kernel whose verdict this is
    if (rc) return rc;
    const bool vec16 = !g->tr_fresh && (g->L.n % 16u) == 0u && ((uintptr_t)pf % 16u) == 0u && ((uintptr_t)pb % 16u) == 0u;
    if (vec16)
        k_markers16<double><<<rblocks(g), 256, 0, g->stream>>>(g->L, g->S, (const uint4*)pf, (const uint4*)pb, g->partials);
    else
        k_markers<double><<<rblocks(g), 256, 0, g->stream>>>(g->L, g->S, (const uint8_t*)pf, (const uint8_t*)pb, g->tr_fresh ? 1 : 0, g->partials);
    g->tr_fresh = false;
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    rc = finish_flow_const(g);
    if (rc) return rc;
    invalidate(g);
    t.stop(0x12u);
    return MGC_OK;
}

int mgc_add_boundary(mgc_graph* g, int32_t kind, const mgc_array* image, double sigma, const double* spacing, double norm)
{
    if (!g || !image) return MGC_E_ARG;
    if (kind < 0 || kind > 7) FAIL(MGC_E_ARG, "unknown boundary term");
    if (g->flow_started) FAIL(MGC_E_STATE, "the graph has been solved (its capacities hold residuals): reset() it before adding terms");
    CK(cudaSetDevice(g->device));
    { int rcl = lazy_materialise_all(g); if (rcl) return rcl; }
    { int rc0 = check_pending(g); if (rc0) return rc0; }
    TermSpan t(g);
    const void* img = nullptr;
    int rc = stage_input(g, image, 2, &img);
    if (rc) return rc;
    BoundaryParams P{};
    rc = boundary_params(g, kind, image->dtype, img, sigma, spacing, norm, &P);
    if (rc) return rc;
    CK(cudaMemsetAsync(g->d_flags, 0, sizeof(int), g->stream));
    cudaEventRecord(g->ev_b[0], g->stream);
    switch (image->dtype) {
        case MGC_F32: boundary_launch<float>(g, (const float*)img, P); break;
        case MGC_F64: boundary_launch<double>(g, (const double*)img, P); break;
        case MGC_U8: boundary_launch<uint8_t>(g, (const uint8_t*)img, P); break;
        case MGC_I16: boundary_launch<int16_t>(g, (const int16_t*)img, P); break;
        case MGC_I32: boundary_launch<int32_t>(g, (const int32_t*)img, P); break;
    }
    cudaEventRecord(g->ev_b[1], g->stream);
    CK(cudaGetLastError());
    invalidate(g);
    g->has_nlinks = true;
    g->boundary_timed = true;
    if (g->defer_check && g->h_bad && image->mem == MGC_MEM_HOST) {
        // verdict later: the next call's host->device copy overlaps this kernel (see MGC_OPT_DEFER_WEIGHT_CHECK)
        CK(cudaMemcpyAsync(g->h_bad, g->d_flags, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
        CK(cudaEventRecord(g->ev_bad, g->stream));
        g->bad_pending = true;
        t.stop(4u);
        return MGC_OK;
    }
    int bad = 0;
    CK(cudaMemcpyAsync(&bad, g->d_flags, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
    t.stop(4u);
    CK(cudaStreamSynchronize(g->stream));      // the weight check must be reported by this call (ValueError)
    if (bad) FAIL(MGC_E_WEIGHT, "Negative or zero weights are not allowed.");
    return MGC_OK;
}

int mgc_can_fuse(const mgc_graph* g) { return g && can_fuse(g) ? 1 : 0; }

int mgc_build_voxel_graph(mgc_graph* g, const mgc_voxel_terms* t)
{
    if (!g || !t) return MGC_E_ARG;
    if (g->flow_started) FAIL(MGC_E_STATE, "the graph has been solved (its capacities hold residuals): reset() it before adding terms");
    const bool has_bits = t->fg_bits || t->bg_bits;
    if (has_bits && (t->fg || t->bg)) FAIL(MGC_E_ARG, "pass the markers either as byte arrays or bit-packed, not both");
    if (t->boundary_kind > 7) FAIL(MGC_E_ARG, "unknown boundary term");
    if (t->boundary_kind >= 0 && !t->image) FAIL(MGC_E_ARG, "boundary term without image");
    const bool fresh = g->caps_fresh && g->tr_fresh && !g->state_init;
    if (!(fresh && can_fuse(g) && t->boundary_kind >= 0)) {
        // the same terms through the one-pass-per-term entry points, in the reference's order (generate.py:159-172)
        if (has_bits) FAIL(MGC_E_ARG, "bit-packed markers need the fused build (fresh 1-D..3-D tile-solver handle with a boundary term)");
        int rc = MGC_OK;
        if (t->prob) { rc = mgc_add_regional_probability(g, t->prob, t->alpha, t->compute_dtype); if (rc) return rc; }
        if (t->boundary_kind >= 0) { rc = mgc_add_boundary(g, t->boundary_kind, t->image, t->sigma, t->spacing, t->norm); if (rc) return rc; }
        return mgc_add_markers(g, t->fg, t->bg);
    }
    if (t->prob && t->prob->dtype != MGC_F32 && t->prob->dtype != MGC_F64) FAIL(MGC_E_ARG, "probability map must be float32 or float64");
    if (t->prob && t->compute_dtype != MGC_F32 && t->compute_dtype != MGC_F64) FAIL(MGC_E_ARG, "compute dtype must be float32 or float64");
    if (t->prob && t->compute_dtype == MGC_F32 && t->prob->dtype != MGC_F32) FAIL(MGC_E_ARG, "float32 products need a float32 probability map");
    if ((t->fg && t->fg->dtype != MGC_U8) || (t->bg && t->bg->dtype != MGC_U8)) FAIL(MGC_E_ARG, "markers must be uint8 / bool");
    if (!dtype_size(t->image->dtype)) FAIL(MGC_E_ARG, "unsupported dtype");
    CK(cudaSetDevice(g->device));
    { int rc0 = check_pending(g); if (rc0) return rc0; }
    Nvtx range("mgc:build_voxel_graph");
    TermSpan span(g);

    const size_t n = (size_t)g->L.n;
    const size_t plane = (size_t)g->L.plane;
    const int Z = g->L.dim[0];
    const int nzt = (Z + BUILD_TZ - 1) / BUILD_TZ;
    const size_t es_img = dtype_size(t->image->dtype), es_prob = t->prob ? dtype_size(t->prob->dtype) : 0;
    const size_t words = (n + 31) / 32;

    // ---- chunked path: contiguous HOST arrays, upload of z-chunk c+1 overlaps the build of chunk c ----
    bool chunked = g->build_chunks > 1 && nzt >= 2 && t->image->mem == MGC_MEM_HOST && c_contiguous(g, t->image) &&
                   !(( t->boundary_kind & 3) == 0 && std::isnan(t->norm));
    if (t->prob) chunked = chunked && t->prob->mem == MGC_MEM_HOST && c_contiguous(g, t->prob);
    if (t->fg) chunked = chunked && t->fg->mem == MGC_MEM_HOST && c_contiguous(g, t->fg);
    if (t->bg) chunked = chunked && t->bg->mem == MGC_MEM_HOST && c_contiguous(g, t->bg);
    if (has_bits) chunked = chunked && t->bits_mem == MGC_MEM_HOST;

    const void *d_img = nullptr, *d_prob = nullptr, *d_fg = nullptr, *d_bg = nullptr;
    int rc = MGC_OK;
    if (!chunked) {
        rc = stage_input(g, t->image, 2, &d_img); if (rc) return rc;
        if (t->prob) { rc = stage_input(g, t->prob, 0, &d_prob); if (rc) return rc; }
        if (t->fg) { rc = stage_input(g, t->fg, 1, &d_fg); if (rc) return rc; }
        if (t->bg) { rc = stage_input(g, t->bg, 4, &d_bg); if (rc) return rc; }
        if (has_bits) {
            if (t->bits_ready_words && t->bits_mem == MGC_MEM_HOST) {
                while (*t->bits_ready_words < (int64_t)words) std::this_thread::yield();
                std::atomic_thread_fence(std::memory_order_acquire);
            }
            const uint32_t* src[2] = {t->fg_bits, t->bg_bits};
            const void** dst[2] = {&d_fg, &d_bg};
            const int slot[2] = {1, 4};
            for (int i = 0; i < 2; ++i) {
                if (!src[i]) continue;
                if (t->bits_mem == MGC_MEM_DEVICE) { *dst[i] = src[i]; continue; }
                rc = ensure_scratch(g, g->scratch[slot[i]], words * 4); if (rc) return rc;
                rc = upload(g, g->scratch[slot[i]].p, src[i], words * 4, slot[i]); if (rc) return rc;
                *dst[i] = g->scratch[slot[i]].p;
            }
        }
    } else {
        rc = ensure_scratch(g, g->scratch[2], n * es_img); if (rc) return rc;
        if (t->prob) { rc = ensure_scratch(g, g->scratch[0], n * es_prob); if (rc) return rc; }
        if (t->fg || t->fg_bits) { rc = ensure_scratch(g, g->scratch[1], has_bits ? words * 4 : n); if (rc) return rc; }
        if (t->bg || t->bg_bits) { rc = ensure_scratch(g, g->scratch[4], has_bits ? words * 4 : n); if (rc) return rc; }
        d_img = g->scratch[2].p;
        if (t->prob) d_prob = g->scratch[0].p;
        if (t->fg || t->fg_bits) d_fg = g->scratch[1].p;
        if (t->bg || t->bg_bits) d_bg = g->scratch[4].p;
        const int slots[4] = {0, 1, 2, 4};
        for (int i = 0; i < 4; ++i) if (g->slot_used[slots[i]]) CK(cudaStreamWaitEvent(g->up_stream, g->ev_slot[slots[i]], 0));
    }

    BoundaryParams P{};
    rc = boundary_params(g, t->boundary_kind, t->image->dtype, d_img, t->sigma, t->spacing, t->norm, &P);
    if (rc) return rc;

    BuildArgs A{};
    A.img = d_img;
    A.prob = d_prob;
    A.prob_f64 = (t->prob && t->prob->dtype == MGC_F64) ? 1 : 0;
    A.compute_f32 = (t->prob && t->compute_dtype == MGC_F32) ? 1 : 0;
    A.alpha = t->alpha;
    if (has_bits) { A.fg_bits = (const unsigned*)d_fg; A.bg_bits = (const unsigned*)d_bg; }
    else { A.fg = (const uint8_t*)d_fg; A.bg = (const uint8_t*)d_bg; }
    BuildMaps imap{};
    A.use_tma = make_image_map(g, d_img, t->image->dtype, &imap.img) ? 1 : 0;
    if (const char* e = getenv("MEDPY_GC_BUILD_TMA")) if (atoi(e) == 0) A.use_tma = 0;
    int tin_tma = A.use_tma;                 // t-link inputs through TMA as well (MEDPY_GC_BUILD_TMA=2: image only)
    if (const char* e = getenv("MEDPY_GC_BUILD_TMA")) if (atoi(e) == 2) tin_tma = 0;
    if (tin_tma) {
        if (d_prob && make_block_map(g, d_prob, t->prob->dtype, &imap.prob)) A.tma_prob = 1;
        if (!has_bits) {
            if (d_fg && make_block_map(g, d_fg, MGC_U8, &imap.fg)) A.tma_mark |= 1;
            if (d_bg && make_block_map(g, d_bg, MGC_U8, &imap.bg)) A.tma_mark |= 2;
        }
    }
    if (const char* e = getenv("MEDPY_GC_BUILD_DBG")) A.dbg = atoi(e);
    // lazy build: materialisation re-reads the inputs until the solve is done -- staged copies are the handle's own,
    // caller-owned device arrays only with MGC_OPT_KEEP_INPUTS
    const bool borrowed = d_img == t->image->data || (t->prob && d_prob == t->prob->data) || (t->fg && d_fg == t->fg->data) ||
                          (t->bg && d_bg == t->bg->data);
    g->lazy = g->lazy_build && !g->slab && g->bflag && (!borrowed || g->keep_inputs) && lazy_variant(A, P, t->image->dtype);
    g->lazy_blocks = 0;
    if (g->lazy) {
        g->lazy_maps = imap; g->lazy_args = A; g->lazy_P = P;
        g->lazy_blocks = (int64_t)nzt * ((g->L.dim[1] + BUILD_TY - 1) / BUILD_TY) * ((g->L.dim[2] + BUILD_TX - 1) / BUILD_TX);
        CK(cudaMemsetAsync(g->d_lazy, 0, sizeof(int), g->stream));
    }

    CK(cudaMemsetAsync(g->d_tcount, 0, 256, g->stream));
    CK(cudaMemsetAsync(g->d_flags, 0, sizeof(int), g->stream));
    { int rcd = dirty_clear(g); if (rcd) return rcd; }
    g->pl_sel[0] = g->pl_sel[1] = 0;
    cudaEventRecord(g->ev_b[0], g->stream);
    if (!chunked) {
        A.z_tile0 = 0;
        rc = build_launch_dtype(g, t->image->dtype, imap, A, P, nzt);
        if (rc) return rc;
    } else {
        int nchunks = g->build_chunks < nzt ? g->build_chunks : nzt;
        const int per = (nzt + nchunks - 1) / nchunks;
        nchunks = (nzt + per - 1) / per;
        const char* h_img = (const char*)t->image->data;
        int prev_l0 = 0, prev_nl = 0;
        for (int c = 0; c < nchunks; ++c) {
            const int l0 = c * per, l1 = (l0 + per < nzt) ? l0 + per : nzt;
            const size_t z0 = (size_t)l0 * BUILD_TZ, z1 = ((size_t)l1 * BUILD_TZ < (size_t)Z) ? (size_t)l1 * BUILD_TZ : (size_t)Z;
            const size_t v0 = z0 * plane, nv = (z1 - z0) * plane;
            CK(cudaMemcpyAsync((char*)g->scratch[2].p + v0 * es_img, h_img + v0 * es_img, nv * es_img, cudaMemcpyHostToDevice, g->up_stream));
            if (c > 0) {
                // chunk c-1 needs the first image plane of chunk c (its +z neighbours) and its own prob / markers
                CK(cudaEventRecord(g->ev_chunk[c & 1], g->up_stream));
                CK(cudaStreamWaitEvent(g->stream, g->ev_chunk[c & 1], 0));
                A.z_tile0 = prev_l0;
                rc = build_launch_dtype(g, t->image->dtype, imap, A, P, prev_nl);
                if (rc) { cudaStreamSynchronize(g->up_stream); return rc; }     // the host arrays are borrowed: no copy may outlive the call
            }
            if (t->prob) CK(cudaMemcpyAsync((char*)g->scratch[0].p + v0 * es_prob, (const char*)t->prob->data + v0 * es_prob, nv * es_prob, cudaMemcpyHostToDevice, g->up_stream));
            if (has_bits) {
                const size_t w0 = v0 / 32, w1 = (v0 + nv + 31) / 32;
                if (t->bits_ready_words) {        // producer thread still packing: wait until this chunk's words exist
                    const int64_t need = (int64_t)(w1 < words ? w1 : words);
                    while (*t->bits_ready_words < need) std::this_thread::yield();   // packing runs at memory speed, far ahead of PCIe
                    std::atomic_thread_fence(std::memory_order_acquire);
                }
                if (t->fg_bits) CK(cudaMemcpyAsync((uint32_t*)g->scratch[1].p + w0, t->fg_bits + w0, (w1 - w0) * 4, cudaMemcpyHostToDevice, g->up_stream));
                if (t->bg_bits) CK(cudaMemcpyAsync((uint32_t*)g->scratch[4].p + w0, t->bg_bits + w0, (w1 - w0) * 4, cudaMemcpyHostToDevice, g->up_stream));
            } else {
                if (t->fg) CK(cudaMemcpyAsync((char*)g->scratch[1].p + v0, (const char*)t->fg->data + v0, nv, cudaMemcpyHostToDevice, g->up_stream));
                if (t->bg) CK(cudaMemcpyAsync((char*)g->scratch[4].p + v0, (const char*)t->bg->data + v0, nv, cudaMemcpyHostToDevice, g->up_stream));
            }
            prev_l0 = l0; prev_nl = l1 - l0;
        }
        CK(cudaEventRecord(g->ev_up, g->up_stream));
        CK(cudaStreamWaitEvent(g->stream, g->ev_up, 0));
        A.z_tile0 = prev_l0;
        rc = build_launch_dtype(g, t->image->dtype, imap, A, P, prev_nl);
        if (rc) { cudaStreamSynchronize(g->up_stream); return rc; }
        CK(cudaEventSynchronize(g->ev_up));       // the host arrays are only borrowed for this call
    }
    cudaEventRecord(g->ev_b[1], g->stream);
    {   // flow constant: one partial per build block, fixed order
        const unsigned nbuild = (unsigned)nzt * (unsigned)((g->L.dim[1] + BUILD_TY - 1) / BUILD_TY) * (unsigned)((g->L.dim[2] + BUILD_TX - 1) / BUILD_TX);
        k_sum_partials<<<1, 256, 0, g->stream>>>(g->partials, nbuild, g->d_scalars);
        g->st.kernel_launches++;
        CK(cudaGetLastError());
    }
    g->caps_fresh = false;
    g->tr_fresh = false;
    g->has_nlinks = true;
    g->boundary_timed = true;
    g->state_init = true;
    g->solved = false;
    g->host_mask_valid = false;
    g->labels_fresh = true;
    g->rl_cur = 0;
    g->sweep_mode = -1;
    g->init_timed = false;
    g->st.ms_init = 0.0;
    span.stop(0x17u);
    if (g->defer_check && g->h_bad) {
        CK(cudaMemcpyAsync(g->h_bad, g->d_flags, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
        CK(cudaEventRecord(g->ev_bad, g->stream));
        g->bad_pending = true;
        return MGC_OK;
    }
    int bad = 0;
    CK(cudaMemcpyAsync(&bad, g->d_flags, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
    CK(cudaStreamSynchronize(g->stream));
    if (bad) FAIL(MGC_E_WEIGHT, "Negative or zero weights are not allowed.");
    return MGC_OK;
}

int mgc_add_nweights_dense(mgc_graph* g, int32_t axis, const mgc_array* fwd, const mgc_array* bwd)
{
    if (!g || !fwd || !bwd) return MGC_E_ARG;
    if (g->flow_started) FAIL(MGC_E_STATE, "the graph has been solved (its capacities hold residuals): reset() it before adding terms");
    if (axis < 0 || axis >= g->user_ndim) FAIL(MGC_E_ARG, "bad axis");
    if (fwd->dtype != MGC_F64 || bwd->dtype != MGC_F64) FAIL(MGC_E_ARG, "dense n-weights must be float64");
    CK(cudaSetDevice(g->device));
    { int rcl = lazy_materialise_all(g); if (rcl) return rcl; }
    { int rc0 = check_pending(g); if (rc0) return rc0; }
    TermSpan t(g);
    const void *pf = nullptr, *pb = nullptr;
    int rc = stage_input(g, fwd, 0, &pf);
    if (rc) return rc;
    rc = stage_input(g, bwd, 1, &pb);
    if (rc) return rc;
    if (g->caps_fresh) {
        const size_t nbz = (size_t)g->L.n;
        for (int k = 0; k < 2 * g->nd; ++k) CK(cudaMemsetAsync(g->S.cap[k], 0, nbz * sizeof(double), g->stream));
        g->caps_fresh = false;
    }
    CK(cudaMemsetAsync(g->d_flags, 0, sizeof(int), g->stream));
    const int ca = axis + g->shift;
    if (g->nd == 3) k_nweights_dense<3, double><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S, ca, (const double*)pf, (const double*)pb, g->d_flags);
    else            k_nweights_dense<4, double><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S, ca, (const double*)pf, (const double*)pb, g->d_flags);
    g->st.kernel_launches++;
    CK(cudaGetLastError());
    int bad = 0;
    CK(cudaMemcpyAsync(&bad, g->d_flags, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
    t.stop(3u);
    CK(cudaStreamSynchronize(g->stream));
    invalidate(g);
    g->has_nlinks = true;
    if (bad) FAIL(MGC_E_WEIGHT, "Negative or zero weights are not allowed.");
    return MGC_OK;
}

int mgc_maxflow(mgc_graph* g, double* energy)
{
    if (!g) return MGC_E_ARG;
    if (g->slab) FAIL(MGC_E_STATE, "z-slab handles are stepped with mgc_slab_*");
    CK(cudaSetDevice(g->device));
    if (g->solved) { if (energy) *energy = g->energy; return MGC_OK; }
    { int rc0 = check_pending(g); if (rc0) return rc0; }
    resolve_term_span(g);
    {
        Timer t(g, &g->st.ms_solve);
        int rc = MGC_OK;
        if (!g->use_tiles || g->use_coop || g->debug_checks) {      // no per-colour hook in these paths
            rc = lazy_materialise_all(g); if (rc) return rc;
        }
        if (g->use_tiles) {
            if (g->debug_checks) {
                rc = materialise_zeros(g); if (rc) return rc;
                if (!g->state_init) { rc = init_tiles(g); if (rc) return rc; }
                rc = debug_invariants(g, false); if (rc) return rc;
            }
            rc = solve_tiles(g);
            if (rc) return rc;
            rc = debug_invariants(g, true);
            if (rc) return rc;
        } else {
        rc = ensure_state(g);
        if (rc) return rc;
        int64_t rounds = 0;
        for (;;) {
            rc = relabel_init(g);
            if (rc) return rc;
            int any = 0;
            rc = relabel_relax(g, &any);
            if (rc) return rc;
            g->st.global_relabels++;
            int64_t active = 0;
            rc = count_active(g, &active);
            if (rc) return rc;
            if (active == 0) break;
            if (++rounds > g->max_rounds) FAIL(MGC_E_NOCONV, "push-relabel did not converge within the round cap");
            // push sweeps until quiescent or the round budget is used
            int done = 0;
            while (done < g->sweeps_per_round) {
                int chunk = g->sweeps_per_round - done;
                if (chunk > 8) chunk = 8;
                int work = 1;
                rc = push_sweeps(g, chunk, &work);
                if (rc) return rc;
                done += chunk;
                if (!work) break;
            }
        }
        }
        t.stop_sync();
    }
    {
        Timer t(g, &g->st.ms_readout);
        double e = 0.0;
        int rc = readout(g, &e);
        if (rc) return rc;
        g->energy = e;
        g->st.energy = e;
        t.stop_sync();
    }
    g->solved = true;
    if (energy) *energy = g->energy;
    return MGC_OK;
}

int mgc_get_mask(mgc_graph* g, uint8_t* out, int32_t mem)
{
    if (!g || !out) return MGC_E_ARG;
    if (!g->solved) FAIL(MGC_E_STATE, "call maxflow first");
    CK(cudaSetDevice(g->device));
    const size_t owned_n = (size_t)(g->L.own1 - g->L.own0) * g->L.plane;
    const uint8_t* src = g->mask_dev + (size_t)g->L.own0 * g->L.plane;
    CK(cudaMemcpyAsync(out, src, owned_n, mem == MGC_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, g->stream));
    CK(cudaStreamSynchronize(g->stream));
    return MGC_OK;
}

int mgc_what_segment(mgc_graph* g, int64_t node, int32_t* segment)
{
    if (!g || !segment) return MGC_E_ARG;
    if (!g->solved) FAIL(MGC_E_STATE, "call maxflow first");
    if (node < 0 || node >= (int64_t)g->L.n) FAIL(MGC_E_ARG, "node id out of range");
    if (!g->host_mask_valid) {
        g->host_mask.resize(g->L.n);
        CK(cudaMemcpyAsync(g->host_mask.data(), g->mask_dev, g->L.n, cudaMemcpyDeviceToHost, g->stream));
        CK(cudaStreamSynchronize(g->stream));
        g->host_mask_valid = true;
    }
    *segment = g->host_mask[(size_t)node] ? MGC_SOURCE : MGC_SINK;
    return MGC_OK;
}

int mgc_get_edge(mgc_graph* g, int64_t i, int64_t j, double* cap)
{
    if (!g || !cap) return MGC_E_ARG;
    const int64_t n = (int64_t)g->L.n;
    if (i < 0 || j < 0 || i >= n || j >= n || i == j) FAIL(MGC_E_ARG, "bad node ids");
    *cap = 0.0;
    if (g->caps_fresh) return MGC_OK;
    CK(cudaSetDevice(g->device));
    { int rcl = lazy_materialise_all(g); if (rcl) return rcl; }
    int c[4] = {0, 0, 0, 0};
    unsigned r = (unsigned)i;
    for (int d = 0; d < g->nd; ++d) { c[d] = (int)(r / g->L.stride[d]); r %= g->L.stride[d]; }
    for (int k = 0; k < 2 * g->nd; ++k) {
        const int d = k >> 1;
        const int64_t off = (k & 1) ? (int64_t)g->L.stride[d] : -(int64_t)g->L.stride[d];
        const int cn = c[d] + ((k & 1) ? 1 : -1);
        if (cn < 0 || cn >= g->L.dim[d]) continue;
        if (i + off == j) {
            CK(cudaMemcpyAsync(cap, g->S.cap[k] + i, sizeof(double), cudaMemcpyDeviceToHost, g->stream));
            CK(cudaStreamSynchronize(g->stream));
            return MGC_OK;
        }
    }
    return MGC_OK;  // not lattice neighbours: 0, like get_edge on a missing arc (graph.h:482-497)
}

int mgc_get_trcap(mgc_graph* g, int64_t node, double* trcap)
{
    if (!g || !trcap) return MGC_E_ARG;
    if (node < 0 || node >= (int64_t)g->L.n) FAIL(MGC_E_ARG, "node id out of range");
    if (g->tr_fresh) { *trcap = 0.0; return MGC_OK; }
    CK(cudaSetDevice(g->device));
    { int rcl = lazy_materialise_all(g); if (rcl) return rcl; }
    if (!g->state_init || !g->flow_started) {      // no flow yet: the net terminal capacity exactly as add_tweights left it
        CK(cudaMemcpyAsync(trcap, g->S.tr + node, sizeof(double), cudaMemcpyDeviceToHost, g->stream));
        CK(cudaStreamSynchronize(g->stream));
        return MGC_OK;
    }
    double e = 0, s = 0;
    uint8_t rm = 0x80u;
    CK(cudaMemcpyAsync(&e, g->S.excess + node, sizeof(double), cudaMemcpyDeviceToHost, g->stream));
    CK(cudaMemcpyAsync(&s, g->S.sink + node, sizeof(double), cudaMemcpyDeviceToHost, g->stream));
    if (g->use_tiles && g->nd == 3) CK(cudaMemcpyAsync(&rm, g->S.rmask + node, 1, cudaMemcpyDeviceToHost, g->stream));
    CK(cudaStreamSynchronize(g->stream));
    if (!(rm & 0x80u)) s = 0;        // RM_SINKV clear: nothing absorbed yet, the entry was never written
    double tr = 0;
    CK(cudaMemcpyAsync(&tr, g->S.tr + node, sizeof(double), cudaMemcpyDeviceToHost, g->stream));
    CK(cudaStreamSynchronize(g->stream));
    *trcap = (tr < 0 && -tr - s > 0) ? -(-tr - s) : e;
    return MGC_OK;
}

int mgc_get_node_num(const mgc_graph* g, int64_t* n)
{
    if (!g || !n) return MGC_E_ARG;
    *n = (int64_t)g->L.n;
    return MGC_OK;
}

int mgc_get_arc_num(const mgc_graph* g, int64_t* n)
{
    if (!g || !n) return MGC_E_ARG;
    int64_t e = 0;
    if (g->has_nlinks)
        for (int d = 0; d < g->nd; ++d)
            if (g->L.dim[d] > 1) e += ((int64_t)g->L.n / g->L.dim[d]) * (g->L.dim[d] - 1);
    *n = 2 * e;
    return MGC_OK;
}

int mgc_get_stats(const mgc_graph* g, mgc_stats* out)
{
    if (!g || !out) return MGC_E_ARG;
    *out = g->st;
    out->device_bytes = g->device_bytes;
    return MGC_OK;
}

int mgc_get_lazy_stats(const mgc_graph* g, int64_t* build_blocks, int64_t* materialised)
{
    if (!g || !build_blocks || !materialised) return MGC_E_ARG;
    *build_blocks = g->lazy_blocks;
    *materialised = g->lazy_materialised;
    return MGC_OK;
}

// ---- z-slab stepping --------------------------------------------------------------------------------

int mgc_slab_plane_elems(const mgc_graph* g, int64_t* n)
{
    if (!g || !n) return MGC_E_ARG;
    *n = (int64_t)g->L.plane;
    return MGC_OK;
}

int mgc_slab_begin(mgc_graph* g)
{
    if (!g) return MGC_E_ARG;
    CK(cudaSetDevice(g->device));
    { int rc0 = check_pending(g); if (rc0) return rc0; }
    resolve_term_span(g);
    if (g->use_tiles) {
        int rc = materialise_zeros(g);
        if (rc) return rc;
        return g->state_init ? MGC_OK : init_tiles(g);
    }
    return ensure_state(g);
}

int mgc_slab_push(mgc_graph* g, int32_t n)
{
    if (!g || n < 0) return MGC_E_ARG;
    if (!g->state_init) FAIL(MGC_E_STATE, "call mgc_slab_begin first");
    CK(cudaSetDevice(g->device));
    g->iters_now = g->tile_iters;
    if (g->use_tiles) return g->use_coop ? solve_coop(g, SOLVE_F_PUSH, n, nullptr) : push_tiles(g, n);
    return push_sweeps(g, n, nullptr);
}

int mgc_slab_pack(mgc_graph* g, int32_t* h_lo, double* f_lo, int32_t* h_hi, double* f_hi)
{
    if (!g) return MGC_E_ARG;
    CK(cudaSetDevice(g->device));
    const unsigned P = g->L.plane;
    const unsigned nb = (P + 255u) / 256u;
    if (g->ghost_lo && h_lo) {
        const size_t border = (size_t)g->L.own0 * P, ghost = border - P;
        k_slab_pack<double><<<nb, 256, 0, g->stream>>>(P, g->S.height + border, g->S.excess + ghost, h_lo, f_lo);
        g->st.kernel_launches++;
    }
    if (g->ghost_hi && h_hi) {
        const size_t border = (size_t)(g->L.own1 - 1) * P, ghost = border + P;
        k_slab_pack<double><<<nb, 256, 0, g->stream>>>(P, g->S.height + border, g->S.excess + ghost, h_hi, f_hi);
        g->st.kernel_launches++;
    }
    CK(cudaGetLastError());
    return MGC_OK;
}

int mgc_slab_unpack(mgc_graph* g, const int32_t* h_lo, const double* f_lo, const int32_t* h_hi, const double* f_hi,
                    int32_t* changed_dev)
{
    if (!g) return MGC_E_ARG;
    CK(cudaSetDevice(g->device));
    const unsigned P = g->L.plane;
    const unsigned nb = (P + 255u) / 256u;
    for (int side = 0; side < 2; ++side) {
        const bool have = side == 0 ? (g->ghost_lo && h_lo) : (g->ghost_hi && h_hi);
        if (!have) continue;
        const int zb = side == 0 ? g->L.own0 : g->L.own1 - 1;
        const int zg = side == 0 ? zb - 1 : zb + 1;
        const int k = side == 0 ? 0 : 1;     // my arc border -> ghost: axis 0, -1 (lo) or +1 (hi)
        const int32_t* hin = side == 0 ? h_lo : h_hi;
        const double* fin = side == 0 ? f_lo : f_hi;
        if (g->use_tiles) {
            k_slab_unpack_tiles<double><<<nb, 256, 0, g->stream>>>(g->L, g->TL, g->S, zg, zb, k, hin, fin, g->rflag, rl(g, 0), rl(g, 1),
                                                                  g->coop_bfs_grid > 0 ? g->d_tcount + CTL_RLCUR : nullptr, g->rl_cur,
                                                                  g->pflag, pl(g, 0, g->pl_sel[0]), pl(g, 1, g->pl_sel[1]), changed_dev);
        } else {
            const size_t border = (size_t)zb * P, ghost = (size_t)zg * P;
            k_slab_unpack<double><<<nb, 256, 0, g->stream>>>(P, g->S.height + ghost, g->S.excess + border, g->S.cap[k] + border,
                                                            hin, fin, changed_dev);
        }
        g->st.kernel_launches++;
    }
    CK(cudaGetLastError());
    return MGC_OK;
}

int mgc_slab_relabel_begin(mgc_graph* g)
{
    if (!g) return MGC_E_ARG;
    if (!g->state_init) FAIL(MGC_E_STATE, "call mgc_slab_begin first");
    CK(cudaSetDevice(g->device));
    g->st.global_relabels++;
    if (g->use_tiles) return relabel_tiles_begin(g);
    return relabel_init(g);
}

int mgc_slab_relabel_relax(mgc_graph* g, int32_t* changed_out)
{
    if (!g) return MGC_E_ARG;
    CK(cudaSetDevice(g->device));
    int any = 0;
    int rc = MGC_OK;
    if (g->use_tiles && g->use_coop) {
        const int64_t before = g->st.relabel_sweeps;
        rc = solve_coop(g, SOLVE_F_BFS, 0, nullptr);
        any = g->st.relabel_sweeps != before;
        g->st.global_relabels--;      // counted by mgc_slab_relabel_begin already
    } else {
        rc = g->use_tiles ? relabel_tiles_run(g, &any, changed_out != nullptr) : relabel_relax(g, &any);
    }
    if (rc) return rc;
    if (changed_out) *changed_out = any ? 1 : 0;
    return MGC_OK;
}

int mgc_slab_count_active(mgc_graph* g, int64_t* active_out)
{
    if (!g || !active_out) return MGC_E_ARG;
    CK(cudaSetDevice(g->device));
    return g->use_tiles ? count_active_tiles(g, active_out) : count_active(g, active_out);
}

int mgc_slab_count_active_dev(mgc_graph* g, unsigned long long* count_dev)
{
    if (!g || !count_dev) return MGC_E_ARG;
    CK(cudaSetDevice(g->device));
    CK(cudaMemsetAsync(count_dev, 0, sizeof(unsigned long long), g->stream));
    if (g->use_tiles) {
        return count_active_tiles_enqueue(g, count_dev);
    } else {
        k_count_active<double><<<nblocks(g), 256, 0, g->stream>>>(g->L, g->S, count_dev);
        g->st.kernel_launches++;
    }
    CK(cudaGetLastError());
    return MGC_OK;
}

int mgc_slab_finish(mgc_graph* g, double* energy_part)
{
    if (!g || !energy_part) return MGC_E_ARG;
    CK(cudaSetDevice(g->device));
    int rc = readout(g, energy_part);
    if (rc) return rc;
    g->energy = *energy_part;
    g->st.energy = g->energy;
    g->solved = true;
    return MGC_OK;
}

// ---- z-slab solve inside the library: NCCL point-to-point on the handle's stream, one host decision per relabel round --

int mgc_slab_comm_unique_id(void* out128)
{
    if (!out128) return MGC_E_ARG;
    NcclApi& N = nccl_api();
    if (!N.ok) { g_create_error = "libnccl.so.2 could not be loaded"; return MGC_E_CUDA; }
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    if (N.GetUniqueId(&id) != ncclSuccess) { g_create_error = "ncclGetUniqueId failed"; return MGC_E_CUDA; }
    memcpy(out128, &id, sizeof(id));
    return MGC_OK;
}

int mgc_slab_comm_init(mgc_graph* g, int32_t rank, int32_t world, const void* unique_id128)
{
    if (!g || !unique_id128 || world < 1 || rank < 0 || rank >= world) return MGC_E_ARG;
    if (!g->slab) FAIL(MGC_E_STATE, "not a z-slab handle");
    NcclApi& N = nccl_api();
    if (!N.ok) FAIL(MGC_E_CUDA, "libnccl.so.2 could not be loaded");
    CK(cudaSetDevice(g->device));
    if ((rank > 0) != g->ghost_lo || (rank < world - 1) != g->ghost_hi) FAIL(MGC_E_ARG, "rank / world do not match the slab's position");
    slab_comm_release(g);
    ncclUniqueId id;
    memcpy(&id, unique_id128, sizeof(id));
    NK(N.CommInitRank(&g->comm, world, id, rank));
    g->comm_rank = rank; g->comm_world = world;
    const size_t P = g->L.plane;
    g->msg_h_bytes = (P * 4 + 7) / 8 * 8;
    g->msg_bytes = g->msg_h_bytes + P * 8;
    void* p = nullptr;
    for (int i = 0; i < 4; ++i) if (!g->msg[i]) { int rc = alloc_buf(g, g->msg_bytes, &p); if (rc) return rc; g->msg[i] = (char*)p; CK(cudaMemsetAsync(p, 0, g->msg_bytes, g->stream)); }
    if (!g->d_stat) { int rc = alloc_buf(g, 64, &p); if (rc) return rc; g->d_stat = (long long*)p; }
    if (!g->d_esum) { int rc = alloc_buf(g, 64, &p); if (rc) return rc; g->d_esum = (double*)p; }
    if (!g->h_stat) { void* hp = nullptr; if (mgc_host_alloc(64, &hp) != MGC_OK) FAIL(MGC_E_NOMEM, "pinned host allocation failed"); g->h_stat = (long long*)hp; }
    return MGC_OK;
}

// The whole distributed solve (what medpy_b200/distributed.py sequenced from Python in round 1).  Distributed global
// relabel = local BFS to a fixed point <-> border-label exchange; two rounds + the active count are enqueued
// speculatively and checked with ONE all-reduce and ONE host synchronisation (valid iff round B changed nothing anywhere).
// Returns the TOTAL energy (all-reduced) in *energy_total.
int mgc_slab_solve(mgc_graph* g, double* energy_total)
{
    if (!g || !energy_total) return MGC_E_ARG;
    if (!g->slab || !g->comm) FAIL(MGC_E_STATE, "call mgc_slab_comm_init first");
    NcclApi& N = nccl_api();
    CK(cudaSetDevice(g->device));
    int rc = mgc_slab_begin(g);
    if (rc) return rc;
    g->slab_exchanges = g->slab_relabel_rounds = g->slab_push_passes = g->slab_global_relabels = 0;
    for (double& x : g->slab_phase_ms) x = 0.0;
    g->ph_used = 0; g->ph_kind.clear();
    auto timed_sync = [&]() -> cudaError_t {
        const auto t0 = std::chrono::steady_clock::now();
        const cudaError_t e = cudaStreamSynchronize(g->stream);
        g->slab_phase_ms[5] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        return e;
    };
    int passes = g->passes0 > 0 ? g->passes0 : 1;
    const int passes_cap = g->passes_max < 8 ? g->passes_max : 8;
    int64_t rounds = 0;
    for (;;) {
        phase_begin(g, 0);
        rc = mgc_slab_relabel_begin(g);
        phase_end(g);
        if (rc) return rc;
        for (;;) {
            CK(cudaMemsetAsync(g->d_stat, 0, 3 * sizeof(long long), g->stream));
            for (int k = 0; k < 2; ++k) {
                phase_begin(g, 0);
                rc = mgc_slab_relabel_relax(g, nullptr);
                phase_end(g);
                if (rc) return rc;
                rc = slab_exchange(g, g->d_stat + k, true);
                if (rc) return rc;
                g->slab_relabel_rounds++;
            }
            phase_begin(g, 2);
            rc = mgc_slab_count_active_dev(g, (unsigned long long*)(g->d_stat + 2));
            if (rc) return rc;
            if (g->comm_world > 1) NK(N.AllReduce(g->d_stat, g->d_stat, 3, ncclInt64, ncclSum, g->comm, g->stream));
            CK(cudaMemcpyAsync(g->h_stat, g->d_stat, 3 * sizeof(long long), cudaMemcpyDeviceToHost, g->stream));
            phase_end(g);
            CK(timed_sync());                                          // the one host decision of this round
            rc = slab_comm_poll(g);
            if (rc) return rc;
            if (g->h_stat[1] == 0) break;
        }
        g->slab_global_relabels++;
        if (g->h_stat[2] == 0) break;
        if (++rounds > g->max_rounds) FAIL(MGC_E_NOCONV, "push-relabel did not converge within the round cap");
        for (int p = 0; p < passes; ++p) {
            phase_begin(g, 3);
            rc = mgc_slab_push(g, 1);
            phase_end(g);
            if (rc) return rc;
            rc = slab_exchange(g, nullptr, false);
            if (rc) return rc;
            g->slab_push_passes++;
        }
        passes = passes * 2 > passes_cap ? passes_cap : passes * 2;
    }
    double part = 0.0;
    phase_begin(g, 4);
    rc = mgc_slab_finish(g, &part);
    if (rc) return rc;
    CK(cudaMemcpyAsync(g->d_esum, &part, sizeof(double), cudaMemcpyHostToDevice, g->stream));
    if (g->comm_world > 1) NK(N.AllReduce(g->d_esum, g->d_esum, 1, ncclFloat64, ncclSum, g->comm, g->stream));
    CK(cudaMemcpyAsync(energy_total, g->d_esum, sizeof(double), cudaMemcpyDeviceToHost, g->stream));
    phase_end(g);
    CK(timed_sync());
    phase_resolve(g);
    return slab_comm_poll(g);
}

int mgc_slab_solve_phase_ms(const mgc_graph* g, double* out6)
{
    if (!g || !out6) return MGC_E_ARG;
    for (int i = 0; i < 6; ++i) out6[i] = g->slab_phase_ms[i];
    return MGC_OK;
}

int mgc_slab_solve_stats(const mgc_graph* g, int64_t* exchanges, int64_t* relabel_rounds, int64_t* push_passes, int64_t* global_relabels)
{
    if (!g) return MGC_E_ARG;
    if (exchanges) *exchanges = g->slab_exchanges;
    if (relabel_rounds) *relabel_rounds = g->slab_relabel_rounds;
    if (push_passes) *push_passes = g->slab_push_passes;
    if (global_relabels) *global_relabels = g->slab_global_relabels;
    return MGC_OK;
}

}  // extern "C"
