// gc_build.cuh -- the whole graph build as ONE pass over the lattice (3-D): n-link stencil + regional t-links + hard
// markers + solver-state initialisation, fused.
//
// Replaces, in one kernel, what the reference does in  energy_voxel.py:611-664 (__skeleton_base, one Python call
// per edge), graph.py:532-552 / :310-380 (set_tweights_all, set_source_nodes, set_sink_nodes -> Graph::add_tweights,
// graph.h:415-425) in the order graph_from_voxels applies them (generate.py:159-172: regional term, boundary term,
// foreground markers, background markers), plus what k_boundary / k_regional / k_markers / k_init_tile did in four
// passes here (r01: 24.5 GB of DRAM traffic per 512^3 step, 6.4 GB of it capacity planes written by one kernel and
// read straight back by the next).  Now every input byte is read once and every state byte written once:
//     read  image 4 + probability 4 + fg 1 + bg 1                         = 10 B/voxel (float32 inputs)
//     write six float64 capacities 48 + tr 8 + excess 8 + label 4 + rmask 1 = 69 B/voxel
// (`sink[]`, the absorbed-flow accumulator, is no longer zero-filled: bit RM_SINKV of rmask says whether a voxel's
// entry has been written, see gc_tiles.cuh.)
//
// Geometry: a 256-thread CTA builds an 8 (z) x 8 (y) x 32 (x) block = four 8^3 solver tiles in a row.  The image
// block with a one-voxel halo on every side (10 x 10 x 34, box 10 x 10 x BuildBox<E>::BX) is staged in shared memory by ONE
// `cp.async.bulk.tensor.3d` box copy against a per-call tensor map (SASS: UTMALDG + SYNCS; out-of-lattice parts are
// zero-filled by the TMA unit and masked by coordinates), or by plain loads when the image does not meet the 16-byte
// stride rule of tensor maps.  Thread (y, x) marches through z = -1 .. 7: per step it evaluates the three FORWARD
// pair weights of its voxel (+z, +y, +x) exactly once -- w(p, q) = g(|I_p - I_q|) or g(max(|I_p|, |I_q|)), float64,
// the arithmetic of gc_terms.cuh -- keeps the +z weight in a register for the next step (where it is the voxel's -z
// capacity), and publishes the +y / +x weights in a shared-memory plane from which the neighbours in y and x take
// their backward capacities.  The only weights evaluated twice are those on the block's low faces (12.5 %).
#pragma once
#include "gc_terms.cuh"
#include "gc_tiles.cuh"
#include "gc_tma.cuh"

#define BUILD_TZ 8
#define BUILD_TY 8
#define BUILD_TX 32
#define BUILD_THREADS 256
// Inner (x) extent of the staged image block.  Measured on B200: UTMALDG raises "illegal instruction" when the box
// start along the innermost axis is negative or not 16-byte aligned, so the box starts BUILD_PAD = 16 / sizeof(E)
// elements in front of the block (x0 is a multiple of 32) instead of 1, or at 0 for the blocks on the low x face; the
// extent covers pad + 32 + 1 elements, rounded up to a multiple of 16 bytes.
// shared-memory offset of the staged t-link inputs: behind image block, weight planes, barrier, flags, reduction scratch
#define BUILD_TIN_OFFSET(img_pad) ((((img_pad) + (2 * 9 * 32 + 2 * 8 * 33 + 8 * 32 + 8 * 8) * 8 + 8 + 32 + 64) + 127) / 128 * 128)
template <typename E> struct BuildBox {
    static constexpr int PAD = 16 / (int)sizeof(E);
    static constexpr int BX = (PAD + 33 + PAD - 1) / PAD * PAD;      // f32 40, f64 36, u8 64, i16 48, i32 40
};
#define BUILD_HY 10
#define BUILD_HZ 10

// tensor maps of one build: image (halo box), probability map and the two marker volumes (8 x 8 x 32 blocks)
struct BuildMaps {
    CUtensorMap img, prob, fg, bg;
};

struct BuildArgs {
    const void* img;           // C-contiguous image over the local lattice (device)
    const void* prob;          // regional_probability_map input or nullptr
    int prob_f64;              // 1: prob is float64
    int compute_f32;           // products in float32 (numpy: float32 map * Python float)
    double alpha;
    const uint8_t* fg;         // marker volumes (bytes) or nullptr
    const uint8_t* bg;
    const unsigned* fg_bits;   // ... or bit-packed (bit v & 31 of word v >> 5), used when fg/bg are nullptr
    const unsigned* bg_bits;
    int use_tma;               // image block staged by TMA (else plain loads)
    int tma_prob;              // probability block (8 x 8 x 32) staged by TMA into shared memory
    int tma_mark;              // fg / bg byte blocks staged by TMA (bit 0: fg, bit 1: bg)
    int z_tile0;               // first z tile layer of this launch (chunked builds)
    int dbg;                   // diagnostics (MEDPY_GC_BUILD_DBG): 1 = do not load the probability map (constant 0.3)
};

template <typename E>
__device__ __forceinline__ double build_val(E x, bool use_max)
{
    return use_max ? Elem<E>::val(Elem<E>::absv(x)) : Elem<E>::val(x);
}

template <int FN, typename E>
__device__ __forceinline__ double build_pair(const BoundaryParams& P, double a, E iq, bool use_max)
{
    const double b = build_val<E>(iq, use_max);
    const double x = use_max ? fmax(a, b) : fabs(__dsub_rn(a, b));
    return g_weight<FN>(P, x);
}

// TIN = 1: the common configuration fixed at compile time -- float32 probability map with float32 products and both
// marker volumes as bytes, all three staged by TMA.  The generic form (TIN = 0) decides each of those per voxel with
// warp-uniform branches: ncu's instruction mix showed ~80 of the 483 instructions per voxel going into that bookkeeping.
// Lazy build (MODE, TIN = 1 only).  A block none of whose voxels holds source excess after the t-links (tr > 0) is COLD:
// the max-flow phase reaches it only if flow is pushed into it, and until then the BFS, the sweeps, the relabel resets
// and the read-out need only its rmask and height.  MODE 1 writes everything for hot blocks and only rmask, height, the
// worklist flags and the flow-constant partial for cold ones (no exponential, 15 instead of 79 B/voxel); bflag[block]
// says whether the cap, tr and excess planes of a block are valid.  MODE 2 materialises a cold block later: the same
// arithmetic, but it writes only those three planes (rmask and height may have moved since) -- excess is 0 there.
//   MODE 0: eager build (all planes, every block)    MODE 1: lazy build    MODE 2: materialise one block
template <typename E, typename T, int FN, int USE_MAX, int SPACING, int TIN, int MODE>
__device__ __forceinline__ void build_block(const Lattice& L, const Tiles& TL, const State<T>& S, const BuildMaps& maps,
                                            const BuildArgs& A, const BoundaryParams& P, int* __restrict__ bad,
                                            double* __restrict__ partials, int* __restrict__ rflag, const WorkList& rl,
                                            int* __restrict__ pflag, const WorkList& pl0, const WorkList& pl1,
                                            int* __restrict__ bflag, int* __restrict__ mcount, int bx, int by, int bz,
                                            bool first, unsigned parity)
{
    static_assert(MODE == 0 || TIN == 1, "the lazy build exists for the staged-input variant only");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int BUILD_BX = BuildBox<E>::BX, BUILD_PAD = BuildBox<E>::PAD;
    E* s_img = reinterpret_cast<E*>(smem_raw);                                   // [10][10][BUILD_BX]
    constexpr int IMG_BYTES = BUILD_HZ * BUILD_HY * BUILD_BX * (int)sizeof(E);
    constexpr int IMG_PAD = (IMG_BYTES + 127) / 128 * 128;
    double* s_wy = reinterpret_cast<double*>(smem_raw + IMG_PAD);                // [2][9][32]: +y weight of row y-1 .. 7
    double* s_wx = s_wy + 2 * 9 * 32;                                            // [2][8][33]: +x weight of column x-1 .. 31
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(s_wx + 2 * 8 * 33 + 8 * 32 + 8 * 8);
    int* s_flags = reinterpret_cast<int*>(bar + 1);                              // [4] needs, [4] has excess
    double* s_red = reinterpret_cast<double*>(s_flags + 8);                      // [8] block reduction
    // TMA-staged t-link inputs (ncu + A/B runs: reading them with LDG from inside the store-saturated loop cost 0.7 ms of
    // a 3.0 ms launch at 512^3; the async-proxy copies are free of the LSU queue)
    unsigned char* s_prob = smem_raw + BUILD_TIN_OFFSET(IMG_PAD);                // [8][8][32] float or double, 128-B aligned
    unsigned char* s_fg = s_prob + BUILD_TZ * BUILD_TY * BUILD_TX * 8;           // [8][8][32] bytes
    unsigned char* s_bg = s_fg + BUILD_TZ * BUILD_TY * BUILD_TX;

    const int tid = threadIdx.x;
    const int lx = tid & 31, ly = tid >> 5;
    const int x0 = bx * BUILD_TX, y0 = by * BUILD_TY, z0 = bz * BUILD_TZ;
    const int nbx = (L.dim[2] + BUILD_TX - 1) / BUILD_TX, nby = (L.dim[1] + BUILD_TY - 1) / BUILD_TY;
    const int blk = (bz * nby + by) * nbx + bx;
    const bool use_max = USE_MAX >= 0 ? (USE_MAX != 0) : (P.use_max != 0);
    const bool spacing = SPACING >= 0 ? (SPACING != 0) : (P.inv_spacing_on != 0.0);

    const int gy = y0 + ly, gx = x0 + lx;
    const bool col_in = gy < L.dim[1] && gx < L.dim[2];
    // t-link inputs of one voxel (probability, marker flags), fetched ONE z-step ahead of their use: ncu showed the loop
    // stalled on these global loads (long scoreboard 7 of 15 cycles per issue) when they were read where they are needed
    struct TIn { double p; unsigned fb; };
    auto fetch = [&](int lz) -> TIn {
        TIn r{0.0, 0u};
        if (TIN == 1) {               // staged float32 probability (kept as the exact double image of the float) + staged marker bytes
            const int si = (lz * BUILD_TY + ly) * BUILD_TX + lx;
            r.p = (double)reinterpret_cast<const float*>(s_prob)[si];
            r.fb = (s_fg[si] ? 1u : 0u) | (s_bg[si] ? 2u : 0u);
            return r;
        }
        const int gz = z0 + lz;
        if (!(col_in && gz < L.dim[0])) return r;
        const unsigned v = (unsigned)gz * L.stride[0] + (unsigned)gy * L.stride[1] + (unsigned)gx;
        const int si = (lz * BUILD_TY + ly) * BUILD_TX + lx;          // index inside the staged 8 x 8 x 32 blocks
        if (A.prob) {
            if (A.tma_prob) r.p = A.prob_f64 ? reinterpret_cast<const double*>(s_prob)[si] : (double)reinterpret_cast<const float*>(s_prob)[si];
            else r.p = (A.dbg & 1) ? 0.3 : (A.prob_f64 ? reinterpret_cast<const double*>(A.prob)[v] : (double)reinterpret_cast<const float*>(A.prob)[v]);
        }
        if (A.fg_bits || A.bg_bits) {
            if (A.fg_bits) r.fb |= (A.fg_bits[v >> 5] >> (v & 31u)) & 1u;
            if (A.bg_bits) r.fb |= ((A.bg_bits[v >> 5] >> (v & 31u)) & 1u) << 1;
        } else {
            if (A.fg && ((A.tma_mark & 1) ? s_fg[si] : A.fg[v])) r.fb |= 1u;
            if (A.bg && ((A.tma_mark & 2) ? s_bg[si] : A.bg[v])) r.fb |= 2u;
        }
        return r;
    };
    // t-links of one voxel: add_tweights replay in the reference's order (regional, fg, bg); returns the flow-constant term
    auto tlinks = [&](const TIn& in, T& tr) -> double {
        double mm = 0.0;
        if (TIN == 1) {
            const float p = (float)in.p;
            const float af = (float)A.alpha;
            mm = add_tweights_dev(tr, (double)__fmul_rn(p, af), (double)__fmul_rn(__fsub_rn(1.0f, p), af));
        } else if (A.prob) {
            double s, t;
            if (A.compute_f32) {
                const float p = (float)in.p;           // exact: the map is float32 when its products are
                const float af = (float)A.alpha;
                s = (double)__fmul_rn(p, af);
                t = (double)__fmul_rn(__fsub_rn(1.0f, p), af);
            } else {
                s = __dmul_rn(in.p, A.alpha);
                t = __dmul_rn(__dsub_rn(1.0, in.p), A.alpha);
            }
            mm = add_tweights_dev(tr, s, t);
        }
        const bool f = (in.fb & 1u) != 0, b = (in.fb & 2u) != 0;
        if (f) mm = __dadd_rn(mm, add_tweights_dev(tr, 65535.0, 0.0));
        if (b) mm = __dadd_rn(mm, add_tweights_dev(tr, 0.0, 65535.0));
        return mm;
    };
    const bool staged_tin = TIN == 1 || (A.use_tma && ((A.prob && A.tma_prob) || A.tma_mark));
    TIn cur{0.0, 0u};
    if (!staged_tin) cur = fetch(0);          // global loads: in flight while the image block is staged

    // ---- stage the image block with halo: local (hz, hy, hx) <-> global (z0 - 1 + hz, y0 - 1 + hy, x0 - 1 + hx) ----
    // TMA: the box starts at a non-negative, 16-byte aligned x (see BuildBox) and at non-negative y / z: blocks on a low
    // face start at 0 and the shared-memory index is shifted instead -- the halo cells in front of the lattice are never
    // read.  Parts of the box beyond the high faces are zero-filled by the TMA unit.  cx / cy / cz: shared-memory index of
    // the logical halo cell 0 (global x0 - 1, y0 - 1, z0 - 1) along each axis.
    const int cx = A.use_tma ? (x0 == 0 ? -1 : BUILD_PAD - 1) : 0;
    const int cy = (A.use_tma && y0 == 0) ? -1 : 0, cz = (A.use_tma && z0 == 0) ? -1 : 0;
    if (tid < 8) s_flags[tid] = 0;
    if (A.use_tma) {
        if (tid == 0) {
            if (first) {
                mbar_init(bar, 1);
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            } else {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic reads of the last block are done
            }
            const unsigned pbytes = (A.prob && A.tma_prob) ? (unsigned)(BUILD_TZ * BUILD_TY * BUILD_TX * (A.prob_f64 ? 8 : 4)) : 0u;
            const unsigned mbytes = (unsigned)(BUILD_TZ * BUILD_TY * BUILD_TX);
            mbar_expect_tx(bar, (unsigned)IMG_BYTES + pbytes + ((A.tma_mark & 1) ? mbytes : 0u) + ((A.tma_mark & 2) ? mbytes : 0u));
            tma_load_3d(s_img, &maps.img, bar, x0 - 1 - cx, y0 - 1 - cy, z0 - 1 - cz);
            if (pbytes) tma_load_3d(s_prob, &maps.prob, bar, x0, y0, z0);
            if (A.tma_mark & 1) tma_load_3d(s_fg, &maps.fg, bar, x0, y0, z0);
            if (A.tma_mark & 2) tma_load_3d(s_bg, &maps.bg, bar, x0, y0, z0);
        }
        __syncthreads();
        mbar_wait(bar, parity);
        if (staged_tin) cur = fetch(0);
    } else {
        const E* img = reinterpret_cast<const E*>(A.img);
        for (int i = tid; i < BUILD_HZ * BUILD_HY * 34; i += BUILD_THREADS) {
            const int hx = i % 34, r = i / 34, hy = r % BUILD_HY, hz = r / BUILD_HY;
            const int gz = z0 - 1 + hz, gy = y0 - 1 + hy, gx = x0 - 1 + hx;
            E val = (E)0;
            if (gz >= 0 && gy >= 0 && gx >= 0 && gz < L.dim[0] && gy < L.dim[1] && gx < L.dim[2])
                val = img[(unsigned)gz * L.stride[0] + (unsigned)gy * L.stride[1] + (unsigned)gx];
            s_img[(hz * BUILD_HY + hy) * BUILD_BX + hx] = val;
        }
        __syncthreads();
    }

    // lazy build: the block is cold unless one of its voxels holds source excess after the t-links
    bool cold = false;
    if (MODE == 1) {
        int hot = 0;
        for (int lz = 0; lz < BUILD_TZ; ++lz) {
            if (!(col_in && z0 + lz < L.dim[0])) continue;
            T tr = (T)0;
            tlinks(fetch(lz), tr);
            if ((double)tr > 0) hot = 1;
        }
        cold = !__syncthreads_or(hot);
    }

    const bool has_py = gy + 1 < L.dim[1], has_px = gx + 1 < L.dim[2];
    const double sp_z = spacing ? P.spacing[0] : 1.0, sp_y = spacing ? P.spacing[1] : 1.0, sp_x = spacing ? P.spacing[2] : 1.0;
    // (cells in front of the lattice do not exist when the box was clamped: their index is clamped too, the value is
    // never used -- every pair that would need it is invalid)
    auto at = [&](int hz, int hy, int hx) -> E {
        const int i = ((hz + cz) * BUILD_HY + (hy + cy)) * BUILD_BX + (hx + cx);
        return s_img[i < 0 ? 0 : i];
    };

    int isbad = 0;
    unsigned needs_any = 0, exc_any = 0;
    double msum = 0.0;
    // one pair weight: value of the neighbour cell, validity, axis spacing
    auto pair_w = [&](double a, E iq, bool valid, double sp) -> double {
        double w = build_pair<FN, E>(P, a, iq, use_max);
        if (spacing) w = __ddiv_rn(w, sp);
        // the exponential term without spacing is clamped to DBL_MIN and can never be <= 0 (NaN compares false)
        if (!(FN == 1 && SPACING == 0)) { if (valid && w <= 0.0) isbad = 1; }
        return valid ? w : 0.0;
    };
    // ---- prologue: the weights on the block's three LOW faces, spread over all threads (one z-face and one y-face
    // weight per thread, the 64 x-face weights on the first two warps) so that no warp carries extra work in the loop ----
    double* s_wyh = s_wx + 2 * 8 * 33;          // [8 z][32 x]: pair (y0 - 1, y0)
    double* s_wxh = s_wyh + 8 * 32;             // [8 z][8 y]:  pair (x0 - 1, x0)
    double wz_back;
    {
        const bool vz = col_in && z0 > 0;
        wz_back = pair_w(build_val<E>(at(0, ly + 1, lx + 1), use_max), at(1, ly + 1, lx + 1), vz, sp_z);
        // thread (ly, lx) -> y-face weight of plane z0 + ly at column x0 + lx
        const bool vy = y0 > 0 && gx < L.dim[2] && z0 + ly < L.dim[0];
        s_wyh[ly * 32 + lx] = pair_w(build_val<E>(at(ly + 1, 0, lx + 1), use_max), at(ly + 1, 1, lx + 1), vy, sp_y);
        if (tid < 64) {
            const int fz = tid >> 3, fy = tid & 7;
            const bool vx = x0 > 0 && y0 + fy < L.dim[1] && z0 + fz < L.dim[0];
            s_wxh[fz * 8 + fy] = pair_w(build_val<E>(at(fz + 1, fy + 1, 0), use_max), at(fz + 1, fy + 1, 1), vx, sp_x);
        }
    }

    for (int lz = 0; lz < BUILD_TZ; ++lz) {
        const int gz = z0 + lz;
        const bool pin = col_in && gz < L.dim[0];            // block-uniform in z, per thread in y/x
        double* wyb = s_wy + (lz & 1) * 9 * 32;
        double* wxb = s_wx + (lz & 1) * 8 * 33;
        const int hz = lz + 1;
        TIn nxt{0.0, 0u};
        if (lz + 1 < BUILD_TZ) nxt = fetch(lz + 1);
        // the three forward pair weights of this voxel: independent, branch-free evaluations
        const double a = build_val<E>(at(hz, ly + 1, lx + 1), use_max);
        double wz, wy, wx;
        if (FN == 1 && SPACING == 0) {
            // exponential term: form the three arguments, let the WARP agree that all of them are ordinary (<= 700, not
            // NaN -- true for every warp of a sane image) and evaluate without any range handling; the rare warp that
            // disagrees takes the general path.  Both paths give bit-identical weights for ordinary arguments.
            auto arg = [&](E iq) -> double {
                const double b = build_val<E>(iq, use_max);
                return exp_term_arg(P, use_max ? fmax(a, b) : fabs(__dsub_rn(a, b)));
            };
            const double tz = arg(at(hz + 1, ly + 1, lx + 1)), ty = arg(at(hz, ly + 2, lx + 1)), tx = arg(at(hz, ly + 1, lx + 2));
            if (cold && __all_sync(0xffffffffu, tz >= 0.0 && tz <= 700.0 && ty >= 0.0 && ty <= 700.0 && tx >= 0.0 && tx <= 700.0)) {
                // a cold block keeps only the residual bits: exp_neg_inrange of an argument in [0, 700] is a positive
                // normal number, so every valid arc of this warp is residual and no weight has to be evaluated
                wz = 1.0; wy = 1.0; wx = 1.0;
            } else if (__all_sync(0xffffffffu, tz <= 700.0 && ty <= 700.0 && tx <= 700.0)) {
                wz = exp_neg_inrange(tz); wy = exp_neg_inrange(ty); wx = exp_neg_inrange(tx);
            } else {
                wz = exp_neg(tz); wy = exp_neg(ty); wx = exp_neg(tx);
                if (wz <= 0.0) wz = DBL_MIN;
                if (wy <= 0.0) wy = DBL_MIN;
                if (wx <= 0.0) wx = DBL_MIN;
            }
            if (!(pin && gz + 1 < L.dim[0])) wz = 0.0;
            if (!(pin && has_py)) wy = 0.0;
            if (!(pin && has_px)) wx = 0.0;
        } else {
            wz = pair_w(a, at(hz + 1, ly + 1, lx + 1), pin && gz + 1 < L.dim[0], sp_z);
            wy = pair_w(a, at(hz, ly + 2, lx + 1), pin && has_py, sp_y);
            wx = pair_w(a, at(hz, ly + 1, lx + 2), pin && has_px, sp_x);
        }
        wyb[(ly + 1) * 32 + lx] = wy;
        wxb[ly * 33 + lx + 1] = wx;
        __syncthreads();
        if (pin) {
            const unsigned v = (unsigned)gz * L.stride[0] + (unsigned)gy * L.stride[1] + (unsigned)gx;
            const double c0 = wz_back, c1 = wz, c3 = wy, c5 = wx;
            const double c2 = ly ? wyb[ly * 32 + lx] : s_wyh[lz * 32 + lx];
            const double c4 = lx ? wxb[ly * 33 + lx] : s_wxh[lz * 8 + ly];
            if (!cold) {
                S.cap[0][v] = (T)c0; S.cap[1][v] = (T)c1; S.cap[2][v] = (T)c2;
                S.cap[3][v] = (T)c3; S.cap[4][v] = (T)c4; S.cap[5][v] = (T)c5;
            }
            T tr = (T)0;
            const double mm = tlinks(cur, tr);
            const bool own = gz >= L.own0 && gz < L.own1;
            if (own) msum = __dadd_rn(msum, mm);
            if (!cold) S.tr[v] = tr;
            // ---- solver state (same arithmetic as k_init_tile) ----
            unsigned m = (c0 > 0 ? 1u : 0u) | (c1 > 0 ? 2u : 0u) | (c2 > 0 ? 4u : 0u) | (c3 > 0 ? 8u : 0u) |
                         (c4 > 0 ? 16u : 0u) | (c5 > 0 ? 32u : 0u);
            const double trd = (double)tr;
            double e = 0.0;
            if (!cold) {            // cold: tr <= 0 everywhere, so excess is 0 and never stored
                double out = __dadd_ru(0.0, c0);
                out = __dadd_ru(out, c1); out = __dadd_ru(out, c2); out = __dadd_ru(out, c3);
                out = __dadd_ru(out, c4); out = __dadd_ru(out, c5);
                if (trd > 0) { const double lim = out * SOURCE_CLAMP_SLACK; e = trd < lim ? trd : lim; if (!(out == out)) e = trd; }
                if (!own) e = 0.0;
                S.excess[v] = (T)e;
            }
            if (trd < 0) m |= RM_SINK;
            if (MODE != 2) {
                S.rmask[v] = (uint8_t)m;
                const int h = (own && trd < 0) ? 1 : MGC_HINF;
                S.height[v] = h;
                if (own && (m & 0x3fu) != 0 && h == MGC_HINF) needs_any = 1u;
            }
            if (e > 0) exc_any = 1u;
        }
        wz_back = wz;
        cur = nxt;
        // the planes of this step are read above; the next step writes the other buffer, the one after waits at its barrier
    }

    if (MODE == 2) return;
    // ---- per solver tile flags and worklists (a warp row covers four 8^3 tiles: lanes 8j .. 8j+7) ----
    const unsigned bn = __ballot_sync(0xffffffffu, needs_any != 0), be = __ballot_sync(0xffffffffu, exc_any != 0);
    if (lx == 0) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if ((bn >> (8 * j)) & 0xffu) atomicOr(&s_flags[j], 1);
            if ((be >> (8 * j)) & 0xffu) atomicOr(&s_flags[4 + j], 1);
        }
    }
    if (isbad) *bad = 1;
    // deterministic block sum of the add_tweights minima (fixed order: thread chain, warp shuffles, 8 warps)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) msum = __dadd_rn(msum, __shfl_down_sync(0xffffffffu, msum, o));
    if (lx == 0) s_red[ly] = msum;
    __syncthreads();
    if (tid == 0) {
        double t = s_red[0];
#pragma unroll
        for (int w = 1; w < 8; ++w) t = __dadd_rn(t, s_red[w]);
        partials[blk] = t;
        if (MODE == 1) {
            bflag[blk] = cold ? 0 : 1;
            if (!cold) atomicAdd(mcount, 1);
        }
    }
    if (tid < 4) {
        const int tx = (x0 >> 3) + tid, ty = y0 >> 3, tz = z0 >> 3;
        if (tx < TL.nt[2] && ty < TL.nt[1] && tz < TL.nt[0]) {
            const int t = (tz * TL.nt[1] + ty) * TL.nt[2] + tx;
            const int any_needs = s_flags[tid], any_exc = s_flags[4 + tid];
            rflag[t] = any_needs;
            if (any_needs) rl.items[atomicAdd(rl.count, 1)] = t;
            pflag[t] = any_exc;
            if (any_exc) {
                const WorkList& pl = ((tz + ty + tx) & 1) ? pl1 : pl0;
                pl.items[atomicAdd(pl.count, 1)] = t;
            }
        }
    }
}

template <typename E, typename T, int FN, int USE_MAX, int SPACING, int TIN = 0, int MODE = 0>
__global__ void __launch_bounds__(BUILD_THREADS)
k_build_tile(Lattice L, Tiles TL, State<T> S, const __grid_constant__ BuildMaps maps, BuildArgs A, BoundaryParams P,
             int* __restrict__ bad, double* __restrict__ partials, int* __restrict__ rflag, WorkList rl,
             int* __restrict__ pflag, WorkList pl0, WorkList pl1, int* __restrict__ bflag, int* __restrict__ mcount)
{
    build_block<E, T, FN, USE_MAX, SPACING, TIN, MODE>(L, TL, S, maps, A, P, bad, partials, rflag, rl, pflag, pl0, pl1, bflag,
                                                       mcount, blockIdx.x, blockIdx.y, A.z_tile0 + (int)blockIdx.z, true, 0u);
}

// Materialise the cold build blocks that the push passes of one colour can reach (gc_api.cu, push_color): every tile on
// the colour's list and each of its face neighbours -- a running tile writes flow only into those -- has its build
// block claimed (bflag 0 -> 1, one winner) and rebuilt in MODE 2 by the CTA that claimed it.  Persistent CTAs over the
// listed tiles; the push launch that follows on the stream sees every block complete.
template <typename E, typename T, int FN, int USE_MAX, int SPACING>
__global__ void __launch_bounds__(BUILD_THREADS)
k_build_materialise(Lattice L, Tiles TL, State<T> S, const __grid_constant__ BuildMaps maps, BuildArgs A, BoundaryParams P,
                    WorkList tiles, int* __restrict__ bflag, int* __restrict__ mcount)
{
    __shared__ int s_claim[8];
    __shared__ int s_n;
    const int n = *(volatile int*)tiles.count;
    const int nbx = (L.dim[2] + BUILD_TX - 1) / BUILD_TX, nby = (L.dim[1] + BUILD_TY - 1) / BUILD_TY;
    unsigned done = 0;                                   // blocks this CTA built so far (mbarrier phase)
    for (int i = blockIdx.x; i < n; i += gridDim.x) {
        const int t = tiles.items[i];
        if (threadIdx.x == 0) s_n = 0;
        __syncthreads();
        if (threadIdx.x < 7) {
            const int tx = t % TL.nt[2], r = t / TL.nt[2], ty = r % TL.nt[1], tz = r / TL.nt[1];
            const int k = threadIdx.x;           // 0..5: face neighbour across face k, 6: the tile itself
            int z = tz, y = ty, x = tx;
            if (k < 6) {
                const int d = (k & 1) ? 1 : -1;
                if ((k >> 1) == 0) z += d; else if ((k >> 1) == 1) y += d; else x += d;
            }
            if (z >= 0 && y >= 0 && x >= 0 && z < TL.nt[0] && y < TL.nt[1] && x < TL.nt[2]) {
                const int b = (z * nby + y) * nbx + (x >> 2);
                if (*(volatile int*)(bflag + b) == 0 && atomicCAS(bflag + b, 0, 1) == 0) {
                    s_claim[atomicAdd(&s_n, 1)] = b;
                    atomicAdd(mcount, 1);
                }
            }
        }
        __syncthreads();
        const int nc = s_n;
        for (int j = 0; j < nc; ++j) {
            const int b = s_claim[j];
            build_block<E, T, FN, USE_MAX, SPACING, 1, 2>(L, TL, S, maps, A, P, nullptr, nullptr, nullptr, WorkList{}, nullptr,
                                                          WorkList{}, WorkList{}, nullptr, nullptr, b % nbx, (b / nbx) % nby,
                                                          b / (nbx * nby), done == 0, done & 1u);
            ++done;
            __syncthreads();                     // staged inputs and weight planes are free for the next block
        }
    }
}

// Materialise every block that is still cold (readers that need the whole lattice): one CTA per build block.
template <typename E, typename T, int FN, int USE_MAX, int SPACING>
__global__ void __launch_bounds__(BUILD_THREADS)
k_build_materialise_all(Lattice L, Tiles TL, State<T> S, const __grid_constant__ BuildMaps maps, BuildArgs A, BoundaryParams P,
                        int* __restrict__ bflag, int* __restrict__ mcount)
{
    const int blk = ((int)blockIdx.z * (int)gridDim.y + (int)blockIdx.y) * (int)gridDim.x + (int)blockIdx.x;
    if (bflag[blk]) return;
    build_block<E, T, FN, USE_MAX, SPACING, 1, 2>(L, TL, S, maps, A, P, nullptr, nullptr, nullptr, WorkList{}, nullptr, WorkList{},
                                                  WorkList{}, nullptr, nullptr, blockIdx.x, blockIdx.y, blockIdx.z, true, 0u);
    if (threadIdx.x == 0) { bflag[blk] = 1; atomicAdd(mcount, 1); }
}

template <typename E>
constexpr size_t build_smem_bytes()
{
    return (size_t)BUILD_TIN_OFFSET((BUILD_HZ * BUILD_HY * BuildBox<E>::BX * (int)sizeof(E) + 127) / 128 * 128) +
           (size_t)BUILD_TZ * BUILD_TY * BUILD_TX * (8 + 1 + 1);
}

// ---------------------------------------------------------------------------------------------------
// marker volumes -> bit planes (device side; the host binding packs on the CPU for the end-to-end path so that the
// markers cross PCIe as 0.25 B/voxel instead of 2): bit (v & 31) of word (v >> 5) = marker[v] != 0
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pack_bits(const uint8_t* __restrict__ src, unsigned n, unsigned* __restrict__ dst)
{
    const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
    const bool on = v < n && src[v] != 0;
    const unsigned w = __ballot_sync(0xffffffffu, on);
    if ((threadIdx.x & 31) == 0 && v < n) dst[v >> 5] = w;
}
