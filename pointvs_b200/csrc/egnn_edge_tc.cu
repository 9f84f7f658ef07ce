// K2 edge stage on the 5th-generation tensor cores (PVS_MATH_BF16X3 / BF16).
//
// Same dataflow as egnn_edge_fwd_kernel (egnn_fwd.cu) but the two per-edge
// 64x64 contractions (edge_mlp.2 and coord_mlp.0; reference
// egnn_satorras.py:76-80, 88-96) run as tcgen05.mma tiles:
//
//   tile      : 128 dst-sorted edges (UMMA M = 128, cta_group::1), N = K = KW
//               (64; 128 for the forward at 64 < k <= 128, see TcCfg);
//               edge-packed (pvs_build_packed_tiles): tile t = edges
//               [128 t, 128 t + 128), nodes cut by a tile boundary go through
//               per-tile partial slots and edge_tile_fixup_kernel
//   A operand : activations written by the CTA's threads into shared memory in
//               the canonical K-major SWIZZLE_128B layout (one 128-byte row per
//               edge), as a bf16 hi tile and, for BF16X3, a bf16 lo tile
//   B operand : nn.Linear weight [out][in] = N x K, K-major, same layout,
//               split hi/lo once per CTA
//   D         : fp32 accumulators in tensor memory (2 x 64 columns)
//   BF16X3    : D = Ahi.Bhi + Alo.Bhi + Ahi.Blo (error ~2^-16, fp32-class);
//   BF16      : D = Ahi.Bhi
//   epilogue  : tcgen05.ld 32x32b -- each thread owns one edge row: bias, SiLU,
//               the 64->1 attention / coordinate heads as in-thread dot
//               products, and the next GEMM's A tile written straight back to
//               shared memory; the coordinate GEMM overlaps the message
//               segment-reduce.
//
// One persistent CTA per SM holds G independent 4-warp groups (5 in the
// error-compensated mode, 8 in the single-pass bf16 mode: see TcCfg).
// The groups share the weight tiles and each own an A-tile pair, 64 TMEM columns,
// an mbarrier and a named barrier; they walk different tiles and drift out of
// phase, so one group's gather latency hides behind another's MUFU-heavy
// epilogue (the first version, 3 CTAs x 4 warps per SM, issued on only 38 % of
// cycles with the gather as the top stall: profiles/r01_c_*).
#include <cstdlib>

#include "egnn_common.cuh"
#include "tc_common.cuh"

#ifndef PVS_EDGE_TC8_DEFAULT
#define PVS_EDGE_TC8_DEFAULT 0
#endif

namespace pvs {

constexpr int TC_GROUP_THREADS = 128;
// groups per CTA; -DPVS_EXP_GROUPS=n builds the concurrency experiment of
// profiles/README.md (capture F)
#ifndef PVS_EXP_GROUPS
#define PVS_EXP_GROUPS 5
#endif
// The error-compensated mode needs a hi and a lo A tile per group (37.9 KB with
// the per-group scalars): five groups fill the 227 KB of shared memory.  The
// single-pass bf16 mode has no lo tiles, so eight groups (1024 threads, all 512
// TMEM columns) fit.
// Arithmetic of the two per-edge GEMMs (template parameter MODE):
//   TCM_BF16   : A bf16, B bf16                 (fast mode, tanh.approx SiLU)
//   TCM_BF16X3 : Ahi.Bhi + Alo.Bhi + Ahi.Blo    (bf16 hi/lo of both operands)
//   TCM_FP16X2 : A16.Bhi + A16.Blo              (activations as ONE fp16 tile,
//                weights as fp16 hi + lo).  Rounding the activations to 11 bits
//                costs ~3e-6 on the scores (the fp32 path itself is at 1e-6;
//                bf16 activations would cost 3e-5) and frees the lo tile.
enum { TCM_BF16 = 0, TCM_BF16X3 = 1, TCM_FP16X2 = 2 };
// KW = padded hidden width of the tile: 64 (k <= 64) or 128 (65 <= k <= 128,
// forward only).  At KW = 128 a K-major operand is two SWIZZLE_128B K-blocks of
// 64 channels, the weights take four times the shared memory and a group
// needs 128 TMEM columns, so fewer groups fit: bf16x3 128 KB of weight tiles +
// 64 KB of A tiles per group -> 1 group; fp16x2 128 + 32 -> 2; bf16 64 + 32 -> 4.
template <int MODE, int KW = 64> struct TcCfg {
    static constexpr bool A_LO = MODE == TCM_BF16X3;      // second activation tile
    static constexpr bool B_LO = MODE != TCM_BF16;        // second weight tile
    static constexpr bool F16 = MODE == TCM_FP16X2;
    static constexpr bool EXACT_SILU = MODE != TCM_BF16;
    static constexpr int GROUPS = KW == 64 ? (A_LO ? PVS_EXP_GROUPS : 8)
                                           : (A_LO ? 1 : (B_LO ? 2 : 4));
    static constexpr int THREADS = TC_GROUP_THREADS * GROUPS;
    static constexpr int KB = KW / 64;                    // 64-channel K-blocks
};
constexpr uint32_t TC_TMEM_COLS = 512;   // whole TMEM: one CTA per SM
// a group's TMEM columns: KW (D1 and D2 alias, never live together)

// byte offset of 16-byte chunk `c` (channels 8c..8c+7) of row `r` in a
// [KW / 64][rows][128 B] tile of K-blocks with `rows` rows each
template <int KW, int ROWS = TE>
__device__ __forceinline__ uint32_t swzk(int r, int c) {
    if constexpr (KW == 64) return swz(r, c);
    else return (uint32_t)((c >> 3) * (ROWS * 128)) + swz(r, c & 7);
}

#ifdef PVS_PHASE_PROF
// Debug build only (scripts/phase_prof.py): cycles each group spends between
// the phase boundaries of a tile, summed over all groups and tiles.
__device__ unsigned long long g_phase_cycles[16];
#define PHASE_MARK(i)                                                         \
    do {                                                                      \
        if (tid == 0) {                                                       \
            const long long now_ = clock64();                                 \
            atomicAdd(&g_phase_cycles[i], (unsigned long long)(now_ - t_prev_)); \
            t_prev_ = now_;                                                   \
        }                                                                     \
    } while (0)
#else
#define PHASE_MARK(i) do { } while (0)
#endif

struct TcGroupMisc {
    float e_rad[TE], e_dx[TE], e_dy[TE], e_dz[TE], e_z[TE], e_c[TE];
    int e_col[TE];
    uint8_t e_rowl[TE], e_attr[TE];
    int rp[TN + 1];
    float xsum[TN][3];
    int split_lo, split_hi;   // first / last node of the window crosses the tile's edge range
    uint64_t mbar;
};

template <int MODE, int KW = 64>
struct __align__(1024) TcSmem {
    static constexpr int G = TcCfg<MODE, KW>::GROUPS, KB = KW / 64;
    static constexpr bool X3 = TcCfg<MODE, KW>::A_LO, BLO = TcCfg<MODE, KW>::B_LO;
    // swizzled bf16 tiles, each 1024-byte aligned (lo tiles only where used);
    // K-block b of a tile starts at b * rows * 128 bytes
    uint8_t A_hi[G][KB * TE * 128];
    uint8_t A_lo[X3 ? G : 1][X3 ? KB * TE * 128 : 1024];
    uint8_t W2_hi[KB * KW * 128];
    uint8_t W2_lo[BLO ? KB * KW * 128 : 1024];
    uint8_t Wc1_hi[KB * KW * 128];
    uint8_t Wc1_lo[BLO ? KB * KW * 128 : 1024];
    float b2[KW], bc1[KW], wc2[KW], wa[KW], wr[KW];
    float T[PVS_MAX_EDGE_CLASSES][KW];
    TcGroupMisc grp[G];
    uint32_t tmem_base;
};

// barrier among the 128 threads of one group (id 0 is __syncthreads)
__device__ __forceinline__ void group_sync(int g) {
    asm volatile("bar.sync %0, %1;" ::"r"(g + 1), "n"(TC_GROUP_THREADS) : "memory");
}

// one 128 x KW x KW GEMM into TMEM columns [d_col, d_col + KW)
template <int MODE, int KW = 64>
__device__ __forceinline__ void issue_gemm(uint32_t tmem_base, uint32_t d_col,
                                           const uint8_t *a_hi, const uint8_t *a_lo,
                                           const uint8_t *b_hi, const uint8_t *b_lo,
                                           uint64_t *bar) {
    const uint32_t d = tmem_base + d_col;
    constexpr uint32_t idesc = tc_idesc(KW, TcCfg<MODE, KW>::F16);
    uint32_t acc = 0;
#pragma unroll
    for (int kb = 0; kb < KW / 64; ++kb) {
        const uint64_t ah = make_desc(smem_u32(a_hi + kb * TE * 128));
        const uint64_t al = make_desc(smem_u32(a_lo + kb * TE * 128));
        const uint64_t bh = make_desc(smem_u32(b_hi + kb * KW * 128));
        const uint64_t bl = make_desc(smem_u32(b_lo + kb * KW * 128));
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            const uint64_t adv = (uint64_t)(ks * 2);   // 16 elements = 32 B = 2 x 16 B
            umma_bf16(d, ah + adv, bh + adv, idesc, acc);
            acc = 1;
            if (TcCfg<MODE, KW>::A_LO) umma_bf16(d, al + adv, bh + adv, idesc, 1);
            if (TcCfg<MODE, KW>::B_LO) umma_bf16(d, ah + adv, bl + adv, idesc, 1);
        }
    }
    umma_commit(bar);
}

template <int MODE, int KW>
__global__ void __launch_bounds__(TcCfg<MODE, KW>::THREADS, 1)
egnn_edge_tc_kernel(const EdgeArgs a) {
    // SWIZZLE_128B tiles need 1024-byte alignment; the kernel has no static
    // shared memory, so the dynamic window starts at its (aligned) base.
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    pdl_launch_dependents();
    constexpr int TC_GROUPS = TcCfg<MODE, KW>::GROUPS, TC_THREADS = TcCfg<MODE, KW>::THREADS;
    constexpr bool X3 = TcCfg<MODE, KW>::A_LO;        // hi + lo activation tiles
    constexpr bool F16 = TcCfg<MODE, KW>::F16;        // fp16 operands
    constexpr bool EXACT = TcCfg<MODE, KW>::EXACT_SILU;
    constexpr int KB = KW / 64, TC_K = KW;
    TcSmem<MODE, KW> &S = *reinterpret_cast<TcSmem<MODE, KW> *>(smem_dyn);
    if ((smem_u32(smem_dyn) & 1023u) != 0u) __trap();
    const int g = threadIdx.x / TC_GROUP_THREADS;          // group
    const int tid = threadIdx.x % TC_GROUP_THREADS;        // thread in group
    const int lane = tid & 31, warp = tid >> 5;            // warp in group
    TcGroupMisc &Gm = S.grp[g];
    uint8_t *A_hi = S.A_hi[g], *A_lo = S.A_lo[X3 ? g : 0];
    const int k = a.k;
    const bool f_att = a.flags & PVS_F_EDGE_ATTENTION;
    const bool f_softmax = f_att && (a.flags & PVS_F_SOFTMAX_ATTENTION);
    const bool f_coords = (a.flags & PVS_F_UPDATE_COORDS) && a.x_out != nullptr;
    const bool f_eres = (a.flags & PVS_F_EDGE_RESIDUAL) && a.m_prev != nullptr;

    // ---- one-time setup (whole CTA) ----
    if constexpr (KW == 64) {
        if (F16) {
            load_weight_tiles_f16(S.W2_hi, S.W2_lo, a.edge_w2, k, k, k);
            load_weight_tiles_f16(S.Wc1_hi, S.Wc1_lo, a.coord_w1, k, k, k);
        } else {
            load_weight_tiles<X3>(S.W2_hi, S.W2_lo, a.edge_w2, k, k, k);
            load_weight_tiles<X3>(S.Wc1_hi, S.Wc1_lo, a.coord_w1, k, k, k);
        }
    } else {
        // K-block b: input channels [64 b, 64 b + 64) of all KW output rows
        for (int b = 0; b < KB; ++b) {
            const int o = b * KW * 128;
            if (F16) {
                load_weight_tiles_f16(S.W2_hi + o, S.W2_lo + o, a.edge_w2 + 64 * b, k, k,
                                      k - 64 * b, KW);
                load_weight_tiles_f16(S.Wc1_hi + o, S.Wc1_lo + o, a.coord_w1 + 64 * b, k, k,
                                      k - 64 * b, KW);
            } else {
                load_weight_tiles<X3>(S.W2_hi + o, S.W2_lo + (X3 ? o : 0),
                                      a.edge_w2 + 64 * b, k, k, k - 64 * b, KW);
                load_weight_tiles<X3>(S.Wc1_hi + o, S.Wc1_lo + (X3 ? o : 0),
                                      a.coord_w1 + 64 * b, k, k, k - 64 * b, KW);
            }
        }
    }
    const int col_r = (a.flags & PVS_F_PERM_INVARIANT) ? k : 2 * k;
    for (int n = threadIdx.x; n < KW; n += TC_THREADS) {
        const bool ok = n < k;
        S.b2[n] = ok ? a.edge_b2[n] : 0.0f;
        S.bc1[n] = ok ? a.coord_b1[n] : 0.0f;
        S.wc2[n] = ok ? a.coord_w2[n] : 0.0f;
        S.wa[n] = (ok && a.att_w) ? a.att_w[n] : 0.0f;
        S.wr[n] = ok ? a.edge_w1[(size_t)n * a.in_e + col_r] : 0.0f;
        for (int c = 0; c < PVS_MAX_EDGE_CLASSES; ++c)
            S.T[c][n] = (ok && c < a.n_classes)
                            ? a.edge_w1[(size_t)n * a.in_e + col_r + 1 + c] : 0.0f;
    }
    if (tid == 0) mbar_init(&Gm.mbar, 1);
    if (threadIdx.x < 32) tmem_alloc<TC_TMEM_COLS>(&S.tmem_base);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = S.tmem_base;
    const uint32_t tmem_grp = tmem_base + (uint32_t)g * (uint32_t)KW;
    const uint32_t tmem_lane = tmem_grp + ((uint32_t)(warp * 32) << 16);
    uint32_t phase = 0;
    const float att_b = (f_att && a.att_b) ? a.att_b[0] : 0.0f;
    float gate = 1.0f;
    if (f_eres && a.edge_gate) gate = a.edge_gate[0];
    const int n_tiles = *a.n_ptiles;
#ifdef PVS_PHASE_PROF
    long long t_prev_ = clock64();
#endif

    // Edge-packed tiles: tile t owns edges [128 t, 128 t + 128) and the nodes
    // from the one after the previous tile's last node (or that node itself
    // when its edges continue here) to the node of its own last edge.  A node
    // cut by a tile boundary leaves its partial sums in Mpart / xpart; the
    // fix-up kernel adds them in tile order.  Runs of edgeless nodes can make
    // the node range longer than the shared-memory window: it is then walked
    // 128 nodes at a time.
    const int E_total = a.row_ptr[a.n_nodes];
    // Round 2: the dependent chain ptile_last -> row_ptr -> col -> x[j] at the
    // top of a tile cost 15 % of a group's time (profiles/README.md).  The
    // tile's cover (previous / own last node, row_ptr of the node after the
    // previous tile's last) is now loaded one tile ahead into three registers,
    // and col / attr of the tile's own edge are requested before the row_ptr
    // window instead of after it.
    // (Only in the 96-register error-compensated mode: at 64 registers the
    // three extra live values spill and cost 5 %.)
    constexpr bool PF = X3;
    const int t_stride = gridDim.x * TC_GROUPS;
    int pf_na = -1, pf_nb = 0, pf_rpn = 0;
    if (PF) {
        const int t0 = blockIdx.x * TC_GROUPS + g;
        if (t0 < n_tiles) {
            if (t0 > 0) { pf_na = a.ptile_last[t0 - 1]; pf_rpn = a.row_ptr[pf_na + 1]; }
            pf_nb = a.ptile_last[t0];
        }
    }
    pdl_wait();      // P, Q, x, m_prev of the kernels before this one
    for (int t = blockIdx.x * TC_GROUPS + g; t < n_tiles; t += t_stride) {
        const int E0 = t * TE, E1 = min(E0 + TE, E_total);
        if (!PF) {
            if (t > 0) { pf_na = a.ptile_last[t - 1]; pf_rpn = a.row_ptr[pf_na + 1]; }
            pf_nb = a.ptile_last[t];
        }
        const int cover_lo = t > 0 ? (pf_rpn > E0 ? pf_na : pf_na + 1) : 0;
        const int cover_hi = (t == n_tiles - 1) ? a.n_nodes - 1 : pf_nb;
        // this thread's edge of the tile (first node window: c0 == E0)
        int my_col = 0, my_attr = 0;
        if (PF && E0 + tid < E1) {
            my_col = a.col[E0 + tid];
            my_attr = a.attr ? a.attr[E0 + tid] : 0;
        }
        // cover of the group's next tile (used at the top of the next iteration)
        const int tn = t + t_stride;
        bool rpn_pending = PF && tn < n_tiles;
        if (PF && tn < n_tiles) {
            pf_na = a.ptile_last[tn - 1];
            pf_nb = a.ptile_last[tn];
        }
        for (int n0 = cover_lo; n0 <= cover_hi; n0 += TN) {
        const int nn = min(TN, cover_hi - n0 + 1);
        group_sync(g);
        for (int i = tid; i <= nn; i += TC_GROUP_THREADS) {
            const int v = a.row_ptr[n0 + i];
            Gm.rp[i] = min(max(v, E0), E1);
            if (i == 0) Gm.split_lo = v < E0;
            if (i == nn) Gm.split_hi = v > E1;
        }
        for (int i = tid; i < nn * 3; i += TC_GROUP_THREADS) (&Gm.xsum[0][0])[i] = 0.0f;
        group_sync(g);
        const int e0 = Gm.rp[0], e1 = Gm.rp[nn];
        {
            const int c0 = e0;
            const int ne = e1 - e0;      // <= 128: one MMA tile
            if (ne > 0) {
                // ---- stage 0: geometry, one thread per edge ----
                if (tid < ne) {
                    const int e = c0 + tid;
                    int lo = 0, hi = nn;
                    while (hi - lo > 1) {
                        int mid = (lo + hi) >> 1;
                        if (Gm.rp[mid] <= e) lo = mid; else hi = mid;
                    }
                    const bool own = PF && c0 == E0;   // first window: hoisted loads
                    const int i = n0 + lo, j = own ? my_col : a.col[e];
                    float dx = a.x_in[3 * i] - a.x_in[3 * j];
                    float dy = a.x_in[3 * i + 1] - a.x_in[3 * j + 1];
                    float dz = a.x_in[3 * i + 2] - a.x_in[3 * j + 2];
                    float r = dx * dx + dy * dy + dz * dz;
                    if (a.flags & PVS_F_NORMALIZE) {
                        float inv = 1.0f / (sqrtf(r) + 1e-8f);
                        dx *= inv; dy *= inv; dz *= inv;
                    }
                    Gm.e_rowl[tid] = (uint8_t)lo;
                    Gm.e_col[tid] = j;
                    Gm.e_attr[tid] = own ? my_attr : (a.attr ? a.attr[e] : 0);
                    Gm.e_rad[tid] = r;
                    Gm.e_dx[tid] = dx; Gm.e_dy[tid] = dy; Gm.e_dz[tid] = dz;
                }
                group_sync(g);
                PHASE_MARK(0);
                // ---- stage 1: s1 = silu(P_i + Q_j + w_r r + T[a]) -> A tile.
                // 8 lanes per edge row (one 16-byte chunk each), 16 rows a pass:
                // every LDG.128 warp instruction reads 4 full 256-byte rows.
                // The loads are unconditional (rows past the chunk end repeat
                // its last row; nobody reads what they produce) and run three
                // passes ahead of the arithmetic, so a pass never waits for
                // its own gather.
                // (KW = 128: one sweep per 64-channel K-block)
#pragma unroll 1
                for (int kb = 0; kb < KB; ++kb) {
                    const int c = (tid & 7) + 8 * kb, slot = tid >> 3;
                    float2 wr2[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        wr2[i] = *reinterpret_cast<const float2 *>(&S.wr[8 * c + 2 * i]);
                    constexpr int DEPTH = 3, PASSES = TE / 16;
                    float4 buf[DEPTH][4];
                    float radv[DEPTH];
                    int attv[DEPTH];
                    auto issue = [&](int p, float4 (&bq)[4], float &rad, int &at) {
                        const int r = min(p * 16 + slot, ne - 1);
                        const float4 *pp = reinterpret_cast<const float4 *>(
                            a.P + (size_t)(n0 + Gm.e_rowl[r]) * TC_K + 8 * c);
                        const float4 *qq = reinterpret_cast<const float4 *>(
                            a.Q + (size_t)Gm.e_col[r] * TC_K + 8 * c);
                        bq[0] = __ldg(pp); bq[1] = __ldg(pp + 1);
                        bq[2] = __ldg(qq); bq[3] = __ldg(qq + 1);
                        rad = Gm.e_rad[r];
                        at = Gm.e_attr[r];
                    };
                    auto finish = [&](int p, const float4 (&bq)[4], float rad, int at) {
                        const int r = p * 16 + slot;
                        const float2 rad2 = make_float2(rad, rad);
                        const float4 *t4 = reinterpret_cast<const float4 *>(&S.T[at][8 * c]);
                        const float4 ta = t4[0], tb = t4[1];
                        const float2 pv[4] = {make_float2(bq[0].x, bq[0].y), make_float2(bq[0].z, bq[0].w),
                                              make_float2(bq[1].x, bq[1].y), make_float2(bq[1].z, bq[1].w)};
                        const float2 qv[4] = {make_float2(bq[2].x, bq[2].y), make_float2(bq[2].z, bq[2].w),
                                              make_float2(bq[3].x, bq[3].y), make_float2(bq[3].z, bq[3].w)};
                        const float2 tv[4] = {make_float2(ta.x, ta.y), make_float2(ta.z, ta.w),
                                              make_float2(tb.x, tb.y), make_float2(tb.z, tb.w)};
                        float2 v[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            v[i] = ffma2(wr2[i], rad2, fadd2(fadd2(pv[i], qv[i]), tv[i]));
                        silu4_mode<EXACT>(v[0], v[1]);
                        silu4_mode<EXACT>(v[2], v[3]);
                        if (F16) {
                            *reinterpret_cast<uint4 *>(A_hi + swzk<KW>(r, c)) = pack8_f16(v);
                        } else {
                            uint4 hi, lo;
                            split8p<X3>(v, hi, lo);
                            *reinterpret_cast<uint4 *>(A_hi + swzk<KW>(r, c)) = hi;
                            if (X3) *reinterpret_cast<uint4 *>(A_lo + swzk<KW>(r, c)) = lo;
                        }
                    };
#pragma unroll
                    for (int p = 0; p < DEPTH; ++p) issue(p, buf[p], radv[p], attv[p]);
#pragma unroll
                    for (int p = 0; p < PASSES; ++p) {
                        finish(p, buf[p % DEPTH], radv[p % DEPTH], attv[p % DEPTH]);
                        if (p + DEPTH < PASSES)
                            issue(p + DEPTH, buf[p % DEPTH], radv[p % DEPTH], attv[p % DEPTH]);
                    }
                }
                if (rpn_pending) {       // pf_na has landed by now
                    pf_rpn = a.row_ptr[pf_na + 1];
                    rpn_pending = false;
                }
                fence_proxy_async();
                tc_fence_before();
                group_sync(g);
                PHASE_MARK(1);
                // ---- GEMM 1: t2 = s1 . W2^T ----
                if (tid == 0) {
                    tc_fence_after();
                    issue_gemm<MODE, KW>(tmem_grp, 0, A_hi, A_lo, S.W2_hi, S.W2_lo, &Gm.mbar);
                }
                mbar_wait(&Gm.mbar, phase);
                phase ^= 1;
                tc_fence_after();
                PHASE_MARK(2);
                // ---- epilogue 1: m = silu(t2 + b2) (+ edge residual), the
                // attention logit, and m back into the A tile for GEMM 2 ----
                {
                    const int r = tid;
                    float2 dot2 = make_float2(0.0f, 0.0f);
#pragma unroll 1
                    for (int q = 0; q < KW / 16; ++q) {
                        float acc[16];
                        tmem_ld16(tmem_lane + 16 * q, acc);
#pragma unroll
                        for (int hlf = 0; hlf < 2; ++hlf) {
                            const int nb = 16 * q + 8 * hlf;
                            const float4 *b4 = reinterpret_cast<const float4 *>(&S.b2[nb]);
                            const float4 *w4 = reinterpret_cast<const float4 *>(&S.wa[nb]);
                            const float4 ba = b4[0], bb = b4[1], wa0 = w4[0], wa1 = w4[1];
                            const float2 bias[4] = {make_float2(ba.x, ba.y), make_float2(ba.z, ba.w),
                                                    make_float2(bb.x, bb.y), make_float2(bb.z, bb.w)};
                            const float2 wat[4] = {make_float2(wa0.x, wa0.y), make_float2(wa0.z, wa0.w),
                                                   make_float2(wa1.x, wa1.y), make_float2(wa1.z, wa1.w)};
                            // Padded channels (n >= k) need no masking: their
                            // weight rows and biases are zero, so m = silu(0) = 0.
                            // Rows >= ne hold values nobody reads.
                            float2 mv[4];
#pragma unroll
                            for (int i = 0; i < 4; ++i)
                                mv[i] = fadd2(
                                    make_float2(acc[8 * hlf + 2 * i], acc[8 * hlf + 2 * i + 1]),
                                    bias[i]);
                            silu4_mode<EXACT>(mv[0], mv[1]);
                            silu4_mode<EXACT>(mv[2], mv[3]);
                            if (f_eres && r < ne) {
#pragma unroll
                                for (int i = 0; i < 8; ++i) {
                                    const int n = nb + i;
                                    if (n < k) {
                                        float &mref = (i & 1) ? mv[i >> 1].y : mv[i >> 1].x;
                                        float mp = a.m_prev[(size_t)(c0 + r) * k + n];
                                        if (a.flags & PVS_F_REZERO) mref = mp + gate * mref;
                                        else if (a.flags & PVS_F_GATED_RESIDUAL) {
                                            float gg = fmaxf(gate, 0.0f);
                                            mref = gg * mref + (1.0f - gg) * mp;
                                        } else mref = mref + mp;
                                    }
                                }
                            }
#pragma unroll
                            for (int i = 0; i < 4; ++i) dot2 = ffma2(wat[i], mv[i], dot2);
                            const int c = 2 * q + hlf;
                            if (F16) {
                                *reinterpret_cast<uint4 *>(A_hi + swzk<KW>(r, c)) = pack8_f16(mv);
                            } else {
                                uint4 hi, lo;
                                split8p<X3>(mv, hi, lo);
                                *reinterpret_cast<uint4 *>(A_hi + swzk<KW>(r, c)) = hi;
                                if (X3) *reinterpret_cast<uint4 *>(A_lo + swzk<KW>(r, c)) = lo;
                            }
                        }
                    }
                    const float dot = dot2.x + dot2.y;
                    // attention value per edge (alpha, or the raw logit when
                    // a softmax pass follows)
                    float al = 1.0f;
                    if (f_att) {
                        const float z = dot + att_b;
                        al = f_softmax ? z : apply_act(z, a.att_act);
                        if (a.att_out && r < ne) a.att_out[c0 + r] = al;
                    }
                    Gm.e_z[r] = al;
                }
                fence_proxy_async();
                tc_fence_before();
                group_sync(g);
                PHASE_MARK(3);
                // ---- GEMM 2 (coordinate MLP; reuses the D columns, which
                // epilogue 1 has fully read) runs while the messages are
                // reduced below ----
                if (f_coords && tid == 0) {
                    tc_fence_after();
                    issue_gemm<MODE, KW>(tmem_grp, 0, A_hi, A_lo, S.Wc1_hi, S.Wc1_lo, &Gm.mbar);
                }
            }
            // ---- M_i = sum_e alpha_e m_e over dst segments: a warp per node,
            // four edges a step (8 lanes per edge row, one 16-byte chunk of the
            // hi and of the lo tile each), partial sums folded by two shuffles.
            // The order of the additions is fixed, so the sums are reproducible.
            if (!f_softmax) {
                const int es = lane >> 3;
#pragma unroll 1
                for (int kb = 0; kb < KB; ++kb) {
                const int cc = (lane & 7) + 8 * kb;
                for (int nl = warp; nl < nn; nl += TC_GROUP_THREADS / 32) {
                    const int lo = Gm.rp[nl] - c0, hi = Gm.rp[nl + 1] - c0;
                    float2 s[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) s[i] = make_float2(0.0f, 0.0f);
                    for (int el = lo + es; el < hi; el += 4) {
                        const uint32_t off = swzk<KW>(el, cc);
                        const uint4 h = *reinterpret_cast<const uint4 *>(A_hi + off);
                        const float al = Gm.e_z[el];
                        const float2 al2 = make_float2(al, al);
                        const uint32_t hw[4] = {h.x, h.y, h.z, h.w};
                        float2 m[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            m[i] = F16 ? unpack_f16x2(hw[i])
                                       : make_float2(__uint_as_float(hw[i] << 16),
                                                     __uint_as_float(hw[i] & 0xffff0000u));
                        if (X3) {
                            const uint4 l = *reinterpret_cast<const uint4 *>(A_lo + off);
                            const uint32_t lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
                            for (int i = 0; i < 4; ++i)
                                m[i] = fadd2(m[i], make_float2(__uint_as_float(lw[i] << 16),
                                                               __uint_as_float(lw[i] & 0xffff0000u)));
                        }
#pragma unroll
                        for (int i = 0; i < 4; ++i) s[i] = ffma2(al2, m[i], s[i]);
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        s[i].x += __shfl_xor_sync(0xffffffffu, s[i].x, 8);
                        s[i].y += __shfl_xor_sync(0xffffffffu, s[i].y, 8);
                        s[i].x += __shfl_xor_sync(0xffffffffu, s[i].x, 16);
                        s[i].y += __shfl_xor_sync(0xffffffffu, s[i].y, 16);
                    }
                    float *row = a.M + (size_t)(n0 + nl) * TC_K;
                    if (nl == 0 && Gm.split_lo) row = a.Mpart + ((size_t)t * 2) * TC_K;
                    else if (nl == nn - 1 && Gm.split_hi) row = a.Mpart + ((size_t)t * 2 + 1) * TC_K;
                    if (es == 0) {
                        float4 *dst = reinterpret_cast<float4 *>(row + 8 * cc);
                        dst[0] = make_float4(s[0].x, s[0].y, s[1].x, s[1].y);
                        dst[1] = make_float4(s[2].x, s[2].y, s[3].x, s[3].y);
                    }
                }
                }   // K-blocks
            }
            // ---- messages out (edge residual of the next layer / softmax) ----
            if (a.m_out != nullptr) {
                for (int idx = tid; idx < ne * (TC_K / 2); idx += TC_GROUP_THREADS) {
                    const int el = idx / (TC_K / 2), w = idx % (TC_K / 2);
                    const uint32_t off = swzk<KW>(el, w >> 2) + ((w & 3) << 2);
                    const uint32_t h = *reinterpret_cast<const uint32_t *>(A_hi + off);
                    float m0 = __uint_as_float(h << 16);
                    float m1 = __uint_as_float(h & 0xffff0000u);
                    if (F16) {
                        const float2 mf = unpack_f16x2(h);
                        m0 = mf.x;
                        m1 = mf.y;
                    }
                    if (X3) {
                        const uint32_t l = *reinterpret_cast<const uint32_t *>(A_lo + off);
                        m0 += __uint_as_float(l << 16);
                        m1 += __uint_as_float(l & 0xffff0000u);
                    }
                    float *dst = a.m_out + (size_t)(c0 + el) * a.ld_m;
                    if (2 * w < a.ld_m) dst[2 * w] = m0;
                    if (2 * w + 1 < a.ld_m) dst[2 * w + 1] = m1;
                }
            }
            PHASE_MARK(4);
            if (ne > 0 && f_coords) {
                // ---- epilogue 2: c = [tanh](wc2 . silu(Wc1 m + bc1)) ----
                mbar_wait(&Gm.mbar, phase);
                phase ^= 1;
                tc_fence_after();
                PHASE_MARK(5);
                float2 d2 = make_float2(0.0f, 0.0f);
#pragma unroll 1
                for (int q = 0; q < KW / 16; ++q) {
                    float acc[16];
                    tmem_ld16(tmem_lane + 16 * q, acc);
#pragma unroll
                    for (int v4 = 0; v4 < 4; ++v4) {
                        const float4 bb = *reinterpret_cast<const float4 *>(&S.bc1[16 * q + 4 * v4]);
                        const float4 ww = *reinterpret_cast<const float4 *>(&S.wc2[16 * q + 4 * v4]);
                        float2 s0 = fadd2(make_float2(acc[4 * v4], acc[4 * v4 + 1]),
                                          make_float2(bb.x, bb.y));
                        float2 s1 = fadd2(make_float2(acc[4 * v4 + 2], acc[4 * v4 + 3]),
                                          make_float2(bb.z, bb.w));
                        silu4_mode<EXACT>(s0, s1);
                        d2 = ffma2(make_float2(ww.x, ww.y), s0, d2);
                        d2 = ffma2(make_float2(ww.z, ww.w), s1, d2);
                    }
                }
                const float dot = d2.x + d2.y;
                Gm.e_c[tid] = (a.flags & PVS_F_TANH) ? tanhf(dot) : dot;
                tc_fence_before();
            }
            group_sync(g);
            PHASE_MARK(6);
            // ---- coordinate messages summed per node ----
            if (f_coords && tid < nn) {
                const int lo = max(Gm.rp[tid], c0) - c0;
                const int hi = min(Gm.rp[tid + 1], c0 + TE) - c0;
                float sx = 0.f, sy = 0.f, sz = 0.f;
                for (int el = lo; el < hi; ++el) {
                    const float c = Gm.e_c[el];
                    sx = fmaf(Gm.e_dx[el], c, sx);
                    sy = fmaf(Gm.e_dy[el], c, sy);
                    sz = fmaf(Gm.e_dz[el], c, sz);
                }
                Gm.xsum[tid][0] += sx;
                Gm.xsum[tid][1] += sy;
                Gm.xsum[tid][2] += sz;
            }
            group_sync(g);
            PHASE_MARK(7);
        }
        if (a.x_out != nullptr && tid < nn) {
            const int i = n0 + tid;
            const bool sp_lo = tid == 0 && Gm.split_lo;
            const bool sp_hi = tid == nn - 1 && Gm.split_hi;
            if (sp_lo || sp_hi) {
                float *xp = a.xpart + ((size_t)t * 2 + (sp_lo ? 0 : 1)) * 4;
                xp[0] = Gm.xsum[tid][0];
                xp[1] = Gm.xsum[tid][1];
                xp[2] = Gm.xsum[tid][2];
            } else {
                const int cnt = Gm.rp[tid + 1] - Gm.rp[tid];
                const float inv = 1.0f / (float)(cnt > 0 ? cnt : 1);
                float ax = 0.f, ay = 0.f, az = 0.f;
                if (f_coords) {
                    ax = Gm.xsum[tid][0] * inv;
                    ay = Gm.xsum[tid][1] * inv;
                    az = Gm.xsum[tid][2] * inv;
                }
                a.x_out[3 * i] = a.x_in[3 * i] + ax;
                a.x_out[3 * i + 1] = a.x_in[3 * i + 1] + ay;
                a.x_out[3 * i + 2] = a.x_in[3 * i + 2] + az;
            }
        }
        }   // node windows of the tile
        if (rpn_pending) pf_rpn = a.row_ptr[pf_na + 1];
    }
    // ---- teardown ----
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc<TC_TMEM_COLS>(tmem_base);
}

// Nodes cut by tile boundaries: the tile where such a node STARTS owns its
// reduction and adds the partials of the following tiles in tile order.
template <int KW>
__global__ void __launch_bounds__(256)
edge_tile_fixup_kernel(const EdgeArgs a, int do_m, int do_x) {
    constexpr int TC_K = KW;
    pdl_launch_dependents();
    pdl_wait();
    const int t = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int n_tiles = *a.n_ptiles;
    if (t >= n_tiles - 1) return;                  // the last tile has no successor
    const int E_total = a.row_ptr[a.n_nodes];
    const int E0 = t * TE, E1 = min(E0 + TE, E_total);
    const int b = a.ptile_last[t];
    const int eb0 = a.row_ptr[b], eb1 = a.row_ptr[b + 1];
    if (eb1 <= E1) return;                         // the node ends in this tile
    if (eb0 < E0) return;                          // it started earlier: not the owner
    // (KW = 128: a lane sums two channel pairs, 2 lane and 64 + 2 lane)
    float2 s[KW / 64];
    float xs = 0.f;
#pragma unroll
    for (int h = 0; h < KW / 64; ++h) {
        s[h] = make_float2(0.f, 0.f);
        if (do_m)
            s[h] = *reinterpret_cast<const float2 *>(a.Mpart + ((size_t)t * 2 + 1) * TC_K + 64 * h +
                                                     2 * lane);
    }
    if (do_x && lane < 3) xs = a.xpart[((size_t)t * 2 + 1) * 4 + lane];
    for (int tt = t + 1; tt < n_tiles; ++tt) {
        if (do_m) {
#pragma unroll
            for (int h = 0; h < KW / 64; ++h) {
                const float2 p = *reinterpret_cast<const float2 *>(
                    a.Mpart + ((size_t)tt * 2) * TC_K + 64 * h + 2 * lane);
                s[h].x += p.x;
                s[h].y += p.y;
            }
        }
        if (do_x && lane < 3) xs += a.xpart[((size_t)tt * 2) * 4 + lane];
        if (eb1 <= min((tt + 1) * TE, E_total)) break;
    }
    if (do_m)
#pragma unroll
        for (int h = 0; h < KW / 64; ++h)
            *reinterpret_cast<float2 *>(a.M + (size_t)b * TC_K + 64 * h + 2 * lane) = s[h];
    if (do_x && lane < 3)
        a.x_out[3 * b + lane] = a.x_in[3 * b + lane] + xs / (float)(eb1 - eb0);
}

#ifdef PVS_PHASE_PROF
extern "C" int pvs_debug_phase_cycles(unsigned long long *out, int reset) {
    cudaDeviceSynchronize();
    if (out) cudaMemcpyFromSymbol(out, g_phase_cycles, sizeof(g_phase_cycles));
    if (reset) {
        unsigned long long z[16] = {0};
        cudaMemcpyToSymbol(g_phase_cycles, z, sizeof(z));
    }
    return 0;
}
#endif

template <int MODE, int KW = 64>
static int launch_mode(const EdgeArgs &a, int n_ptiles_cap, cudaStream_t st) {
    constexpr int G = TcCfg<MODE, KW>::GROUPS;
    static_assert(sizeof(TcSmem<MODE, KW>) <= 227 * 1024, "shared memory of one CTA");
    static_assert(G * KW <= (int)TC_TMEM_COLS, "TMEM columns of one CTA");
    const size_t smem = sizeof(TcSmem<MODE, KW>);
    int grid = num_sms();   // one persistent CTA per SM
    const int need = (n_ptiles_cap + G - 1) / G;
    if (need < grid) grid = need;
    if (grid < 1) grid = 1;
    const int rc = ensure_smem(egnn_edge_tc_kernel<MODE, KW>, smem);
    if (rc) return rc;
    if (launch_chained(egnn_edge_tc_kernel<MODE, KW>, dim3(grid), dim3(TcCfg<MODE, KW>::THREADS),
                       smem, st, a) != cudaSuccess)
        return check_launch(0);
    return PVS_OK;
}

int launch_edge_tc(const EdgeArgs &a, int n_ptiles_cap, int mode, cudaStream_t st) {
    if (a.ptile_last == nullptr || a.n_ptiles == nullptr || a.Mpart == nullptr ||
        a.xpart == nullptr)
        return PVS_ERR_INVALID_ARG;   // the tcgen05 kernel walks edge-packed tiles
    int rc;
    // PVS_EDGE_TC8 = 1 / 0 selects the bf16x3 variant (read once per process)
    static const int tc8 = [] {
        const char *e = getenv("PVS_EDGE_TC8");
        return e ? atoi(e) : PVS_EDGE_TC8_DEFAULT;
    }();
    // 65 <= k <= 128: the 128-wide tiles (forward only; P, Q, M at pitch 128)
    const bool wide = a.k > 64;
    if (wide && mode == PVS_MATH_BF16X3) rc = launch_mode<TCM_BF16X3, 128>(a, n_ptiles_cap, st);
    else if (wide && mode == PVS_MATH_FP16X2) rc = launch_mode<TCM_FP16X2, 128>(a, n_ptiles_cap, st);
    else if (wide) rc = launch_mode<TCM_BF16, 128>(a, n_ptiles_cap, st);
    else if (mode == PVS_MATH_BF16X3 && tc8) rc = launch_edge_tc8(a, n_ptiles_cap, st);
    else if (mode == PVS_MATH_BF16X3) rc = launch_mode<TCM_BF16X3>(a, n_ptiles_cap, st);
    else if (mode == PVS_MATH_FP16X2) rc = launch_mode<TCM_FP16X2>(a, n_ptiles_cap, st);
    else rc = launch_mode<TCM_BF16>(a, n_ptiles_cap, st);
    if (rc) return rc;
    const bool softmax = (a.flags & PVS_F_EDGE_ATTENTION) && (a.flags & PVS_F_SOFTMAX_ATTENTION);
    const int do_m = softmax ? 0 : 1, do_x = a.x_out != nullptr ? 1 : 0;
    if ((do_m || do_x) && wide)
        launch_chained(edge_tile_fixup_kernel<128>, dim3((n_ptiles_cap + 7) / 8), dim3(256), 0,
                       st, a, do_m, do_x);
    else if (do_m || do_x)
        launch_chained(edge_tile_fixup_kernel<64>, dim3((n_ptiles_cap + 7) / 8), dim3(256), 0, st,
                       a, do_m, do_x);
    return check_launch(do_m || do_x ? 2 : 1);
}

}  // namespace pvs
