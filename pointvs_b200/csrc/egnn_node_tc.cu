// Node-level stages of K2 on the tensor cores (PVS_MATH_BF16X3 / BF16):
//
//   node_pre_tc : [P | Q] = h . [W1a ; W1b]^T (+ b1 on P)      (N = 128, K = 64)
//   node_tc     : o = Wn2 silu(Wn1 [h ; M] + bn1) + bn2, node attention,
//                 residual -> h'                                (two K blocks of
//                 64 into one accumulator, then a 64x64 GEMM)
//
// Reference: egnn_satorras.py:82-86, 103-106, 134-166 (node_model) and the
// first Linear of edge_mlp :76-77 (factorised per node, see egnn_fwd.cu).
// Same machinery as egnn_edge_tc.cu: tiles of 128 nodes, rows converted to
// bf16 hi(/lo) K-major SWIZZLE_128B tiles by the threads, tcgen05.mma into
// TMEM, one thread per row in the epilogue, several independent 4-warp groups
// per persistent CTA sharing the weight tiles.  Outputs are staged through
// shared memory so global stores are full 256-byte rows.
#include <cstdlib>

#include <cuda.h>       // CUtensorMap (types only: the encoder comes from the runtime)

#include "egnn_common.cuh"
#include "egnn_bwd_common.cuh"
#include "tc_common.cuh"

namespace pvs {

#ifdef PVS_PHASE_PROF
// Debug build only (scripts/phase_prof.py --node): cycles of each group's
// thread 0 between the phase boundaries of node_tc_kernel.
__device__ unsigned long long g_node_phase_cycles[16];
#define NPH(i)                                                                \
    do {                                                                      \
        if (tid == 0) {                                                       \
            const long long now_ = clock64();                                 \
            atomicAdd(&g_node_phase_cycles[i], (unsigned long long)(now_ - t_prev_)); \
            t_prev_ = now_;                                                   \
        }                                                                     \
    } while (0)
extern "C" int pvs_debug_node_phase_cycles(unsigned long long *out, int reset) {
    cudaDeviceSynchronize();
    if (out) cudaMemcpyFromSymbol(out, g_node_phase_cycles, sizeof(g_node_phase_cycles));
    if (reset) {
        unsigned long long z[16] = {0};
        cudaMemcpyToSymbol(g_node_phase_cycles, z, sizeof(z));
    }
    return 0;
}
#else
#define NPH(i) do { } while (0)
#endif

constexpr int NODE_STORE_UNROLL = 4;
constexpr int NT_GROUP_THREADS = 128;
constexpr int NT_ROWS = 128;

__device__ __forceinline__ void nt_group_sync(int g) {
    asm volatile("bar.sync %0, %1;" ::"r"(g + 1), "n"(NT_GROUP_THREADS) : "memory");
}

// Row partition of the node kernels: every 4-warp group of the grid gets an
// equal share of the rows and walks it in equal tiles of at most 128 rows.
// (Fixed 128-row tiles dealt round-robin left 1000 tiles on 740 groups for the
// 128 x 1000-atom batch: a quarter of the groups did two tiles, the rest one,
// and the kernel took two tile times.)
struct RowShare { int begin, end, tile_rows; };
// rows per tile and tiles per group (host: the box height of the TMA stores)
__host__ __device__ inline void row_share_tiling(int n_rows, int n_groups, int *tile_rows,
                                                 int *tiles) {
    const int per = (n_rows + n_groups - 1) / n_groups;
    *tiles = per > NT_ROWS ? (per + NT_ROWS - 1) / NT_ROWS : 1;
    const int tr = (per + *tiles - 1) / *tiles;
    *tile_rows = tr > 1 ? tr : 1;
}
__device__ __forceinline__ RowShare row_share(int n_rows, int group_id, int n_groups) {
    RowShare r;
    int tiles;
    row_share_tiling(n_rows, n_groups, &r.tile_rows, &tiles);
    // whole tiles only: every tile of the grid has tile_rows rows (the box of
    // the TMA stores) except where the array ends
    const int per = tiles * r.tile_rows;
    r.begin = (int)min((long long)n_rows, (long long)group_id * per);
    r.end = min(n_rows, r.begin + per);
    return r;
}

// whole rows [row0, row_end) of a [*, ld] fp32 array -> L2 (one bulk prefetch
// per 32 KB; issued by one thread)
__device__ __forceinline__ void l2_prefetch_rows(const float *base, int ld, int row0, int row_end) {
    if (row_end <= row0) return;
    const char *p = reinterpret_cast<const char *>(base + (size_t)row0 * ld);
    const size_t bytes = (size_t)(row_end - row0) * ld * sizeof(float);
    const char *p16 = reinterpret_cast<const char *>((reinterpret_cast<uintptr_t>(p) + 15) & ~(uintptr_t)15);
    const size_t n16 = (bytes - (size_t)(p16 - p)) & ~(size_t)15;
    if (n16 >= 16)
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p16), "r"((uint32_t)n16)
                     : "memory");
}

// rows [row0, row0 + 128) x 64 columns of `src` (pitch ld, `cols` valid columns,
// `n_rows` valid rows overall) -> bf16 hi/lo swizzled A tiles.  8 lanes per row.
template <bool X3>
__device__ __forceinline__ void load_block(uint8_t *A_hi, uint8_t *A_lo,
                                           const float *__restrict__ src, int ld, int cols,
                                           int row0, int n_rows, int tid) {
    const int c = tid & 7, slot = tid >> 3;
    const bool vec = (cols == 64) && ((ld & 3) == 0);
#pragma unroll 4
    for (int p = 0; p < NT_ROWS / 16; ++p) {
        const int r = p * 16 + slot;
        float v[8];
        if (row0 + r < n_rows) {
            const float *s = src + (size_t)(row0 + r) * ld + 8 * c;
            if (vec) {
                const float4 a = __ldg(reinterpret_cast<const float4 *>(s));
                const float4 b = __ldg(reinterpret_cast<const float4 *>(s) + 1);
                v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
                v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = (8 * c + i < cols) ? __ldg(s + i) : 0.0f;
            }
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = 0.0f;
        }
        uint4 hi, lo;
        split8<X3>(v, hi, lo);
        *reinterpret_cast<uint4 *>(A_hi + swz(r, c)) = hi;
        if (X3) *reinterpret_cast<uint4 *>(A_lo + swz(r, c)) = lo;
    }
}

// fp32 staging tile [128][64] with the 16-byte chunk index XOR-swizzled by the
// row, so both the row-per-thread writes and the row-per-half-warp reads are
// conflict free.
__device__ __forceinline__ float4 *stage_ptr(float *stage, int r, int c4) {
    return reinterpret_cast<float4 *>(stage + r * 64 + ((c4 ^ (r & 15)) << 2));
}

// ---------------------------------------------------------------------------
// TMA tensor stores of fp32 output tiles.  A [rows][64] fp32 output leaves a
// tile as 32-column boxes: in shared memory a box is rows x 128 bytes with the
// 16-byte chunks XOR-swizzled by the row (SWIZZLE_128B: the same swz() the bf16
// operand tiles use, so row-per-thread writes are conflict free), and the
// tensor map un-swizzles it on the way to the row-major array in HBM.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void tma_store_2d(const CUtensorMap *tm, const void *smem, int c0,
                                             int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(smem)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_commit() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N>
__device__ __forceinline__ void tma_wait_read() {     // <= N groups still reading smem
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_wait_all() {
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// [n_rows][64] fp32 row-major array -> tensor map with boxes of 32 columns x
// box_rows rows, SWIZZLE_128B.  false if the driver entry point is unavailable.
static bool make_rows_tensor_map(CUtensorMap *tm, const float *base, int n_rows, int box_rows) {
    typedef CUresult (*EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                 const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                 const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = [] {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) !=
                cudaSuccess || q != cudaDriverEntryPointSuccess)
            fn = nullptr;
        return (EncodeFn)fn;
    }();
    if (!encode || n_rows < 1 || box_rows < 1 || box_rows > 256 ||
        (reinterpret_cast<uintptr_t>(base) & 15))
        return false;
    const cuuint64_t dims[2] = {64, (cuuint64_t)n_rows};
    const cuuint64_t strides[1] = {64 * sizeof(float)};
    const cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims,
                  strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) ==
           CUDA_SUCCESS;
}

// ---------------------------------------------------------------------------
// node_pre: P, Q
// ---------------------------------------------------------------------------
constexpr int NP_GROUPS = 4;
constexpr int NP_THREADS = NP_GROUPS * NT_GROUP_THREADS;

struct __align__(1024) NpSmem {
    uint8_t A_hi[NP_GROUPS][NT_ROWS * 128];
    uint8_t A_lo[NP_GROUPS][NT_ROWS * 128];
    uint8_t W_hi[128 * 128];    // rows 0..63: W1a (P), rows 64..127: W1b (Q)
    uint8_t W_lo[128 * 128];
    float b1[64];
    uint64_t mbar[NP_GROUPS];
    uint32_t tmem_base;
};

struct NodePreArgs {
    CUtensorMap tm_p, tm_q;   // P and Q as [N][64] fp32, boxes of 32 columns x tile_rows rows
    const float *h;       // [N][k]
    const float *edge_w1; // [k][in_e]
    const float *edge_b1; // [k]
    float *P, *Q;         // [N][64]
    int n_nodes, k, in_e, perm_invariant;
    int use_tma;          // P / Q tiles leave through the tensor maps
};

template <bool X3>
__global__ void __launch_bounds__(NP_THREADS, 1)
node_pre_tc_kernel(const __grid_constant__ NodePreArgs a) {
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    NpSmem &S = *reinterpret_cast<NpSmem *>(smem_dyn);
    pdl_launch_dependents();
    if ((smem_u32(smem_dyn) & 1023u) != 0u) __trap();
    const int g = threadIdx.x / NT_GROUP_THREADS, tid = threadIdx.x % NT_GROUP_THREADS;
    const int warp = tid >> 5;
    uint8_t *A_hi = S.A_hi[g], *A_lo = S.A_lo[g];
    const int k = a.k;
    load_weight_tiles<X3>(S.W_hi, S.W_lo, a.edge_w1, a.in_e, k, k, 64);
    load_weight_tiles<X3>(S.W_hi + 64 * 128, S.W_lo + 64 * 128,
                          a.edge_w1 + (a.perm_invariant ? 0 : k), a.in_e, k, k, 64);
    for (int n = threadIdx.x; n < 64; n += NP_THREADS) S.b1[n] = n < k ? a.edge_b1[n] : 0.0f;
    if (tid == 0) mbar_init(&S.mbar[g], 1);
    if (threadIdx.x < 32) tmem_alloc<512>(&S.tmem_base);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = S.tmem_base;
    const uint32_t tmem_grp = tmem_base + (uint32_t)g * 128u;
    const uint32_t tmem_lane = tmem_grp + ((uint32_t)(warp * 32) << 16);
    uint32_t phase = 0;
    const RowShare rs = row_share(a.n_nodes, blockIdx.x * NP_GROUPS + g, gridDim.x * NP_GROUPS);
    pdl_wait();      // h of the kernel before this one; P / Q still read by the edge kernel
    for (int row0 = rs.begin; row0 < rs.end; row0 += rs.tile_rows) {
        const int row_end = min(rs.end, row0 + rs.tile_rows);
        nt_group_sync(g);   // staging of the previous tile fully stored
        load_block<X3>(A_hi, A_lo, a.h, k, k, row0, row_end, tid);
        fence_proxy_async();
        tc_fence_before();
        nt_group_sync(g);
        if (tid == 0) {
            tc_fence_after();
            issue_kblock<X3>(tmem_grp, tc_idesc(128), A_hi, A_lo, S.W_hi, S.W_lo, 0);
            umma_commit(&S.mbar[g]);
        }
        mbar_wait(&S.mbar[g], phase);
        phase ^= 1;
        tc_fence_after();
        if (a.use_tma) {
            // The A tiles are free once the MMA has completed.  Four boxes of 32
            // columns (P low, P high, Q low, Q high) alternate between them: a
            // thread writes its row of the box (swizzled, conflict free), one
            // thread hands the box to the TMA engine, and the next box is
            // written while that store drains.
#pragma unroll 1
            for (int sq = 0; sq < 4; ++sq) {
                uint8_t *buf = (sq & 1) ? A_lo : A_hi;
                if (sq >= 2) {                    // the store issued two boxes ago has
                    if (tid == 0) tma_wait_read<1>();   // finished reading this buffer
                    nt_group_sync(g);
                }
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    float acc[16];
                    tmem_ld16(tmem_lane + 32 * sq + 16 * b, acc);
#pragma unroll
                    for (int v4 = 0; v4 < 4; ++v4) {
                        float4 o = make_float4(acc[4 * v4], acc[4 * v4 + 1], acc[4 * v4 + 2],
                                               acc[4 * v4 + 3]);
                        if (sq < 2) {
                            const float4 bb = *reinterpret_cast<const float4 *>(
                                &S.b1[32 * sq + 16 * b + 4 * v4]);
                            o.x += bb.x; o.y += bb.y; o.z += bb.z; o.w += bb.w;
                        }
                        *reinterpret_cast<float4 *>(buf + swz(tid, 4 * b + v4)) = o;
                    }
                }
                fence_proxy_async();
                nt_group_sync(g);
                if (tid == 0) {
                    tma_store_2d(sq < 2 ? &a.tm_p : &a.tm_q, buf, 32 * (sq & 1), row0);
                    tma_commit();
                }
            }
            if (tid == 0) tma_wait_read<0>();     // before the next tile refills the A tiles
            tc_fence_before();
            continue;
        }
        // (thread-store path: tensor maps unavailable)  Each 16 KB tile stages
        // 64 rows of fp32 output (rows 0..63 in A_hi, 64..127 in A_lo), P first,
        // then Q.
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {   // half 0: P (cols 0..63), 1: Q
            const int r = tid;
            float *st = reinterpret_cast<float *>(r < 64 ? A_hi : A_lo);
            const int rr = r & 63;
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {
                float acc[16];
                tmem_ld16(tmem_lane + 64 * half + 16 * q, acc);
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4) {
                    float4 o = make_float4(acc[4 * v4], acc[4 * v4 + 1], acc[4 * v4 + 2],
                                           acc[4 * v4 + 3]);
                    if (half == 0) {
                        const float4 b = *reinterpret_cast<const float4 *>(&S.b1[16 * q + 4 * v4]);
                        o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
                    }
                    *stage_ptr(st, rr, 4 * q + v4) = o;
                }
            }
            nt_group_sync(g);
            // coalesced store: 128 rows in two 64-row staging tiles
            {
                float *dst = half == 0 ? a.P : a.Q;
                const int c4 = tid & 15, slot = tid >> 4;
#pragma unroll 4
                for (int p = 0; p < NT_ROWS / 8; ++p) {
                    const int row = p * 8 + slot;
                    if (row0 + row >= row_end) continue;
                    const float *sp = reinterpret_cast<const float *>(row < 64 ? A_hi : A_lo);
                    const float4 v = *stage_ptr(const_cast<float *>(sp), row & 63, c4);
                    *reinterpret_cast<float4 *>(dst + (size_t)(row0 + row) * 64 + 4 * c4) = v;
                }
            }
            nt_group_sync(g);
        }
        tc_fence_before();
    }
    if (a.use_tma && tid == 0) tma_wait_all();     // the tiles have reached HBM
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------
// node model
// ---------------------------------------------------------------------------
constexpr int NM_GROUPS = 5;
constexpr int NM_THREADS = NM_GROUPS * NT_GROUP_THREADS;

struct __align__(1024) NmSmem {
    uint8_t A_hi[NM_GROUPS][NT_ROWS * 128];
    uint8_t A_lo[NM_GROUPS][NT_ROWS * 128];
    uint8_t W1h_hi[64 * 128], W1h_lo[64 * 128];   // node_w1[:, 0:k]   (h part)
    uint8_t W1m_hi[64 * 128], W1m_lo[64 * 128];   // node_w1[:, k:2k]  (M part)
    uint8_t W2_hi[64 * 128], W2_lo[64 * 128];
    float b1[64], b2[64], wn[64], ga[64], gb[64];
    float srow[NM_GROUPS][NT_ROWS];   // node attention value of each row of the tile
    uint64_t mbar[NM_GROUPS];
    uint32_t tmem_base;
};

struct NodeTcArgs {
    CUtensorMap tm_h;    // h_out as [N][64] fp32 (k == 64), boxes of 32 columns x tile_rows
    int use_tma;         // h_out tiles leave through tm_h
    const float *h_in;   // [N][k]
    const float *M;      // [N][64]
    float *h_out;        // [N][k]
    float *natt_out;     // [N] or null
    const float *node_w1, *node_b1, *node_w2, *node_b2, *natt_w, *natt_b, *node_gate;
    int n_nodes, k;
    uint32_t flags;
    int att_act;
    // GraphNorm (batch-wide statistics between the two Linears,
    // egnn_satorras.py:84): phase 1 stops after Wn1 and writes the
    // pre-activation V; phase 2 resumes from V with the affine gn_a * v + gn_b
    float *V;            // [N][64]
    const float *gn_a, *gn_b;
    int phase;           // 0: whole node model
};

// V rows -> u = silu(ga * v + gb) -> bf16 hi/lo A tiles (phase 2 of GraphNorm)
template <bool X3>
__device__ __forceinline__ void load_block_gn(uint8_t *A_hi, uint8_t *A_lo,
                                              const float *__restrict__ V, const float *ga,
                                              const float *gb, int row0, int n_rows, int tid) {
    const int c = tid & 7, slot = tid >> 3;
    float a8[8], b8[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { a8[i] = ga[8 * c + i]; b8[i] = gb[8 * c + i]; }
#pragma unroll 4
    for (int p = 0; p < NT_ROWS / 16; ++p) {
        const int r = p * 16 + slot;
        float v[8];
        if (row0 + r < n_rows) {
            const float4 *s4 = reinterpret_cast<const float4 *>(V + (size_t)(row0 + r) * 64 + 8 * c);
            const float4 x = __ldg(s4), y = __ldg(s4 + 1);
            const float in[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = silu_mode<X3>(fmaf(a8[i], in[i], b8[i]));
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = 0.0f;
        }
        uint4 hi, lo;
        split8<X3>(v, hi, lo);
        *reinterpret_cast<uint4 *>(A_hi + swz(r, c)) = hi;
        if (X3) *reinterpret_cast<uint4 *>(A_lo + swz(r, c)) = lo;
    }
}

template <bool X3>
__global__ void __launch_bounds__(NM_THREADS, 1)
node_tc_kernel(const __grid_constant__ NodeTcArgs a) {
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    NmSmem &S = *reinterpret_cast<NmSmem *>(smem_dyn);
    pdl_launch_dependents();
    if ((smem_u32(smem_dyn) & 1023u) != 0u) __trap();
    const int g = threadIdx.x / NT_GROUP_THREADS, tid = threadIdx.x % NT_GROUP_THREADS;
#ifdef PVS_PHASE_PROF
    long long t_prev_ = clock64();
#endif
    const int warp = tid >> 5;
    uint8_t *A_hi = S.A_hi[g], *A_lo = S.A_lo[g];
    const int k = a.k;
    // this group's rows of h (written two kernels ago: usually evicted) and of M
    // start their way from HBM to L2 while the CTA builds its weight tiles
    // (one bulk prefetch each; measured -0.2 % on the scoring pass)
    if (tid == 0 && a.phase != 2) {
        const RowShare pf = row_share(a.n_nodes, blockIdx.x * NM_GROUPS + g, gridDim.x * NM_GROUPS);
        l2_prefetch_rows(a.h_in, k, pf.begin, pf.end);
        l2_prefetch_rows(a.M, 64, pf.begin, pf.end);
    }
    load_weight_tiles<X3>(S.W1h_hi, S.W1h_lo, a.node_w1, 2 * k, k, k);
    load_weight_tiles<X3>(S.W1m_hi, S.W1m_lo, a.node_w1 + k, 2 * k, k, k);
    load_weight_tiles<X3>(S.W2_hi, S.W2_lo, a.node_w2, k, k, k);
    for (int n = threadIdx.x; n < 64; n += NM_THREADS) {
        S.b1[n] = n < k ? a.node_b1[n] : 0.0f;
        S.b2[n] = n < k ? a.node_b2[n] : 0.0f;
        S.wn[n] = (n < k && a.natt_w) ? a.natt_w[n] : 0.0f;
        S.ga[n] = (n < k && a.gn_a) ? a.gn_a[n] : 1.0f;
        S.gb[n] = (n < k && a.gn_b) ? a.gn_b[n] : 0.0f;
    }
    if (tid == 0) mbar_init(&S.mbar[g], 1);
    if (threadIdx.x < 32) tmem_alloc<512>(&S.tmem_base);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = S.tmem_base;
    const uint32_t tmem_grp = tmem_base + (uint32_t)g * 64u;
    const uint32_t tmem_lane = tmem_grp + ((uint32_t)(warp * 32) << 16);
    uint32_t phase = 0;
    const bool f_natt = (a.flags & PVS_F_NODE_ATTENTION) && a.natt_w != nullptr;
    const bool f_res = a.flags & PVS_F_RESIDUAL;
    const float natt_b = (f_natt && a.natt_b) ? a.natt_b[0] : 0.0f;
    const float gate = a.node_gate ? a.node_gate[0] : 1.0f;
    NPH(0);   // prologue: weight tiles, TMEM
    const RowShare rs = row_share(a.n_nodes, blockIdx.x * NM_GROUPS + g, gridDim.x * NM_GROUPS);
    pdl_wait();      // M (and h) of the kernels before this one
    for (int row0 = rs.begin; row0 < rs.end; row0 += rs.tile_rows) {
        const int row_end = min(rs.end, row0 + rs.tile_rows);
        nt_group_sync(g);
        if (a.phase != 2) {
            // ---- v = Wn1 [h ; M]: two K blocks through the same A tiles ----
            load_block<X3>(A_hi, A_lo, a.h_in, k, k, row0, row_end, tid);
            fence_proxy_async();
            tc_fence_before();
            nt_group_sync(g);
            NPH(1);   // h block
            if (tid == 0) {
                tc_fence_after();
                issue_kblock<X3>(tmem_grp, tc_idesc(64), A_hi, A_lo, S.W1h_hi, S.W1h_lo, 0);
                umma_commit(&S.mbar[g]);
            }
            mbar_wait(&S.mbar[g], phase);
            phase ^= 1;
            NPH(2);   // GEMM 1a
            load_block<X3>(A_hi, A_lo, a.M, 64, 64, row0, row_end, tid);
            fence_proxy_async();
            tc_fence_before();
            nt_group_sync(g);
            NPH(3);   // M block
            if (tid == 0) {
                tc_fence_after();
                issue_kblock<X3>(tmem_grp, tc_idesc(64), A_hi, A_lo, S.W1m_hi, S.W1m_lo, 1);
                umma_commit(&S.mbar[g]);
            }
            mbar_wait(&S.mbar[g], phase);
            phase ^= 1;
            tc_fence_after();
            NPH(4);   // GEMM 1b
        }
        if (a.phase == 1) {
            // ---- GraphNorm phase 1: V = v + b1 (fp32) -> staging -> HBM ----
            const int r = tid;
            float *st = reinterpret_cast<float *>(r < 64 ? A_hi : A_lo);
            const int rr = r & 63;
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {
                float acc[16];
                tmem_ld16(tmem_lane + 16 * q, acc);
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4) {
                    const int n = 16 * q + 4 * v4;
                    *stage_ptr(st, rr, 4 * q + v4) =
                        make_float4(acc[4 * v4] + S.b1[n], acc[4 * v4 + 1] + S.b1[n + 1],
                                    acc[4 * v4 + 2] + S.b1[n + 2], acc[4 * v4 + 3] + S.b1[n + 3]);
                }
            }
            tc_fence_before();
            nt_group_sync(g);
            const int c4 = tid & 15, slot = tid >> 4;
#pragma unroll 4
            for (int p = 0; p < NT_ROWS / 8; ++p) {
                const int row = p * 8 + slot;
                if (row0 + row >= row_end) continue;
                const float *sp = reinterpret_cast<const float *>(row < 64 ? A_hi : A_lo);
                *reinterpret_cast<float4 *>(a.V + (size_t)(row0 + row) * 64 + 4 * c4) =
                    *stage_ptr(const_cast<float *>(sp), row & 63, c4);
            }
            continue;
        }
        if (a.phase == 2) {
            load_block_gn<X3>(A_hi, A_lo, a.V, S.ga, S.gb, row0, row_end, tid);
        } else {
            // ---- u = silu(v + b1) -> A tiles ----
            {
                const int r = tid;
    #pragma unroll 1
                for (int q = 0; q < 4; ++q) {
                    float acc[16];
                    tmem_ld16(tmem_lane + 16 * q, acc);
    #pragma unroll
                    for (int hlf = 0; hlf < 2; ++hlf) {
                        const int nb = 16 * q + 8 * hlf;
                        const float4 ba = *reinterpret_cast<const float4 *>(&S.b1[nb]);
                        const float4 bb = *reinterpret_cast<const float4 *>(&S.b1[nb + 4]);
                        const float bias[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
                        float u[8];
    #pragma unroll
                        for (int i = 0; i < 8; ++i) u[i] = silu_mode<X3>(acc[8 * hlf + i] + bias[i]);
                        uint4 hi, lo;
                        split8<X3>(u, hi, lo);
                        *reinterpret_cast<uint4 *>(A_hi + swz(r, 2 * q + hlf)) = hi;
                        if (X3) *reinterpret_cast<uint4 *>(A_lo + swz(r, 2 * q + hlf)) = lo;
                    }
                }
            }
        }
        fence_proxy_async();
        tc_fence_before();
        nt_group_sync(g);
        NPH(5);   // epilogue 1
        if (tid == 0) {
            tc_fence_after();
            issue_kblock<X3>(tmem_grp, tc_idesc(64), A_hi, A_lo, S.W2_hi, S.W2_lo, 0);
            umma_commit(&S.mbar[g]);
        }
        mbar_wait(&S.mbar[g], phase);
        phase ^= 1;
        tc_fence_after();
        NPH(6);   // GEMM 2
        if (a.use_tma) {
            // ---- k == 64: the thread owns its whole row, so the attention logit
            // is thread-local; a second pass over TMEM forms
            // h' = residual(h, s (D + b2)) straight into two 32-column boxes
            // (SWIZZLE_128B, conflict free) which the TMA engine stores.  h is
            // read per thread (a 256-byte row each, L2-hot from the A-tile load).
            const int r = tid;
            const bool ok = row0 + r < row_end;
            float s = 1.0f;
            if (f_natt) {
                float dot = 0.0f;
#pragma unroll 1
                for (int q = 0; q < 4; ++q) {
                    float acc[16];
                    tmem_ld16(tmem_lane + 16 * q, acc);
#pragma unroll
                    for (int i = 0; i < 16; ++i)
                        dot = fmaf(S.wn[16 * q + i], acc[i] + S.b2[16 * q + i], dot);
                }
                const float zn = dot + natt_b;
                s = (a.flags & PVS_F_SOFTMAX_ATTENTION) ? zn : apply_act(zn, a.att_act);
                if (a.natt_out && ok) a.natt_out[row0 + r] = s;
            }
            const float4 *hrow = reinterpret_cast<const float4 *>(
                a.h_in + (size_t)(row0 + (ok ? r : 0)) * 64);
            const float G = fmaxf(gate, 0.0f);
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {
                float acc[16];
                tmem_ld16(tmem_lane + 16 * q, acc);
                uint8_t *buf = q < 2 ? A_hi : A_lo;
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4) {
                    const int n = 16 * q + 4 * v4;
                    float o[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) o[i] = s * (acc[4 * v4 + i] + S.b2[n + i]);
                    if (f_res) {
                        const float4 h4 = __ldg(hrow + 4 * q + v4);
                        const float hv[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            if (a.flags & PVS_F_REZERO) o[i] = hv[i] + gate * o[i];
                            else if (a.flags & PVS_F_GATED_RESIDUAL)
                                o[i] = G * o[i] + (1.0f - G) * hv[i];
                            else o[i] = hv[i] + o[i];
                        }
                    }
                    *reinterpret_cast<float4 *>(buf + swz(r, 4 * (q & 1) + v4)) =
                        make_float4(o[0], o[1], o[2], o[3]);
                }
            }
            fence_proxy_async();
            tc_fence_before();
            nt_group_sync(g);
            NPH(7);
            if (tid == 0) {
                tma_store_2d(&a.tm_h, A_hi, 0, row0);
                tma_store_2d(&a.tm_h, A_lo, 32, row0);
                tma_commit();
                tma_wait_read<0>();    // the loop-top barrier then frees the A tiles
            }
#ifdef PVS_PHASE_PROF
            nt_group_sync(g);
#endif
            NPH(8);
            continue;
        }
        // ---- o = D + b2 and the node-attention logit in ONE pass over TMEM
        // (thread per row); o goes to the fp32 staging tile unscaled.  The
        // attention factor and the residual are applied in the store pass, where
        // a row of h is read as full 256-byte lines instead of per-thread rows.
        {
            const int r = tid;
            const bool ok = row0 + r < row_end;
            // A tiles are free (GEMM 2 has completed): 64 rows of fp32 staging in
            // each 16 KB tile
            float *st = reinterpret_cast<float *>(r < 64 ? A_hi : A_lo);
            const int rr = r & 63;
            float dot = 0.0f;
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {
                float acc[16];
                tmem_ld16(tmem_lane + 16 * q, acc);
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4) {
                    const int n = 16 * q + 4 * v4;
                    float o[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        o[i] = acc[4 * v4 + i] + S.b2[n + i];
                        dot = fmaf(S.wn[n + i], o[i], dot);
                    }
                    *stage_ptr(st, rr, 4 * q + v4) = make_float4(o[0], o[1], o[2], o[3]);
                }
            }
            float s = 1.0f;
            if (f_natt) {
                const float zn = dot + natt_b;
                s = (a.flags & PVS_F_SOFTMAX_ATTENTION) ? zn : apply_act(zn, a.att_act);
                if (a.natt_out && ok) a.natt_out[row0 + r] = s;
            }
            S.srow[g][r] = s;
        }
        tc_fence_before();
        nt_group_sync(g);
        NPH(7);   // epilogue 2
        {
            const int c4 = tid & 15, slot = tid >> 4;
            const bool vec = (k & 3) == 0;
            const float G = fmaxf(gate, 0.0f);
#pragma unroll NODE_STORE_UNROLL
            for (int p = 0; p < NT_ROWS / 8; ++p) {
                const int row = p * 8 + slot;
                if (row0 + row >= row_end) continue;
                const float *sp = reinterpret_cast<const float *>(row < 64 ? A_hi : A_lo);
                float4 v = *stage_ptr(const_cast<float *>(sp), row & 63, c4);
                const float s = S.srow[g][row];
                const float *hrow = a.h_in + (size_t)(row0 + row) * k + 4 * c4;
                float o[4] = {v.x * s, v.y * s, v.z * s, v.w * s};
                if (f_res) {
                    float hv[4] = {0.f, 0.f, 0.f, 0.f};
                    if (vec && 4 * c4 + 3 < k) {
                        const float4 h4 = __ldg(reinterpret_cast<const float4 *>(hrow));
                        hv[0] = h4.x; hv[1] = h4.y; hv[2] = h4.z; hv[3] = h4.w;
                    } else {
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            hv[i] = (4 * c4 + i < k) ? __ldg(hrow + i) : 0.0f;
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        if (a.flags & PVS_F_REZERO) o[i] = hv[i] + gate * o[i];
                        else if (a.flags & PVS_F_GATED_RESIDUAL) o[i] = G * o[i] + (1.0f - G) * hv[i];
                        else o[i] = hv[i] + o[i];
                    }
                }
                float *d = a.h_out + (size_t)(row0 + row) * k + 4 * c4;
                if (vec && 4 * c4 + 3 < k) {
                    *reinterpret_cast<float4 *>(d) = make_float4(o[0], o[1], o[2], o[3]);
                } else {
                    if (4 * c4 < k) d[0] = o[0];
                    if (4 * c4 + 1 < k) d[1] = o[1];
                    if (4 * c4 + 2 < k) d[2] = o[2];
                    if (4 * c4 + 3 < k) d[3] = o[3];
                }
            }
        }
#ifdef PVS_PHASE_PROF
        nt_group_sync(g);
#endif
        NPH(8);   // store pass
    }
    if (a.use_tma && tid == 0) tma_wait_all();     // the tiles have reached HBM
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------
// K3, first edge layer (factorised): d_h += dP . W1a + dQ . W1b
// ---------------------------------------------------------------------------
// The transpose of node_pre (K = 128 as two blocks of 64, N = 64), same shape
// as the first stage of node_tc: dP rows, then dQ rows, through the same A
// tiles into one accumulator; B = W1a^T / W1b^T.  Replaces two FFMA linear
// launches per layer (14 us each at 16 k nodes, launch- and latency-bound).
constexpr int DG_GROUPS = 5;
constexpr int DG_THREADS = DG_GROUPS * NT_GROUP_THREADS;

struct __align__(1024) DgSmem {
    uint8_t A_hi[DG_GROUPS][NT_ROWS * 128];
    uint8_t A_lo[DG_GROUPS][NT_ROWS * 128];
    uint8_t Wa_hi[64 * 128], Wa_lo[64 * 128];   // tile[c][j] = W1a[j][c]
    uint8_t Wb_hi[64 * 128], Wb_lo[64 * 128];
    uint64_t mbar[DG_GROUPS];
    uint32_t tmem_base;
};

struct DgradPqArgs {
    const float *dP, *dQ;     // [N][64]
    const float *edge_w1;     // [k][in_e]: W1a = columns 0..k-1, W1b = columns k..2k-1
    float *d_h;               // [N][k], accumulated into
    int n_nodes, k, in_e;
};

__global__ void __launch_bounds__(DG_THREADS, 1)
dgrad_pq_tc_kernel(const DgradPqArgs a) {
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    DgSmem &S = *reinterpret_cast<DgSmem *>(smem_dyn);
    if ((smem_u32(smem_dyn) & 1023u) != 0u) __trap();
    const int g = threadIdx.x / NT_GROUP_THREADS, tid = threadIdx.x % NT_GROUP_THREADS;
    const int warp = tid >> 5;
    uint8_t *A_hi = S.A_hi[g], *A_lo = S.A_lo[g];
    const int k = a.k;
    load_weight_tiles_T(S.Wa_hi, S.Wa_lo, a.edge_w1, a.in_e, k, k);
    load_weight_tiles_T(S.Wb_hi, S.Wb_lo, a.edge_w1 + k, a.in_e, k, k);
    if (tid == 0) mbar_init(&S.mbar[g], 1);
    if (threadIdx.x < 32) tmem_alloc<512>(&S.tmem_base);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = S.tmem_base;
    const uint32_t tmem_grp = tmem_base + (uint32_t)g * 64u;
    const uint32_t tmem_lane = tmem_grp + ((uint32_t)(warp * 32) << 16);
    uint32_t phase = 0;
    const RowShare rs = row_share(a.n_nodes, blockIdx.x * DG_GROUPS + g, gridDim.x * DG_GROUPS);
    pdl_wait();                  // dP, dQ, d_h of the kernels before this one
    pdl_launch_dependents();
    for (int row0 = rs.begin; row0 < rs.end; row0 += rs.tile_rows) {
        const int row_end = min(rs.end, row0 + rs.tile_rows);
        nt_group_sync(g);
        load_block<true>(A_hi, A_lo, a.dP, 64, 64, row0, row_end, tid);
        fence_proxy_async();
        tc_fence_before();
        nt_group_sync(g);
        if (tid == 0) {
            tc_fence_after();
            issue_kblock<true>(tmem_grp, tc_idesc(64), A_hi, A_lo, S.Wa_hi, S.Wa_lo, 0);
            umma_commit(&S.mbar[g]);
        }
        mbar_wait(&S.mbar[g], phase);
        phase ^= 1;
        load_block<true>(A_hi, A_lo, a.dQ, 64, 64, row0, row_end, tid);
        fence_proxy_async();
        tc_fence_before();
        nt_group_sync(g);
        if (tid == 0) {
            tc_fence_after();
            issue_kblock<true>(tmem_grp, tc_idesc(64), A_hi, A_lo, S.Wb_hi, S.Wb_lo, 1);
            umma_commit(&S.mbar[g]);
        }
        mbar_wait(&S.mbar[g], phase);
        phase ^= 1;
        tc_fence_after();
        // D -> fp32 staging (64 rows in each 16 KB A tile), then d_h += staged
        // rows as full lines
        {
            const int r = tid;
            float *st = reinterpret_cast<float *>(r < 64 ? A_hi : A_lo);
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {
                float acc[16];
                tmem_ld16(tmem_lane + 16 * q, acc);
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4)
                    *stage_ptr(st, r & 63, 4 * q + v4) =
                        make_float4(acc[4 * v4], acc[4 * v4 + 1], acc[4 * v4 + 2], acc[4 * v4 + 3]);
            }
        }
        tc_fence_before();
        nt_group_sync(g);
        {
            const int c4 = tid & 15, slot = tid >> 4;
            const bool vec = (k & 3) == 0;
#pragma unroll 4
            for (int p = 0; p < NT_ROWS / 8; ++p) {
                const int row = p * 8 + slot;
                if (row0 + row >= row_end) continue;
                const float *sp = reinterpret_cast<const float *>(row < 64 ? A_hi : A_lo);
                const float4 v = *stage_ptr(const_cast<float *>(sp), row & 63, c4);
                float *d = a.d_h + (size_t)(row0 + row) * k + 4 * c4;
                if (vec && 4 * c4 + 3 < k) {
                    float4 o = *reinterpret_cast<float4 *>(d);
                    o.x += v.x; o.y += v.y; o.z += v.z; o.w += v.w;
                    *reinterpret_cast<float4 *>(d) = o;
                } else {
                    if (4 * c4 < k) d[0] += v.x;
                    if (4 * c4 + 1 < k) d[1] += v.y;
                    if (4 * c4 + 2 < k) d[2] += v.z;
                    if (4 * c4 + 3 < k) d[3] += v.w;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc<512>(tmem_base);
}

int launch_dgrad_pq_tc(const float *dP, const float *dQ, const float *edge_w1, float *d_h,
                       int n_nodes, int k, int in_e, cudaStream_t st) {
    DgradPqArgs a{dP, dQ, edge_w1, d_h, n_nodes, k, in_e};
    const size_t smem = sizeof(DgSmem);
    int grid = num_sms();
    const int need = (n_nodes + 16 * DG_GROUPS - 1) / (16 * DG_GROUPS);
    if (need < grid) grid = need;
    if (grid < 1) grid = 1;
    const int rc = ensure_smem(dgrad_pq_tc_kernel, smem);
    if (rc) return rc;
    launch_chained(dgrad_pq_tc_kernel, dim3(grid), dim3(DG_THREADS), smem, st, a);
    return check_launch();
}

// ---------------------------------------------------------------------------
// K3, node model backward (no GraphNorm) on tcgen05
// ---------------------------------------------------------------------------
// Autograd of node_model (egnn_satorras.py:134-166), same mathematics as
// egnn_node_bwd_kernel (egnn_bwd.cu, FFMA) with its four contractions as UMMA
// in bf16x3:
//   V  = [h ; M] . W1^T          recompute    two K blocks, B = W1h, W1m (K-major)
//   O  = U . W2^T                recompute    B = W2 (K-major)
//   dU = dO . W2                 data grad    B = the SAME W2 tile read MN-major
//   dh = dV . W1h, dM = dV . W1m data grads   B = the W1h / W1m tiles read MN-major
// A weight tile image [out][in] serves both directions: K-major it is W^T as
// the forward needs it, MN-major (rows = K) it is W.  Row-per-thread epilogues
// as in node_tc: the attention logit, the gate products and d(attention) are
// thread-local sums over the row; V stays in tensor memory and is re-read for
// silu'(V).  The factors of the node weight gradients (U, O, dO, dV) go to HBM
// for wgrad_group_tc_kernel as before.
constexpr int NB_GROUPS = 4;
constexpr int NB_THREADS = NB_GROUPS * NT_GROUP_THREADS;
constexpr uint32_t NB_IDESC_BMN = tc_idesc(64) | (1u << 16);    // B MN-major

struct __align__(1024) NbSmem {
    uint8_t A_hi[NB_GROUPS][NT_ROWS * 128];
    uint8_t A_lo[NB_GROUPS][NT_ROWS * 128];
    uint8_t W1h_hi[64 * 128], W1h_lo[64 * 128];
    uint8_t W1m_hi[64 * 128], W1m_lo[64 * 128];
    uint8_t W2_hi[64 * 128], W2_lo[64 * 128];
    float b1[64], b2[64], wn[64];
    uint64_t mbar[NB_GROUPS];
    uint32_t tmem_base;
};

// D[128 x 64] (+)= A . B with A K-major and B read MN-major (tile rows = K)
__device__ __forceinline__ void issue_kblock_bmn(uint32_t tmem_d, const uint8_t *a_hi,
                                                 const uint8_t *a_lo, const uint8_t *b_hi,
                                                 const uint8_t *b_lo, uint32_t acc) {
    const uint64_t ah = make_desc(smem_u32(a_hi)), al = make_desc(smem_u32(a_lo));
    const uint64_t bh = make_desc(smem_u32(b_hi)), bl = make_desc(smem_u32(b_lo));
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
        const uint64_t aadv = (uint64_t)(ks * 2);              // 16 bf16 along a row
        const uint64_t badv = (uint64_t)(ks * (2048 >> 4));    // 16 rows of 128 bytes
        umma_bf16(tmem_d, ah + aadv, bh + badv, NB_IDESC_BMN, acc);
        acc = 1;
        umma_bf16(tmem_d, al + aadv, bh + badv, NB_IDESC_BMN, 1);
        umma_bf16(tmem_d, ah + aadv, bl + badv, NB_IDESC_BMN, 1);
    }
}

// 16 floats [c0, c0 + 16) of a row with `kv` valid columns (zeros beyond / !ok)
__device__ __forceinline__ void row_load16(const float *row, int kv, int c0, bool ok, bool vec,
                                           float (&v)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.0f;
    if (!ok || c0 >= kv) return;
    if (vec && c0 + 16 <= kv) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float4 t = __ldg(reinterpret_cast<const float4 *>(row + c0) + j);
            v[4 * j] = t.x; v[4 * j + 1] = t.y; v[4 * j + 2] = t.z; v[4 * j + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (c0 + i < kv) v[i] = __ldg(row + c0 + i);
    }
}
__device__ __forceinline__ void row_store16(float *row, int kv, int c0, bool ok, bool vec,
                                            const float (&v)[16]) {
    if (!ok || c0 >= kv) return;
    if (vec && c0 + 16 <= kv) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            reinterpret_cast<float4 *>(row + c0)[j] =
                make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    } else {
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (c0 + i < kv) row[c0 + i] = v[i];
    }
}

__global__ void __launch_bounds__(NB_THREADS, 1)
node_bwd_tc_kernel(const NodeBwdArgs a) {
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    NbSmem &S = *reinterpret_cast<NbSmem *>(smem_dyn);
    if ((smem_u32(smem_dyn) & 1023u) != 0u) __trap();
    const int g = threadIdx.x / NT_GROUP_THREADS, tid = threadIdx.x % NT_GROUP_THREADS;
    const int warp = tid >> 5;
    uint8_t *A_hi = S.A_hi[g], *A_lo = S.A_lo[g];
    const int k = a.k;
    load_weight_tiles<true>(S.W1h_hi, S.W1h_lo, a.node_w1, 2 * k, k, k);
    load_weight_tiles<true>(S.W1m_hi, S.W1m_lo, a.node_w1 + k, 2 * k, k, k);
    load_weight_tiles<true>(S.W2_hi, S.W2_lo, a.node_w2, k, k, k);
    for (int n = threadIdx.x; n < 64; n += NB_THREADS) {
        S.b1[n] = n < k ? a.node_b1[n] : 0.0f;
        S.b2[n] = n < k ? a.node_b2[n] : 0.0f;
        S.wn[n] = (n < k && a.natt_w) ? a.natt_w[n] : 0.0f;
    }
    if (tid == 0) mbar_init(&S.mbar[g], 1);
    if (threadIdx.x < 32) tmem_alloc<512>(&S.tmem_base);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = S.tmem_base;
    const uint32_t tmem_grp = tmem_base + (uint32_t)g * 128u;     // V: +0, work: +64
    const uint32_t tl = tmem_grp + ((uint32_t)(warp * 32) << 16);
    constexpr uint32_t C_V = 0, C_W = 64;
    uint32_t phase = 0;
    const bool f_natt = (a.flags & PVS_F_NODE_ATTENTION) && a.natt_w != nullptr;
    const bool f_res = a.flags & PVS_F_RESIDUAL;
    const bool f_rez = f_res && (a.flags & PVS_F_REZERO);
    const bool f_gat = f_res && (a.flags & PVS_F_GATED_RESIDUAL);
    const float natt_b = (f_natt && a.natt_b) ? a.natt_b[0] : 0.0f;
    const float gate = a.node_gate ? a.node_gate[0] : 1.0f;
    const float G = fmaxf(gate, 0.0f);
    const bool vec = (k & 3) == 0;
    auto publish = [&]() {
        fence_proxy_async();
        tc_fence_before();
        nt_group_sync(g);
    };
    auto commit_wait = [&]() {
        if (tid == 0) umma_commit(&S.mbar[g]);
        mbar_wait(&S.mbar[g], phase);
        phase ^= 1;
        tc_fence_after();
    };
    // 16 values of this thread's row -> chunks 2 q, 2 q + 1 of the A tiles
    auto to_tile = [&](int q, const float (&v)[16]) {
#pragma unroll
        for (int hlf = 0; hlf < 2; ++hlf) {
            float u8[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) u8[i] = v[8 * hlf + i];
            uint4 hi, lo;
            split8<true>(u8, hi, lo);
            *reinterpret_cast<uint4 *>(A_hi + swz(tid, 2 * q + hlf)) = hi;
            *reinterpret_cast<uint4 *>(A_lo + swz(tid, 2 * q + hlf)) = lo;
        }
    };
    const RowShare rs = row_share(a.n_nodes, blockIdx.x * NB_GROUPS + g, gridDim.x * NB_GROUPS);
    pdl_wait();                  // chain kernel (backward order): see pvs_common.cuh
    pdl_launch_dependents();
    for (int row0 = rs.begin; row0 < rs.end; row0 += rs.tile_rows) {
        const int row_end = min(rs.end, row0 + rs.tile_rows);
        const int r = tid;
        const bool ok = row0 + r < row_end;
        const size_t row = (size_t)(row0 + (ok ? r : 0));
        nt_group_sync(g);
        // ---- V = [h ; M] . W1^T ----
        load_block<true>(A_hi, A_lo, a.h_in, k, k, row0, row_end, tid);
        publish();
        if (tid == 0) {
            tc_fence_after();
            issue_kblock<true>(tmem_grp + C_V, tc_idesc(64), A_hi, A_lo, S.W1h_hi, S.W1h_lo, 0);
        }
        commit_wait();
        load_block<true>(A_hi, A_lo, a.M, 64, 64, row0, row_end, tid);
        publish();
        if (tid == 0) {
            tc_fence_after();
            issue_kblock<true>(tmem_grp + C_V, tc_idesc(64), A_hi, A_lo, S.W1m_hi, S.W1m_lo, 1);
        }
        commit_wait();
        // ---- U = silu(V + b1) -> A tiles, HBM ----
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
            float v[16];
            tmem_ld16(tl + C_V + 16 * q, v);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = siluf_(v[i] + S.b1[16 * q + i]);
            to_tile(q, v);
            row_store16(a.U + row * 64, 64, 16 * q, ok, true, v);
        }
        tc_fence_before();
        publish();
        // ---- O = U . W2^T ----
        if (tid == 0) {
            tc_fence_after();
            issue_kblock<true>(tmem_grp + C_W, tc_idesc(64), A_hi, A_lo, S.W2_hi, S.W2_lo, 0);
        }
        commit_wait();
        // ---- attention, residual variants and their backward down to dO ----
        const float *ghrow = a.d_h_out + row * k;
        const float *hrow = a.h_in + row * k;
        float zdot = 0.0f, dsd = 0.0f, gho = 0.0f, ghh = 0.0f;
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
            float o[16], gh[16];
            tmem_ld16(tl + C_W + 16 * q, o);
            row_load16(ghrow, k, 16 * q, ok, vec, gh);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                o[i] += S.b2[16 * q + i];
                zdot = fmaf(S.wn[16 * q + i], o[i], zdot);
                const float do2 = f_rez ? gate * gh[i] : (f_gat ? G * gh[i] : gh[i]);
                dsd = fmaf(do2, o[i], dsd);
                gho = fmaf(gh[i], o[i], gho);
            }
            if (f_gat) {
                float hv[16];
                row_load16(hrow, k, 16 * q, ok, vec, hv);
#pragma unroll
                for (int i = 0; i < 16; ++i) ghh = fmaf(gh[i], hv[i], ghh);
            }
            row_store16(a.O + row * 64, 64, 16 * q, ok, true, o);
        }
        float s = 1.0f, dz = 0.0f;
        if (f_natt) {
            const float zn = zdot + natt_b;
            const bool soft = a.flags & PVS_F_SOFTMAX_ATTENTION;
            s = soft ? zn : apply_act(zn, a.att_act);
            dz = dsd * (soft ? 1.0f : act_grad(zn, s, a.att_act));
        }
        if (ok) {
            a.dzn[row0 + r] = dz;
            a.gdot[row0 + r] = f_rez ? s * gho : (f_gat ? (gate > 0.0f ? s * gho - ghh : 0.0f) : 0.0f);
        }
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
            float o[16], gh[16];
            tmem_ld16(tl + C_W + 16 * q, o);
            row_load16(ghrow, k, 16 * q, ok, vec, gh);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float do2 = f_rez ? gate * gh[i] : (f_gat ? G * gh[i] : gh[i]);
                o[i] = fmaf(dz, S.wn[16 * q + i], do2 * s);     // dO
            }
            to_tile(q, o);
            row_store16(a.DO + row * 64, 64, 16 * q, ok, true, o);
        }
        tc_fence_before();
        publish();
        // ---- dU = dO . W2 ----
        if (tid == 0) {
            tc_fence_after();
            issue_kblock_bmn(tmem_grp + C_W, A_hi, A_lo, S.W2_hi, S.W2_lo, 0);
        }
        commit_wait();
        // ---- dV = dU * silu'(V + b1) -> A tiles, HBM ----
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
            float du[16], v[16];
            tmem_ld16(tl + C_W + 16 * q, du);
            tmem_ld16(tl + C_V + 16 * q, v);
#pragma unroll
            for (int i = 0; i < 16; ++i)
                du[i] = (ok && 16 * q + i < k) ? du[i] * silu_gradf_(v[i] + S.b1[16 * q + i]) : 0.0f;
            to_tile(q, du);
            row_store16(a.DV + row * 64, 64, 16 * q, ok, true, du);
        }
        tc_fence_before();
        publish();           // every thread is done with V in tensor memory
        // ---- dh = dV . W1h -> work columns, dM = dV . W1m -> V's columns ----
        if (tid == 0) {
            tc_fence_after();
            issue_kblock_bmn(tmem_grp + C_W, A_hi, A_lo, S.W1h_hi, S.W1h_lo, 0);
            issue_kblock_bmn(tmem_grp + C_V, A_hi, A_lo, S.W1m_hi, S.W1m_lo, 0);
        }
        commit_wait();
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
            float dh[16], gh[16], dm[16];
            tmem_ld16(tl + C_W + 16 * q, dh);
            tmem_ld16(tl + C_V + 16 * q, dm);
            row_load16(ghrow, k, 16 * q, ok, vec, gh);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                // residual branch of dL/dh: gh (plain, rezero), (1 - G) gh (gated)
                const float dres = !f_res ? 0.0f : (f_gat ? (1.0f - G) * gh[i] : gh[i]);
                dh[i] += dres;
            }
            row_store16(a.d_h_in + row * k, k, 16 * q, ok, vec, dh);
            row_store16(a.dM + row * 64, 64, 16 * q, ok, true, dm);
        }
        tc_fence_before();
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc<512>(tmem_base);
}

int launch_node_bwd_tc(const NodeBwdArgs &a, cudaStream_t st) {
    const size_t smem = sizeof(NbSmem);
    int grid = num_sms();
    const int need = (a.n_nodes + 16 * NB_GROUPS - 1) / (16 * NB_GROUPS);
    if (need < grid) grid = need;
    if (grid < 1) grid = 1;
    const int rc = ensure_smem(node_bwd_tc_kernel, smem);
    if (rc) return rc;
    launch_chained(node_bwd_tc_kernel, dim3(grid), dim3(NB_THREADS), smem, st, a);
    return check_launch();
}

int launch_node_pre_tc(const float *h, const float *edge_w1, const float *edge_b1, float *P,
                       float *Q, int n_nodes, int k, int in_e, int perm, int mode,
                       cudaStream_t st) {
    if (k > 64)
        return launch_wide_node_pre_tc(h, edge_w1, edge_b1, P, Q, n_nodes, k, in_e, perm, mode, st);
    NodePreArgs a{};
    a.h = h; a.edge_w1 = edge_w1; a.edge_b1 = edge_b1; a.P = P; a.Q = Q;
    a.n_nodes = n_nodes; a.k = k; a.in_e = in_e; a.perm_invariant = perm;
    const size_t smem = sizeof(NpSmem);
    // one persistent CTA per SM; fewer only when a group's share would fall
    // under 16 rows
    int grid = num_sms();
    const int need = (n_nodes + 16 * NP_GROUPS - 1) / (16 * NP_GROUPS);
    if (need < grid) grid = need;
    if (grid < 1) grid = 1;
    // P and Q leave their tiles through tensor maps (boxes of tile_rows rows);
    // PVS_NO_TMA=1 keeps the thread-store path (A/B switch)
    static const bool no_tma = getenv("PVS_NO_TMA") != nullptr;
    int tile_rows, tiles;
    row_share_tiling(n_nodes, grid * NP_GROUPS, &tile_rows, &tiles);
    a.use_tma = !no_tma && make_rows_tensor_map(&a.tm_p, P, n_nodes, tile_rows) &&
                make_rows_tensor_map(&a.tm_q, Q, n_nodes, tile_rows);
    int rc;
    if (mode != PVS_MATH_BF16) {   // BF16X3, and the node stages of FP16X2
        rc = ensure_smem(node_pre_tc_kernel<true>, smem);
        if (rc) return rc;
        launch_chained(node_pre_tc_kernel<true>, dim3(grid), dim3(NP_THREADS), smem, st, a);
    } else {
        rc = ensure_smem(node_pre_tc_kernel<false>, smem);
        if (rc) return rc;
        launch_chained(node_pre_tc_kernel<false>, dim3(grid), dim3(NP_THREADS), smem, st, a);
    }
    return check_launch();
}

int launch_node_tc(const float *h_in, const float *M, float *h_out, float *natt_out,
                   const pvs_layer_params *p, int n_nodes, int k, uint32_t flags, int att_act,
                   int mode, cudaStream_t st, int phase, float *V, const float *gn_a,
                   const float *gn_b) {
    if (k > 64)
        return launch_wide_node_tc(h_in, M, h_out, natt_out, p, n_nodes, k, flags, att_act, mode,
                                   st, phase, V, gn_a, gn_b);
    NodeTcArgs a{};
    a.phase = phase; a.V = V; a.gn_a = gn_a; a.gn_b = gn_b;
    a.h_in = h_in; a.M = M; a.h_out = h_out; a.natt_out = natt_out;
    a.node_w1 = p->node_w1; a.node_b1 = p->node_b1; a.node_w2 = p->node_w2;
    a.node_b2 = p->node_b2; a.natt_w = p->natt_w; a.natt_b = p->natt_b;
    a.node_gate = p->node_gate;
    a.n_nodes = n_nodes; a.k = k; a.flags = flags; a.att_act = att_act;
    const size_t smem = sizeof(NmSmem);
    // one persistent CTA per SM; fewer only when a group's share would fall
    // under 16 rows
    int grid = num_sms();
    const int need = (n_nodes + 16 * NM_GROUPS - 1) / (16 * NM_GROUPS);
    if (need < grid) grid = need;
    if (grid < 1) grid = 1;
    // Opt-in (PVS_NODE_TC_TMA=1): h' through a tensor map when it is a [N][64]
    // array (k == 64).  Measured 1.4 % SLOWER on the scoring pass than the
    // staged thread stores: the residual then needs h per thread (a 256-byte row
    // each instead of full lines per half warp) and a second pass over TMEM,
    // which costs more than the store pass it removes (node_pre, whose output
    // needs neither, gains 0.4 % from its TMA stores).
    static const bool tma = getenv("PVS_NODE_TC_TMA") != nullptr;
    a.use_tma = 0;
    if (tma && k == 64 && phase != 1 && h_out != nullptr) {
        int tile_rows, tiles;
        row_share_tiling(n_nodes, grid * NM_GROUPS, &tile_rows, &tiles);
        a.use_tma = make_rows_tensor_map(&a.tm_h, h_out, n_nodes, tile_rows) ? 1 : 0;
    }
    int rc;
    if (mode != PVS_MATH_BF16) {   // BF16X3, and the node stages of FP16X2
        rc = ensure_smem(node_tc_kernel<true>, smem);
        if (rc) return rc;
        launch_chained(node_tc_kernel<true>, dim3(grid), dim3(NM_THREADS), smem, st, a);
    } else {
        rc = ensure_smem(node_tc_kernel<false>, smem);
        if (rc) return rc;
        launch_chained(node_tc_kernel<false>, dim3(grid), dim3(NM_THREADS), smem, st, a);
    }
    return check_launch();
}

}  // namespace pvs
