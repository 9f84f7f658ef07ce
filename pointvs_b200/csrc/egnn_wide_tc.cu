// Node stages of the 128-wide forward (65 <= k <= 128, tensor-core math modes).
//
//   node_pre : [P | Q] = h . [W1a ; W1b]^T (+ b1 on P)          K = 128, N = 128 each
//   node MLP : u = silu([h | M] . W1^T + b1)  (K = 2 x 128)      N = 128
//              h' = residual(h, s . (u . W2^T + b2)), s = node attention
//              GraphNorm models: phase 1 stops at V = [h | M] . W1^T + b1,
//              phase 2 resumes from V with the batch affine (gn_a, gn_b)
//
// Same tcgen05 machinery as egnn_node_tc.cu (K-major SWIZZLE_128B bf16 hi/lo
// tiles, fp32 accumulators in TMEM, one row per thread in the epilogues), but
// the weights do not fit beside the activation tiles at this width (W1 alone
// is 128 KB of hi/lo tiles), so a CTA keeps the two 64-channel K-blocks of its
// 128-row activation tile and streams one 128 x 64 weight K-block at a time
// from L2.  96 KB of shared memory and 128 TMEM columns per CTA: two CTAs per
// SM, one builds its tiles while the other's MMAs run.
#include "egnn_common.cuh"
#include "tc_common.cuh"

namespace pvs {
namespace {

constexpr int WN_THREADS = 128;   // one tile row per thread in the epilogues
constexpr int WN_ROWS = 128;      // UMMA M
constexpr int WK = 128;           // padded width: pitch of P, Q, M, V; UMMA N

struct __align__(1024) WnSmem {
    uint8_t A_hi[2][WN_ROWS * 128];   // activation K-blocks: channels [0, 64), [64, 128)
    uint8_t A_lo[2][WN_ROWS * 128];
    uint8_t B_hi[WK * 128];           // one weight K-block: 128 output rows x 64 inputs
    uint8_t B_lo[WK * 128];
    float b1[WK], b2[WK], wn[WK], ga[WK], gb[WK];
    uint64_t mbar;
    uint32_t tmem_base;
};

struct WideNodeArgs {
    int op;                  // 0: node_pre, 1: node MLP
    int phase;               // node MLP: 0 whole, 1 stop at V, 2 resume from V
    const float *h;          // [N][k]
    const float *M;          // [N][128]
    float *P, *Q;            // [N][128] (node_pre)
    float *V;                // [N][128] (GraphNorm phases 1 / 2)
    float *h_out;            // [N][k]
    float *natt_out;         // [N] or null
    const float *w1a, *w1b;  // node_pre: W1a, W1b; node MLP: W1[:, :k], W1[:, k:]
    int ld_w1;
    const float *b1, *w2, *b2, *natt_w, *natt_b, *node_gate, *gn_a, *gn_b;
    int n_nodes, k;
    uint32_t flags;
    int att_act;
};

// rows [row0, row0 + 128) x channels [0, 128) of src (pitch ld, k valid
// channels) -> the two activation K-blocks; GN: u = silu(ga v + gb) on the way
template <bool X3, bool GN>
__device__ void load_act(WnSmem &S, const float *__restrict__ src, int ld, int k, int row0,
                         int n_rows) {
    for (int idx = threadIdx.x; idx < WN_ROWS * 16; idx += WN_THREADS) {
        const int r = idx >> 4, c = idx & 15;   // 16 lanes per row, 8 channels each
        const bool rok = row0 + r < n_rows;
        const float *s = src + (size_t)(row0 + r) * ld + 8 * c;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int n = 8 * c + i;
            float x = (rok && n < k) ? __ldg(s + i) : 0.0f;
            if (GN) x = (rok && n < k) ? silu_mode<X3>(fmaf(S.ga[n], x, S.gb[n])) : 0.0f;
            v[i] = x;
        }
        uint4 hi, lo;
        split8<X3>(v, hi, lo);
        *reinterpret_cast<uint4 *>(S.A_hi[c >> 3] + swz(r, c & 7)) = hi;
        if (X3) *reinterpret_cast<uint4 *>(S.A_lo[c >> 3] + swz(r, c & 7)) = lo;
    }
}

// D (+)= A . W^T over both activation K-blocks, W = [k][ld] (k valid rows and
// input channels), one weight K-block at a time.  Whole CTA; returns with D
// complete and the tiles free.
template <bool X3>
__device__ void gemm_k128(WnSmem &S, uint32_t tmem_d, const float *__restrict__ W, int ld,
                          int k, uint32_t acc, uint32_t &phase) {
#pragma unroll 1
    for (int b = 0; b < 2; ++b) {
        load_weight_tiles<X3>(S.B_hi, S.B_lo, W + 64 * b, ld, k, k - 64 * b, WK);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (threadIdx.x == 0) {
            tc_fence_after();
            issue_kblock<X3>(tmem_d, tc_idesc(WK), S.A_hi[b], S.A_lo[b], S.B_hi, S.B_lo,
                             b ? 1u : acc);
            umma_commit(&S.mbar);
        }
        mbar_wait(&S.mbar, phase);
        phase ^= 1;
        tc_fence_after();
    }
}

// this thread's row of D (+ bias) -> out[row][0, 128)
__device__ __forceinline__ void store_row(uint32_t tmem_lane, const float *bias, float *out,
                                          bool ok) {
#pragma unroll 1
    for (int q = 0; q < WK / 16; ++q) {
        float acc[16];
        tmem_ld16(tmem_lane + 16 * q, acc);
        if (!ok) continue;
        float4 *dst = reinterpret_cast<float4 *>(out + 16 * q);
#pragma unroll
        for (int v4 = 0; v4 < 4; ++v4) {
            const int n = 16 * q + 4 * v4;
            dst[v4] = make_float4(acc[4 * v4] + bias[n], acc[4 * v4 + 1] + bias[n + 1],
                                  acc[4 * v4 + 2] + bias[n + 2], acc[4 * v4 + 3] + bias[n + 3]);
        }
    }
}

template <bool X3>
__global__ void __launch_bounds__(WN_THREADS, 1)
wide_node_tc_kernel(const WideNodeArgs a) {
    extern __shared__ __align__(1024) uint8_t smem_dyn[];
    WnSmem &S = *reinterpret_cast<WnSmem *>(smem_dyn);
    pdl_launch_dependents();
    if ((smem_u32(smem_dyn) & 1023u) != 0u) __trap();
    const int tid = threadIdx.x, warp = tid >> 5;
    const int k = a.k;
    if (tid == 0) mbar_init(&S.mbar, 1);
    if (warp == 0) tmem_alloc<WK>(&S.tmem_base);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_d = S.tmem_base;
    const uint32_t tmem_lane = tmem_d + ((uint32_t)(warp * 32) << 16);
    pdl_wait();      // h, M, V and the GraphNorm affine of the kernels before this one
    for (int n = tid; n < WK; n += WN_THREADS) {
        const bool ok = n < k;
        S.b1[n] = (ok && a.b1) ? a.b1[n] : 0.0f;
        S.b2[n] = (ok && a.b2) ? a.b2[n] : 0.0f;
        S.wn[n] = (ok && a.natt_w) ? a.natt_w[n] : 0.0f;
        S.ga[n] = (ok && a.gn_a) ? a.gn_a[n] : 1.0f;
        S.gb[n] = (ok && a.gn_b) ? a.gn_b[n] : 0.0f;
    }
    __syncthreads();
    const bool f_natt = (a.flags & PVS_F_NODE_ATTENTION) && a.natt_w != nullptr;
    const bool f_res = a.flags & PVS_F_RESIDUAL;
    const float natt_b = (f_natt && a.natt_b) ? a.natt_b[0] : 0.0f;
    const float gate = a.node_gate ? a.node_gate[0] : 1.0f;
    uint32_t phase = 0;
    for (int row0 = blockIdx.x * WN_ROWS; row0 < a.n_nodes; row0 += gridDim.x * WN_ROWS) {
        const int r = tid, row = row0 + r;
        const bool ok = row < a.n_nodes;
        __syncthreads();     // the previous tile's epilogue is done with the A tiles
        if (a.op == 0) {
            // ---- [P | Q]: padded channels come out zero (zero weight rows and bias) ----
            load_act<X3, false>(S, a.h, k, k, row0, a.n_nodes);
            gemm_k128<X3>(S, tmem_d, a.w1a, a.ld_w1, k, 0, phase);
            store_row(tmem_lane, S.b1, a.P + (size_t)row * WK, ok);
            gemm_k128<X3>(S, tmem_d, a.w1b, a.ld_w1, k, 0, phase);
            store_row(tmem_lane, S.b2, a.Q + (size_t)row * WK, ok);   // b2 = 0 here
            continue;
        }
        if (a.phase != 2) {
            // ---- v = W1 [h ; M] + b1: h, then M through the same tiles ----
            load_act<X3, false>(S, a.h, k, k, row0, a.n_nodes);
            gemm_k128<X3>(S, tmem_d, a.w1a, a.ld_w1, k, 0, phase);
            __syncthreads();
            load_act<X3, false>(S, a.M, WK, k, row0, a.n_nodes);
            gemm_k128<X3>(S, tmem_d, a.w1b, a.ld_w1, k, 1, phase);
            if (a.phase == 1) {
                store_row(tmem_lane, S.b1, a.V + (size_t)row * WK, ok);
                continue;
            }
            // ---- u = silu(v + b1) -> A tiles (free: GEMM 1 has completed) ----
#pragma unroll 1
            for (int q = 0; q < WK / 16; ++q) {
                float acc[16];
                tmem_ld16(tmem_lane + 16 * q, acc);
#pragma unroll
                for (int hlf = 0; hlf < 2; ++hlf) {
                    const int c = 2 * q + hlf;
                    float u[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        u[i] = silu_mode<X3>(acc[8 * hlf + i] + S.b1[8 * c + i]);
                    uint4 hi, lo;
                    split8<X3>(u, hi, lo);
                    *reinterpret_cast<uint4 *>(S.A_hi[c >> 3] + swz(r, c & 7)) = hi;
                    if (X3) *reinterpret_cast<uint4 *>(S.A_lo[c >> 3] + swz(r, c & 7)) = lo;
                }
            }
        } else {
            load_act<X3, true>(S, a.V, WK, k, row0, a.n_nodes);
        }
        // ---- o = u W2^T + b2, node attention, residual ----
        gemm_k128<X3>(S, tmem_d, a.w2, k, k, 0, phase);
        float s = 1.0f;
        if (f_natt) {
            float dot = 0.0f;
#pragma unroll 1
            for (int q = 0; q < WK / 16; ++q) {
                float acc[16];
                tmem_ld16(tmem_lane + 16 * q, acc);
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    dot = fmaf(S.wn[16 * q + i], acc[i] + S.b2[16 * q + i], dot);
            }
            const float zn = dot + natt_b;
            s = (a.flags & PVS_F_SOFTMAX_ATTENTION) ? zn : apply_act(zn, a.att_act);
            if (a.natt_out && ok) a.natt_out[row] = s;
        }
        const float G = fmaxf(gate, 0.0f);
        const float *hrow = a.h + (size_t)(ok ? row : 0) * k;
        float *orow = a.h_out + (size_t)(ok ? row : 0) * k;
#pragma unroll 1
        for (int q = 0; q < WK / 16; ++q) {
            float acc[16];
            tmem_ld16(tmem_lane + 16 * q, acc);
            if (!ok) continue;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int n = 16 * q + i;
                if (n >= k) break;
                float o = s * (acc[i] + S.b2[n]);
                if (f_res) {
                    const float hv = hrow[n];
                    if (a.flags & PVS_F_REZERO) o = hv + gate * o;
                    else if (a.flags & PVS_F_GATED_RESIDUAL) o = G * o + (1.0f - G) * hv;
                    else o = hv + o;
                }
                orow[n] = o;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc<WK>(tmem_d);
}

int launch_wide(const WideNodeArgs &a, int mode, cudaStream_t st) {
    static_assert(2 * sizeof(WnSmem) <= 227 * 1024, "two CTAs per SM");
    const size_t smem = sizeof(WnSmem);
    int grid = 2 * num_sms();
    const int tiles = (a.n_nodes + WN_ROWS - 1) / WN_ROWS;
    if (tiles < grid) grid = tiles;
    if (grid < 1) return PVS_OK;
    int rc;
    if (mode != PVS_MATH_BF16) {   // BF16X3, and the node stages of FP16X2
        rc = ensure_smem(wide_node_tc_kernel<true>, smem);
        if (rc) return rc;
        launch_chained(wide_node_tc_kernel<true>, dim3(grid), dim3(WN_THREADS), smem, st, a);
    } else {
        rc = ensure_smem(wide_node_tc_kernel<false>, smem);
        if (rc) return rc;
        launch_chained(wide_node_tc_kernel<false>, dim3(grid), dim3(WN_THREADS), smem, st, a);
    }
    return check_launch();
}

}  // namespace

int launch_wide_node_pre_tc(const float *h, const float *edge_w1, const float *edge_b1, float *P,
                            float *Q, int n_nodes, int k, int in_e, int perm, int mode,
                            cudaStream_t st) {
    WideNodeArgs a{};
    a.op = 0;
    a.h = h; a.P = P; a.Q = Q;
    a.w1a = edge_w1; a.w1b = edge_w1 + (perm ? 0 : k); a.ld_w1 = in_e;
    a.b1 = edge_b1;
    a.n_nodes = n_nodes; a.k = k;
    return launch_wide(a, mode, st);
}

int launch_wide_node_tc(const float *h_in, const float *M, float *h_out, float *natt_out,
                        const pvs_layer_params *p, int n_nodes, int k, uint32_t flags,
                        int att_act, int mode, cudaStream_t st, int phase, float *V,
                        const float *gn_a, const float *gn_b) {
    WideNodeArgs a{};
    a.op = 1; a.phase = phase;
    a.h = h_in; a.M = M; a.V = V; a.h_out = h_out; a.natt_out = natt_out;
    a.w1a = p->node_w1; a.w1b = p->node_w1 + k; a.ld_w1 = 2 * k;
    a.b1 = p->node_b1; a.w2 = p->node_w2; a.b2 = p->node_b2;
    a.natt_w = p->natt_w; a.natt_b = p->natt_b; a.node_gate = p->node_gate;
    a.gn_a = gn_a; a.gn_b = gn_b;
    a.n_nodes = n_nodes; a.k = k; a.flags = flags; a.att_act = att_act;
    return launch_wide(a, mode, st);
}

}  // namespace pvs
