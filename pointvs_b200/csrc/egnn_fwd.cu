// K2 (PVS_MATH_FP32): one EGNN layer forward, plus the dense helpers
// (embedding / heads / mean pool).
//
// Replaces EGNNLayer.forward, /root/reference/point_vs/models/geometric/
// egnn_satorras.py:189-206 (coord2radial :178-187, edge_model :123-132,
// coord_model :168-176, node_model :134-166, segment sum/mean :332-347).
//
// Dataflow per layer (all fp32):
//   node_pre : P = h.W1a^T + b1, Q = h.W1b^T           (edge L1 factorised
//              per node: W1.[h_i;h_j;r;onehot] = P_i + Q_j + w_r r + T[attr])
//   edge     : per work tile of <=128 dst-sorted edges:
//              s1 = silu(P_i+Q_j+w_r r+T[a]) -> m = silu(W2 s1+b2)
//              -> c = [tanh] wc2.silu(Wc1 m+bc1), alpha = act(wa.m+ba)
//              -> M_i = sum alpha m (segment reduce, no atomics),
//                 x_i' = x_i + mean(d_hat c)
//   node     : o = Wn2 silu([gn](Wn1 [h;M] + bn1)) + bn2, node attention,
//              residual
#include "pvs_common.cuh"
#include "tile_gemm.cuh"
#include "egnn_common.cuh"

namespace pvs {

constexpr int FWD_THREADS = 256;
constexpr int NODE_ROWS = 64;

// ---------------------------------------------------------------------------
// generic linear: out = act(in . W^T + b), persistent over 64-row tiles
// ---------------------------------------------------------------------------
template <int NJ4>
__global__ void __launch_bounds__(FWD_THREADS)
linear_fwd_kernel(const float *__restrict__ in, int ld_in, int rows, int ki,
                  const float *__restrict__ W, int ld_w,
                  const float *__restrict__ b, int ko, int act,
                  float *__restrict__ out, int ld_out, int w_in_major,
                  int accumulate) {
    pdl_wait();                  // chain kernel: see pvs_common.cuh
    pdl_launch_dependents();
    extern __shared__ __align__(16) float smem[];
    constexpr int LDW = 64 * NJ4;
    const int KIP = (ki + 3) & ~3;
    const int lda = KIP + 4;
    float *Wt = smem;                  // [KIP][LDW]
    float *A = Wt + KIP * LDW;         // [64][lda]
    float *bias = A + NODE_ROWS * lda; // [LDW]
    if (w_in_major) {   // W given as [ki][ko] (backward: out = in . W)
        for (int idx = threadIdx.x; idx < KIP * LDW; idx += blockDim.x) {
            int kk = idx / LDW, n = idx - kk * LDW;
            Wt[idx] = (kk < ki && n < ko) ? W[(size_t)kk * ld_w + n] : 0.0f;
        }
    } else {
        load_wt(Wt, KIP, LDW, W, ld_w, ki, ko);
    }
    for (int n = threadIdx.x; n < LDW; n += blockDim.x)
        bias[n] = (b != nullptr && n < ko) ? b[n] : 0.0f;
    const int rg = threadIdx.x >> 4, cg = threadIdx.x & 15;
    const int n_tiles = (rows + NODE_ROWS - 1) / NODE_ROWS;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int r0 = t * NODE_ROWS;
        __syncthreads();
        for (int idx = threadIdx.x; idx < NODE_ROWS * KIP; idx += blockDim.x) {
            int r = idx / KIP, c = idx - r * KIP;
            A[r * lda + c] = (r0 + r < rows && c < ki)
                                 ? in[(size_t)(r0 + r) * ld_in + c] : 0.0f;
        }
        __syncthreads();
        float acc[4][NJ4][4] = {};
        tile_gemm<4, NJ4>(A, lda, Wt, KIP, acc);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = r0 + rg + 16 * i;
            if (r >= rows) continue;
#pragma unroll
            for (int j = 0; j < NJ4; ++j)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int n = 4 * cg + 64 * j + c;
                    if (n < ko) {
                        float v = apply_act(acc[i][j][c] + bias[n], act);
                        float *dst = &out[(size_t)r * ld_out + n];
                        *dst = accumulate ? *dst + v : v;
                    }
                }
        }
    }
}

// ---------------------------------------------------------------------------
// linear with a short input (the atom-feature embedding: ki = 13..32 -> 64):
// streaming, one thread per (row, four output columns), 64 rows per block; the
// weights sit in shared memory, a row's inputs are broadcast loads.  The
// generic kernel stages 64-row tiles for a K = 13 product and spent 33 us on
// what is a 40 MB copy.  Same accumulation order (k ascending, bias last).
// ---------------------------------------------------------------------------
constexpr int LSK_MAX_KI = 32;
__global__ void __launch_bounds__(256)
linear_smallk_kernel(const float *__restrict__ in, int ld_in, int rows, int ki,
                     const float *__restrict__ W, int ld_w, const float *__restrict__ b,
                     int ko, int act, float *__restrict__ out, int ld_out) {
    pdl_wait();                  // chain kernel: see pvs_common.cuh
    pdl_launch_dependents();
    __shared__ __align__(16) float Ws[LSK_MAX_KI][64];
    __shared__ __align__(16) float bs[64];
    for (int idx = threadIdx.x; idx < ki * 64; idx += blockDim.x) {
        const int kk = idx >> 6, n = idx & 63;
        Ws[kk][n] = n < ko ? W[(size_t)n * ld_w + kk] : 0.0f;
    }
    if (threadIdx.x < 64) bs[threadIdx.x] = (b != nullptr && threadIdx.x < ko) ? b[threadIdx.x] : 0.0f;
    __syncthreads();
    const int cg = threadIdx.x & 15, rg = threadIdx.x >> 4;
    const bool vec = (ld_out & 3) == 0 && (ko & 3) == 0 &&
                     (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    // the 16 lanes of a row fetch its inputs once (one or two coalesced loads)
    // and pass them round by shuffle; a weight vector read from shared memory
    // serves the thread's four rows
    float xa[4], xb[4], acc[4][4] = {};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = blockIdx.x * 64 + rg + 16 * i;
        const bool ok = r < rows;
        const float *x = in + (size_t)(ok ? r : 0) * ld_in;
        xa[i] = (ok && cg < ki) ? __ldg(x + cg) : 0.0f;
        xb[i] = (ok && 16 + cg < ki) ? __ldg(x + 16 + cg) : 0.0f;
    }
    for (int kk = 0; kk < ki; ++kk) {
        const float4 w4 = *reinterpret_cast<const float4 *>(&Ws[kk][4 * cg]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float xv = __shfl_sync(0xffffffffu, kk < 16 ? xa[i] : xb[i], kk & 15, 16);
            acc[i][0] = fmaf(xv, w4.x, acc[i][0]); acc[i][1] = fmaf(xv, w4.y, acc[i][1]);
            acc[i][2] = fmaf(xv, w4.z, acc[i][2]); acc[i][3] = fmaf(xv, w4.w, acc[i][3]);
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = blockIdx.x * 64 + rg + 16 * i;
        if (r >= rows) continue;
        float v[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) v[c] = apply_act(acc[i][c] + bs[4 * cg + c], act);
        float *dst = out + (size_t)r * ld_out + 4 * cg;
        if (vec && 4 * cg + 3 < ko) {
            *reinterpret_cast<float4 *>(dst) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (4 * cg + c < ko) dst[c] = v[c];
        }
    }
}

// ---------------------------------------------------------------------------
// mean pool: one CTA per graph
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
mean_pool_kernel(const float *__restrict__ h, const int32_t *__restrict__ ptr,
                 int k, float *__restrict__ pooled) {
    __shared__ float part[4][64];
    __shared__ __align__(16) float part16[16][64];
    const int g = blockIdx.x;
    const int lo = ptr[g], hi = ptr[g + 1];
    if (k == 64 && (reinterpret_cast<uintptr_t>(h) & 15) == 0) {
        // 16 lanes x float4 per row, 16 rows in flight per step, two steps
        // unrolled; partials added in a fixed order
        const int c4 = threadIdx.x & 15, rgp = threadIdx.x >> 4;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s;
        int r = lo + rgp;
        for (; r + 16 < hi; r += 32) {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(h + (size_t)r * 64) + c4);
            const float4 b = __ldg(reinterpret_cast<const float4 *>(h + (size_t)(r + 16) * 64) + c4);
            s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
            s2.x += b.x; s2.y += b.y; s2.z += b.z; s2.w += b.w;
        }
        if (r < hi) {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(h + (size_t)r * 64) + c4);
            s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
        }
        *reinterpret_cast<float4 *>(&part16[rgp][4 * c4]) =
            make_float4(s.x + s2.x, s.y + s2.y, s.z + s2.z, s.w + s2.w);
        __syncthreads();
        if (threadIdx.x < 64) {
            float tot = 0.0f;
#pragma unroll
            for (int q = 0; q < 16; ++q) tot += part16[q][threadIdx.x];
            const int cnt = hi - lo;
            pooled[(size_t)g * 64 + threadIdx.x] = tot / (float)(cnt > 0 ? cnt : 1);
        }
        return;
    }
    const int cl = threadIdx.x & 63, grp = threadIdx.x >> 6;
    for (int c0 = 0; c0 < k; c0 += 64) {
        const int c = c0 + cl;
        float s = 0.0f;
        if (c < k)
            for (int r = lo + grp; r < hi; r += 4) s += h[(size_t)r * k + c];
        part[grp][cl] = s;
        __syncthreads();
        if (grp == 0 && c < k) {
            float tot = (part[0][cl] + part[1][cl]) + (part[2][cl] + part[3][cl]);
            int cnt = hi - lo;
            pooled[(size_t)g * k + c] = tot / (float)(cnt > 0 ? cnt : 1);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// edge kernel
// ---------------------------------------------------------------------------
template <int KP>
struct EdgeSmem {
    static constexpr int LDA = KP + 4;
    float W2t[KP * 64];
    float Wc1t[KP * 64];
    float A1[TE * LDA];
    float A2[TE * LDA];
    float b2[64], bc1[64], wc2[64], wa[64], wr[64];
    float T[PVS_MAX_EDGE_CLASSES][64];
    float e_rad[TE], e_dx[TE], e_dy[TE], e_dz[TE], e_z[TE], e_c[TE], e_alpha[TE];
    int e_rowl[TE], e_col[TE], e_attr[TE];
    int rp[TN + 1];
    float xsum[TN][3];
};

template <int KP>
__global__ void __launch_bounds__(FWD_THREADS, (KP <= 64 ? 2 : 1))
egnn_edge_fwd_kernel(const EdgeArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EdgeSmem<KP> &S = *reinterpret_cast<EdgeSmem<KP> *>(smem_raw);
    constexpr int LDA = EdgeSmem<KP>::LDA;
    constexpr int CPL = KP / 32;   // channels per lane in the gather stage
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rg = tid >> 4, cg = tid & 15;
    const int k = a.k;
    const bool f_att = a.flags & PVS_F_EDGE_ATTENTION;
    const bool f_softmax = f_att && (a.flags & PVS_F_SOFTMAX_ATTENTION);
    const bool f_coords = (a.flags & PVS_F_UPDATE_COORDS) && a.x_out != nullptr;
    const bool f_eres = (a.flags & PVS_F_EDGE_RESIDUAL) && a.m_prev != nullptr;

    // ---- parameters -> smem (once per CTA) ----
    load_wt(S.W2t, KP, 64, a.edge_w2, k, k, k);
    load_wt(S.Wc1t, KP, 64, a.coord_w1, k, k, k);
    const int col_r = (a.flags & PVS_F_PERM_INVARIANT) ? k : 2 * k;
    for (int n = tid; n < 64; n += FWD_THREADS) {
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
    const float att_b = (f_att && a.att_b) ? a.att_b[0] : 0.0f;
    float gate = 1.0f;
    if (f_eres && a.edge_gate) gate = a.edge_gate[0];
    const int n_tiles = *a.n_tiles;
    __syncthreads();

    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int n0 = a.tile_ptr[t], n1 = a.tile_ptr[t + 1];
        const int nn = n1 - n0;
        __syncthreads();   // previous tile fully consumed
        for (int i = tid; i <= nn; i += FWD_THREADS) S.rp[i] = a.row_ptr[n0 + i];
        for (int i = tid; i < nn * 3; i += FWD_THREADS) (&S.xsum[0][0])[i] = 0.0f;
        __syncthreads();
        const int e0 = S.rp[0], e1 = S.rp[nn];

        const int n_chunks = max(1, (e1 - e0 + TE - 1) / TE);
        for (int ch = 0; ch < n_chunks; ++ch) {
            const int c0 = e0 + ch * TE;
            const int ne = min(TE, e1 - c0);   // 0 only for an edgeless tile
            if (ne > 0) {
            // ---- stage 0: per-edge geometry ----
            if (tid < TE) {
                if (tid < ne) {
                    const int e = c0 + tid;
                    int lo = 0, hi = nn;   // last node with rp[node] <= e
                    while (hi - lo > 1) {
                        int mid = (lo + hi) >> 1;
                        if (S.rp[mid] <= e) lo = mid; else hi = mid;
                    }
                    const int i = n0 + lo, j = a.col[e];
                    float dx = a.x_in[3 * i] - a.x_in[3 * j];
                    float dy = a.x_in[3 * i + 1] - a.x_in[3 * j + 1];
                    float dz = a.x_in[3 * i + 2] - a.x_in[3 * j + 2];
                    float r = dx * dx + dy * dy + dz * dz;   // :181
                    if (a.flags & PVS_F_NORMALIZE) {          // :183-185
                        float inv = 1.0f / (sqrtf(r) + 1e-8f);
                        dx *= inv; dy *= inv; dz *= inv;
                    }
                    S.e_rowl[tid] = lo;
                    S.e_col[tid] = j;
                    S.e_attr[tid] = a.attr ? a.attr[e] : 0;
                    S.e_rad[tid] = r;
                    S.e_dx[tid] = dx; S.e_dy[tid] = dy; S.e_dz[tid] = dz;
                } else {
                    S.e_rowl[tid] = -1;
                }
            }
            __syncthreads();
            // ---- stage 1: s1 = silu(P_i + Q_j + w_r r + T[attr]) -> A1 ----
            for (int el = warp; el < TE; el += FWD_THREADS / 32) {
                float v[CPL];
                if (el < ne) {
                    const float *p = a.P + (size_t)(n0 + S.e_rowl[el]) * KP + CPL * lane;
                    const float *q = a.Q + (size_t)S.e_col[el] * KP + CPL * lane;
                    const float r = S.e_rad[el];
                    const int at = S.e_attr[el];
                    float pv[CPL], qv[CPL];
                    if constexpr (CPL == 2) {
                        const float2 p2 = __ldg(reinterpret_cast<const float2 *>(p));
                        const float2 q2 = __ldg(reinterpret_cast<const float2 *>(q));
                        pv[0] = p2.x; pv[1] = p2.y; qv[0] = q2.x; qv[1] = q2.y;
                    } else {
                        pv[0] = __ldg(p); qv[0] = __ldg(q);
                    }
#pragma unroll
                    for (int c = 0; c < CPL; ++c) {
                        const int chn = CPL * lane + c;
                        float t1 = pv[c] + qv[c];
                        t1 = fmaf(S.wr[chn], r, t1) + S.T[at][chn];
                        v[c] = siluf_(t1);
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < CPL; ++c) v[c] = 0.0f;
                }
#pragma unroll
                for (int c = 0; c < CPL; ++c) S.A1[el * LDA + CPL * lane + c] = v[c];
            }
            __syncthreads();
            const bool active = 4 * cg < KP;
            // ---- stage 2: m = silu(W2 s1 + b2) (+ edge residual) -> A2 ----
            {
                float acc[8][1][4] = {};
                if (active) tile_gemm<8, 1>(S.A1, LDA, S.W2t, KP, acc);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = rg + 16 * i;
                    float dot = 0.0f;
                    if (active) {
                        float mv[4];
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const int n = 4 * cg + c;
                            float m = siluf_(acc[i][0][c] + S.b2[n]);
                            if (f_eres && r < ne && n < k) {   // :194-202
                                float mp = a.m_prev[(size_t)(c0 + r) * k + n];
                                if (a.flags & PVS_F_REZERO) m = mp + gate * m;
                                else if (a.flags & PVS_F_GATED_RESIDUAL) {
                                    float g = fmaxf(gate, 0.0f);
                                    m = g * m + (1.0f - g) * mp;
                                } else m = m + mp;
                            }
                            if (n >= k || r >= ne) m = 0.0f;
                            mv[c] = m;
                            dot = fmaf(S.wa[n], m, dot);
                        }
                        *reinterpret_cast<float4 *>(&S.A2[r * LDA + 4 * cg]) =
                            make_float4(mv[0], mv[1], mv[2], mv[3]);
                    }
                    if (f_att) {
                        dot = rowgroup_sum(dot);
                        if (cg == 0) S.e_z[r] = dot + att_b;
                    }
                }
            }
            __syncthreads();
            // ---- stage 3: c = [tanh](wc2 . silu(Wc1 m + bc1)) ----
            if (f_coords) {
                float acc[8][1][4] = {};
                if (active) tile_gemm<8, 1>(S.A2, LDA, S.Wc1t, KP, acc);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = rg + 16 * i;
                    float dot = 0.0f;
                    if (active) {
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const int n = 4 * cg + c;
                            dot = fmaf(S.wc2[n], siluf_(acc[i][0][c] + S.bc1[n]), dot);
                        }
                    }
                    dot = rowgroup_sum(dot);
                    if (cg == 0)
                        S.e_c[r] = (a.flags & PVS_F_TANH) ? tanhf(dot) : dot;
                }
            }
            }   // ne > 0
            // ---- stage 4a: attention value per edge ----
            if (tid < ne) {
                float al = 1.0f;
                if (f_att) {
                    const float z = S.e_z[tid];
                    al = f_softmax ? z : apply_act(z, a.att_act);
                    if (a.att_out) a.att_out[c0 + tid] = al;
                }
                S.e_alpha[tid] = al;
            }
            __syncthreads();
            // ---- stage 4b: M_i = sum_e alpha_e m_e over dst segments ----
            if (!f_softmax) {
                for (int nl = warp; nl < nn; nl += FWD_THREADS / 32) {
                    const int lo = max(S.rp[nl], c0) - c0;
                    const int hi = min(S.rp[nl + 1], c0 + TE) - c0;
                    float s[CPL];
#pragma unroll
                    for (int c = 0; c < CPL; ++c) s[c] = 0.0f;
                    for (int el = lo; el < hi; ++el) {
                        const float al = S.e_alpha[el];
#pragma unroll
                        for (int c = 0; c < CPL; ++c)
                            s[c] = fmaf(al, S.A2[el * LDA + CPL * lane + c], s[c]);
                    }
                    float *dst = a.M + (size_t)(n0 + nl) * KP + CPL * lane;
                    if (c0 == e0) {
#pragma unroll
                        for (int c = 0; c < CPL; ++c) dst[c] = s[c];
                    } else if (hi > lo) {
#pragma unroll
                        for (int c = 0; c < CPL; ++c) dst[c] += s[c];
                    }
                }
            }
            // ---- stage 4c: messages out (next layer's m_prev / softmax pass)
            if (a.m_out != nullptr) {
                for (int idx = tid; idx < ne * KP; idx += FWD_THREADS) {
                    const int el = idx / KP, c = idx - el * KP;
                    if (c < a.ld_m)
                        a.m_out[(size_t)(c0 + el) * a.ld_m + c] = S.A2[el * LDA + c];
                }
            }
            // ---- stage 4d: coordinate messages, summed per node ----
            if (f_coords && tid < nn) {
                const int lo = max(S.rp[tid], c0) - c0;
                const int hi = min(S.rp[tid + 1], c0 + TE) - c0;
                float sx = 0.f, sy = 0.f, sz = 0.f;
                for (int el = lo; el < hi; ++el) {
                    const float c = S.e_c[el];
                    sx = fmaf(S.e_dx[el], c, sx);
                    sy = fmaf(S.e_dy[el], c, sy);
                    sz = fmaf(S.e_dz[el], c, sz);
                }
                S.xsum[tid][0] += sx;
                S.xsum[tid][1] += sy;
                S.xsum[tid][2] += sz;
            }
            __syncthreads();
        }
        // ---- x' = x + mean (count clamped at 1, :340-347) ----
        if (a.x_out != nullptr && tid < nn) {
            const int i = n0 + tid;
            const int cnt = S.rp[tid + 1] - S.rp[tid];
            const float inv = 1.0f / (float)(cnt > 0 ? cnt : 1);
            float ax = 0.f, ay = 0.f, az = 0.f;
            if (f_coords) {
                ax = S.xsum[tid][0] * inv;
                ay = S.xsum[tid][1] * inv;
                az = S.xsum[tid][2] * inv;
            }
            a.x_out[3 * i] = a.x_in[3 * i] + ax;
            a.x_out[3 * i + 1] = a.x_in[3 * i + 1] + ay;
            a.x_out[3 * i + 2] = a.x_in[3 * i + 2] + az;
        }
    }
}

// softmax attention (egnn_satorras.py:139-147): alpha = softmax over each dst
// segment of the logits, M_i = sum alpha m.  One warp per node.
__global__ void __launch_bounds__(256)
segment_softmax_agg_kernel(const int32_t *__restrict__ row_ptr, int n_nodes,
                           const float *__restrict__ m, int ld_m, int kp,
                           float *__restrict__ att /* in: logits, out: alpha */,
                           float *__restrict__ M) {
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= n_nodes) return;
    const int lo = row_ptr[i], hi = row_ptr[i + 1];
    float mx = -INFINITY;
    for (int e = lo + lane; e < hi; e += 32) mx = fmaxf(mx, att[e]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float den = 0.0f;
    for (int e = lo + lane; e < hi; e += 32) den += expf(att[e] - mx);
    den = warp_sum(den);
    __syncwarp();
    for (int e = lo + lane; e < hi; e += 32) att[e] = expf(att[e] - mx) / den;
    __syncwarp();
    for (int c = lane; c < kp; c += 32) {
        float s = 0.0f;
        if (c < ld_m)
            for (int e = lo; e < hi; ++e) s = fmaf(att[e], m[(size_t)e * ld_m + c], s);
        M[(size_t)i * kp + c] = s;
    }
}

// ---------------------------------------------------------------------------
// node kernel
// ---------------------------------------------------------------------------
struct NodeArgs {
    const float *h_in;   // [N][k]
    const float *M;      // [N][KP]
    float *h_out;        // [N][k]
    float *V;            // [N][KP] graphnorm pre-activation (phase 1 out / 2 in)
    const float *gn_a, *gn_b;   // [KP] affine of the normalisation (phase 2)
    float *natt_out;     // [N] or null
    const float *node_w1, *node_b1, *node_w2, *node_b2, *natt_w, *natt_b, *node_gate;
    int n_nodes, k;
    uint32_t flags;
    int att_act;
    int phase;           // 0: whole node model, 1: stop after Wn1 (write V),
                         // 2: resume from V
};

template <int KP>
__global__ void __launch_bounds__(FWD_THREADS)
egnn_node_fwd_kernel(const NodeArgs a) {
    extern __shared__ __align__(16) float smem[];
    constexpr int LDIN = 2 * KP + 4;
    constexpr int LDU = KP + 4;
    float *W1t = smem;                      // [2KP][64]
    float *W2t = W1t + 2 * KP * 64;         // [KP][64]
    float *IN = W2t + KP * 64;              // [64][LDIN]  = [h | M]
    float *U = IN + NODE_ROWS * LDIN;       // [64][LDU]
    float *b1 = U + NODE_ROWS * LDU;        // [64]
    float *b2 = b1 + 64, *wn = b2 + 64, *ga = wn + 64, *gb = ga + 64;
    const int tid = threadIdx.x, rg = tid >> 4, cg = tid & 15;
    const int k = a.k;
    // W1 is [k][2k]: columns [0,k) multiply h, [k,2k) multiply M (:150)
    for (int idx = tid; idx < 2 * KP * 64; idx += FWD_THREADS) {
        int kk = idx >> 6, n = idx & 63;
        int src = kk < KP ? kk : k + (kk - KP);
        bool ok = n < k && (kk < KP ? kk < k : (kk - KP) < k);
        W1t[idx] = ok ? a.node_w1[(size_t)n * 2 * k + src] : 0.0f;
    }
    load_wt(W2t, KP, 64, a.node_w2, k, k, k);
    for (int n = tid; n < 64; n += FWD_THREADS) {
        const bool ok = n < k;
        b1[n] = ok ? a.node_b1[n] : 0.0f;
        b2[n] = ok ? a.node_b2[n] : 0.0f;
        wn[n] = (ok && a.natt_w) ? a.natt_w[n] : 0.0f;
        ga[n] = (ok && a.gn_a) ? a.gn_a[n] : 1.0f;
        gb[n] = (ok && a.gn_b) ? a.gn_b[n] : 0.0f;
    }
    const bool f_natt = (a.flags & PVS_F_NODE_ATTENTION) && a.natt_w != nullptr;
    const float natt_b = (f_natt && a.natt_b) ? a.natt_b[0] : 0.0f;
    const float gate = a.node_gate ? a.node_gate[0] : 1.0f;
    const int n_tiles = (a.n_nodes + NODE_ROWS - 1) / NODE_ROWS;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const int r0 = t * NODE_ROWS;
        __syncthreads();
        for (int idx = tid; idx < NODE_ROWS * KP; idx += FWD_THREADS) {
            int r = idx / KP, c = idx - r * KP;
            bool ok = r0 + r < a.n_nodes;
            IN[r * LDIN + c] = (ok && c < k) ? a.h_in[(size_t)(r0 + r) * k + c] : 0.0f;
            if (a.phase != 2)
                IN[r * LDIN + KP + c] = ok ? a.M[(size_t)(r0 + r) * KP + c] : 0.0f;
        }
        __syncthreads();
        if (4 * cg < KP) {
            if (a.phase != 2) {
                float acc[4][1][4] = {};
                tile_gemm<4, 1>(IN, LDIN, W1t, 2 * KP, acc);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int r = rg + 16 * i;
                    float v[4];
#pragma unroll
                    for (int c = 0; c < 4; ++c) v[c] = acc[i][0][c] + b1[4 * cg + c];
                    if (a.phase == 1) {
                        if (r0 + r < a.n_nodes)
                            *reinterpret_cast<float4 *>(
                                &a.V[(size_t)(r0 + r) * KP + 4 * cg]) =
                                make_float4(v[0], v[1], v[2], v[3]);
                    } else {
                        *reinterpret_cast<float4 *>(&U[r * LDU + 4 * cg]) =
                            make_float4(siluf_(v[0]), siluf_(v[1]), siluf_(v[2]),
                                        siluf_(v[3]));
                    }
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int r = rg + 16 * i;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (r0 + r < a.n_nodes)
                        v = *reinterpret_cast<const float4 *>(
                            &a.V[(size_t)(r0 + r) * KP + 4 * cg]);
                    const int n = 4 * cg;
                    *reinterpret_cast<float4 *>(&U[r * LDU + n]) = make_float4(
                        siluf_(fmaf(ga[n], v.x, gb[n])),
                        siluf_(fmaf(ga[n + 1], v.y, gb[n + 1])),
                        siluf_(fmaf(ga[n + 2], v.z, gb[n + 2])),
                        siluf_(fmaf(ga[n + 3], v.w, gb[n + 3])));
                }
            }
        }
        if (a.phase == 1) continue;
        __syncthreads();
        float acc[4][1][4] = {};
        if (4 * cg < KP) tile_gemm<4, 1>(U, LDU, W2t, KP, acc);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int r = rg + 16 * i;
            float o[4];
            float dot = 0.0f;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int n = 4 * cg + c;
                o[c] = (4 * cg < KP) ? acc[i][0][c] + b2[n] : 0.0f;
                dot = fmaf(wn[n], o[c], dot);
            }
            float s = 1.0f;
            if (f_natt) {   // :154-157
                dot = rowgroup_sum(dot) + natt_b;
                s = (a.flags & PVS_F_SOFTMAX_ATTENTION) ? dot : apply_act(dot, a.att_act);
                if (cg == 0 && a.natt_out && r0 + r < a.n_nodes) a.natt_out[r0 + r] = s;
            }
            if (r0 + r >= a.n_nodes || 4 * cg >= KP) continue;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int n = 4 * cg + c;
                if (n >= k) continue;
                float out = o[c] * s;
                if (a.flags & PVS_F_RESIDUAL) {   // :158-165
                    const float hv = IN[r * LDIN + n];
                    if (a.flags & PVS_F_REZERO) out = hv + gate * out;
                    else if (a.flags & PVS_F_GATED_RESIDUAL) {
                        float g = fmaxf(gate, 0.0f);
                        out = g * out + (1.0f - g) * hv;
                    } else out = hv + out;
                }
                a.h_out[(size_t)(r0 + r) * k + n] = out;
            }
        }
    }
}

// ---------------------------------------------------------------------------
// GraphNorm statistics over ALL nodes of the batch (the reference calls
// GraphNorm without `batch`, egnn_satorras.py:84)
// ---------------------------------------------------------------------------
// partial[b][c] = sum over this block's rows of f(V[r][c]),
// f = v (sq == 0) or (v - shift[c])^2 (sq == 1)
__global__ void __launch_bounds__(256)
gn_colsum_kernel(const float *__restrict__ V, int n, int kp,
                 const float *__restrict__ shift, int sq,
                 float *__restrict__ partial) {
    __shared__ float part[4][64];
    const int cl = threadIdx.x & 63, grp = threadIdx.x >> 6;
    const int rows_per = (n + gridDim.x - 1) / gridDim.x;
    const int lo = blockIdx.x * rows_per, hi = min(n, lo + rows_per);
    float s = 0.0f;
    if (cl < kp) {
        const float sh = sq ? shift[cl] : 0.0f;
        for (int r = lo + grp; r < hi; r += 4) {
            float v = V[(size_t)r * kp + cl] - sh;
            s += sq ? v * v : v;
        }
    }
    part[grp][cl] = s;
    __syncthreads();
    if (grp == 0)
        partial[blockIdx.x * 64 + cl] =
            (part[0][cl] + part[1][cl]) + (part[2][cl] + part[3][cl]);
}

// stage 0: shift[c] = mean[c] * mean_scale[c]
// stage 1: a[c] = w[c] / sqrt(var[c] + eps), b[c] = bias[c] - a[c] * shift[c]
__global__ void gn_finalize_kernel(const float *__restrict__ partial, int nblocks,
                                   int n, int k, int stage,
                                   const float *__restrict__ gn_w,
                                   const float *__restrict__ gn_b,
                                   const float *__restrict__ gn_ms,
                                   float *__restrict__ shift,
                                   float *__restrict__ ga, float *__restrict__ gb,
                                   float *__restrict__ mean_out,
                                   float *__restrict__ invstd_out) {
    const int c = threadIdx.x;
    if (c >= 64) return;
    float s = 0.0f;
    for (int b = 0; b < nblocks; ++b) s += partial[b * 64 + c];
    const float mean = s / (float)(n > 0 ? n : 1);
    if (stage == 0) {
        shift[c] = c < k ? mean * gn_ms[c] : 0.0f;
        mean_out[c] = c < k ? mean : 0.0f;
    } else {
        const float inv = 1.0f / sqrtf(mean + 1e-5f);
        const float av = c < k ? gn_w[c] * inv : 0.0f;
        ga[c] = av;
        gb[c] = c < k ? gn_b[c] - av * shift[c] : 0.0f;
        invstd_out[c] = c < k ? inv : 0.0f;
    }
}

int persistent_grid(int work_items, int blocks_per_sm) {
    int g = num_sms() * blocks_per_sm;
    if (work_items < g) g = work_items;
    return g < 1 ? 1 : g;
}

int launch_linear(const float *in, int ld_in, int rows, int ki,
                  const float *w, int ld_w, const float *b, int ko,
                  int act, float *out, int ld_out, cudaStream_t st,
                  int w_in_major, int accumulate) {
    if (rows == 0) return PVS_OK;
    if (ki <= LSK_MAX_KI && ko <= 64 && !w_in_major && !accumulate && rows >= 4096) {
        launch_chained(linear_smallk_kernel, dim3((rows + 63) / 64), dim3(256), 0, st, in, ld_in,
                       rows, ki, w, ld_w, b, ko, act, out, ld_out);
        return check_launch();
    }
    const int kip = (ki + 3) & ~3;
    const int nj4 = ko <= 64 ? 1 : 2;
    const int ldw = 64 * nj4;
    size_t smem = ((size_t)kip * ldw + (size_t)NODE_ROWS * (kip + 4) + ldw) * sizeof(float);
    const int tiles = (rows + NODE_ROWS - 1) / NODE_ROWS;
    const int grid = persistent_grid(tiles, 2);
    int rc;
    if (nj4 == 1) {
        rc = ensure_smem(linear_fwd_kernel<1>, smem);
        if (rc) return rc;
        launch_chained(linear_fwd_kernel<1>, dim3(grid), dim3(FWD_THREADS), smem, st, in, ld_in,
                       rows, ki, w, ld_w, b, ko, act, out, ld_out, w_in_major, accumulate);
    } else {
        rc = ensure_smem(linear_fwd_kernel<2>, smem);
        if (rc) return rc;
        launch_chained(linear_fwd_kernel<2>, dim3(grid), dim3(FWD_THREADS), smem, st, in, ld_in,
                       rows, ki, w, ld_w, b, ko, act, out, ld_out, w_in_major, accumulate);
    }
    return check_launch();
}

template <int KP>
static int launch_edge(const EdgeArgs &a, int n_tiles_cap, cudaStream_t st) {
    size_t smem = sizeof(EdgeSmem<KP>);
    int rc = ensure_smem(egnn_edge_fwd_kernel<KP>, smem);
    if (rc) return rc;
    const int grid = persistent_grid(n_tiles_cap, 2);
    egnn_edge_fwd_kernel<KP><<<grid, FWD_THREADS, smem, st>>>(a);
    return check_launch();
}

template <int KP>
static int launch_node(const NodeArgs &a, cudaStream_t st) {
    size_t smem = ((size_t)3 * KP * 64 + (size_t)NODE_ROWS * (2 * KP + 4) +
                   (size_t)NODE_ROWS * (KP + 4) + 5 * 64) * sizeof(float);
    int rc = ensure_smem(egnn_node_fwd_kernel<KP>, smem);
    if (rc) return rc;
    const int tiles = (a.n_nodes + NODE_ROWS - 1) / NODE_ROWS;
    const int grid = persistent_grid(tiles, 2);
    egnn_node_fwd_kernel<KP><<<grid, FWD_THREADS, smem, st>>>(a);
    return check_launch();
}

constexpr int GN_BLOCKS = 128;

// Pitch of P, Q, M and V in pvs_egnn_layer_fwd's workspace: the tcgen05 tiles
// are 64 or 128 wide, the FFMA kernels 32 or 64.
static int layer_pitch(const pvs_layer_config *cfg) {
    return cfg->k > 64 ? 128 : (cfg->k <= 32 && cfg->math == PVS_MATH_FP32) ? 32 : 64;
}
// The backward kernels read P, Q, M and V at pitch 64: its recompute writes
// them at that pitch whatever the forward's, and it reads the forward's own
// workspace (fwd_saved) only where layer_pitch is 64 too.
constexpr int RECOMPUTE_PITCH = 64;

// The one layout of a layer's forward workspace, from `base` rounded up to 256 B.
static FwdWorkspace carve_workspace(const void *base, int n, int e, int kp, uint32_t flags) {
    FwdWorkspace w{};
    w.kp = kp;
    char *const start = (char *)align_up((int64_t)(uintptr_t)base, 256);
    char *p = start;
    auto take = [&](int64_t count) {
        float *r = (float *)p;
        p += align_up(count * (int64_t)sizeof(float), 256);
        return r;
    };
    w.P = take((int64_t)n * kp);
    w.Q = take((int64_t)n * kp);
    w.M = take((int64_t)n * kp);
    const int kv = kp > 64 ? kp : 64;   // channels of the per-channel vectors
    if (flags & PVS_F_GRAPHNORM) {
        w.V = take((int64_t)n * kp);
        w.gn_partial = take(GN_BLOCKS * 64);
        w.gn_shift = take(kv);
        w.gn_a = take(kv);
        w.gn_b = take(kv);
        w.gn_mean = take(kv);
        w.gn_invstd = take(kv);
    }
    if ((flags & PVS_F_EDGE_ATTENTION) && (flags & PVS_F_SOFTMAX_ATTENTION)) {
        w.m_ws = take((int64_t)e * kp);
        w.z_ws = take((int64_t)e);
    }
    {
        const int64_t tcap = pvs_packed_tiles_capacity(e);
        w.Mpart = take(tcap * 2 * kv);
        w.xpart = take(tcap * 2 * 4);
    }
    w.bytes = p - start;
    return w;
}

// Batch-wide GraphNorm statistics of V (two passes: mean, then the centred
// second moment) -> the per-channel affine gn_a * v + gn_b, mean and 1/std.
// The kernels take 64 channels at a time: at pitch 128 (k > 64) the four
// launches run once per 64-channel half, on offset pointers.
static int graphnorm_stats(const FwdWorkspace &w, const pvs_layer_params *p, int n, int k,
                           cudaStream_t st) {
    const int kp = w.kp;
    int launches = 0;
    for (int c0 = 0; c0 < kp; c0 += 64) {
        const int kc = k - c0;
        const float *gw = p->gn_weight + c0, *gb = p->gn_bias + c0, *gm = p->gn_mean_scale + c0;
        float *sh = w.gn_shift + c0, *ga = w.gn_a + c0, *gbo = w.gn_b + c0;
        float *mean = w.gn_mean + c0, *inv = w.gn_invstd + c0;
        gn_colsum_kernel<<<GN_BLOCKS, 256, 0, st>>>(w.V + c0, n, kp, nullptr, 0, w.gn_partial);
        gn_finalize_kernel<<<1, 64, 0, st>>>(w.gn_partial, GN_BLOCKS, n, kc, 0, gw, gb, gm, sh, ga,
                                             gbo, mean, inv);
        gn_colsum_kernel<<<GN_BLOCKS, 256, 0, st>>>(w.V + c0, n, kp, sh, 1, w.gn_partial);
        gn_finalize_kernel<<<1, 64, 0, st>>>(w.gn_partial, GN_BLOCKS, n, kc, 1, gw, gb, gm, sh, ga,
                                             gbo, mean, inv);
        launches += 4;
    }
    return check_launch(launches);
}

int64_t fwd_recompute_bytes(int n, int e, uint32_t flags) {
    return carve_workspace(nullptr, n, e, RECOMPUTE_PITCH, flags).bytes + 256;
}

FwdWorkspace fwd_saved(const void *saved_workspace, int n, int e, const pvs_layer_config *cfg) {
    return carve_workspace(saved_workspace, n, e, layer_pitch(cfg), cfg->flags);
}

// node_pre: P = h W1a^T + b1 ; Q = h W1b^T (perm-invariant: Q = h W1a^T)
static int node_pre_stage(const pvs_layer_config *cfg, const pvs_layer_params *p,
                          const float *h_in, int n, const FwdWorkspace &w, cudaStream_t st) {
    const int k = cfg->k, in_e = edge_in_width(cfg);
    const bool perm = cfg->flags & PVS_F_PERM_INVARIANT;
    if (cfg->math != PVS_MATH_FP32)
        return launch_node_pre_tc(h_in, p->edge_w1, p->edge_b1, w.P, w.Q, n, k, in_e,
                                  perm ? 1 : 0, cfg->math, st);
    int rc;
    if (k < w.kp) {
        rc = cuda_call(cudaMemsetAsync(w.P, 0, (size_t)((char *)w.M - (char *)w.P), st));
        if (rc) return rc;
    }
    rc = launch_linear(h_in, k, n, k, p->edge_w1, in_e, p->edge_b1, k, PVS_ACT_NONE, w.P, w.kp,
                       st);
    if (rc) return rc;
    return launch_linear(h_in, k, n, k, p->edge_w1 + (perm ? 0 : k), in_e, nullptr, k,
                         PVS_ACT_NONE, w.Q, w.kp, st);
}

// edge: messages, their sums M and the coordinate update; with softmax
// attention, the aggregation over each node's segment.  edge_events records
// cfg->ev_edge_begin / ev_edge_end around the stage.
static int edge_stage(const pvs_graph *g, const pvs_layer_config *cfg, const pvs_layer_params *p,
                      const float *x_in, const float *m_prev, float *x_out, float *m_out,
                      float *att_out, const FwdWorkspace &w, bool edge_events, cudaStream_t st) {
    const uint32_t f = cfg->flags;
    const int n = g->n_nodes;
    const bool softmax = (f & PVS_F_EDGE_ATTENTION) && (f & PVS_F_SOFTMAX_ATTENTION);
    EdgeArgs ea{};
    ea.row_ptr = g->row_ptr; ea.col = g->col; ea.tile_ptr = g->tile_ptr;
    ea.n_tiles = g->n_tiles; ea.attr = cfg->n_edge_classes > 0 ? g->attr : nullptr;
    ea.ptile_last = g->ptile_last; ea.n_ptiles = g->n_ptiles; ea.n_nodes = n;
    ea.Mpart = w.Mpart; ea.xpart = w.xpart;
    ea.P = w.P; ea.Q = w.Q; ea.x_in = x_in; ea.m_prev = m_prev; ea.M = w.M;
    ea.x_out = x_out;
    // the softmax pass needs every message and logit of a segment
    ea.m_out = m_out ? m_out : softmax ? w.m_ws : nullptr;
    ea.ld_m = m_out ? cfg->k : w.kp;
    ea.att_out = att_out ? att_out : softmax ? w.z_ws : nullptr;
    ea.edge_w1 = p->edge_w1; ea.edge_w2 = p->edge_w2; ea.edge_b2 = p->edge_b2;
    ea.coord_w1 = p->coord_w1 ? p->coord_w1 : p->edge_w2;
    ea.coord_b1 = p->coord_b1 ? p->coord_b1 : p->edge_b2;
    ea.coord_w2 = p->coord_w2 ? p->coord_w2 : p->edge_b2;
    ea.att_w = p->att_w; ea.att_b = p->att_b; ea.edge_gate = p->edge_gate;
    ea.k = cfg->k; ea.in_e = edge_in_width(cfg); ea.n_classes = cfg->n_edge_classes;
    ea.flags = f; ea.att_act = cfg->att_act;
    if (edge_events && cfg->ev_edge_begin) cudaEventRecord((cudaEvent_t)cfg->ev_edge_begin, st);
    int rc;
    if (cfg->math != PVS_MATH_FP32) rc = launch_edge_tc(ea, g->n_ptiles_cap, cfg->math, st);
    else rc = w.kp == 32 ? launch_edge<32>(ea, g->n_tiles_cap, st)
                         : launch_edge<64>(ea, g->n_tiles_cap, st);
    if (rc) return rc;
    if (softmax) {
        segment_softmax_agg_kernel<<<(n + 7) / 8, 256, 0, st>>>(
            g->row_ptr, n, ea.m_out, ea.ld_m, w.kp, ea.att_out, w.M);
        rc = check_launch();
        if (rc) return rc;
    }
    if (edge_events && cfg->ev_edge_end) cudaEventRecord((cudaEvent_t)cfg->ev_edge_end, st);
    return PVS_OK;
}

// FULL: the node model, h_out and natt_out.  GN_STATS: only GraphNorm's
// pre-activation V and its batch statistics (nothing without GraphNorm).
enum class NodeStage { FULL, GN_STATS };

// node: phase 0, or with GraphNorm phase 1 (Wn1 -> V), the batch statistics
// and phase 2 (resume from V)
static int node_stage(const pvs_layer_config *cfg, const pvs_layer_params *p, const float *h_in,
                      float *h_out, float *natt_out, int n, const FwdWorkspace &w,
                      NodeStage mode, cudaStream_t st) {
    const uint32_t f = cfg->flags;
    const int k = cfg->k;
    const bool graphnorm = f & PVS_F_GRAPHNORM;
    if (mode == NodeStage::GN_STATS && !graphnorm) return PVS_OK;
    NodeArgs na{};   // the FFMA kernel's
    na.h_in = h_in; na.M = w.M; na.h_out = h_out; na.V = w.V;
    na.natt_out = natt_out;
    na.node_w1 = p->node_w1; na.node_b1 = p->node_b1; na.node_w2 = p->node_w2;
    na.node_b2 = p->node_b2; na.natt_w = p->natt_w; na.natt_b = p->natt_b;
    na.node_gate = p->node_gate;
    na.n_nodes = n; na.k = k; na.flags = f; na.att_act = cfg->att_act;
    auto run = [&](int phase) {
        if (cfg->math != PVS_MATH_FP32) {
            const bool out = phase != 1;
            return launch_node_tc(h_in, w.M, out ? h_out : nullptr, out ? natt_out : nullptr, p,
                                  n, k, f, cfg->att_act, cfg->math, st, phase,
                                  phase ? w.V : nullptr, phase == 2 ? w.gn_a : nullptr,
                                  phase == 2 ? w.gn_b : nullptr);
        }
        na.phase = phase;
        if (phase == 2) { na.gn_a = w.gn_a; na.gn_b = w.gn_b; }
        return w.kp == 32 ? launch_node<32>(na, st) : launch_node<64>(na, st);
    };
    if (!graphnorm) return run(0);
    int rc = run(1);
    if (rc) return rc;
    rc = graphnorm_stats(w, p, n, k, st);
    if (rc || mode == NodeStage::GN_STATS) return rc;
    return run(2);
}

// One layer forward, over the stages set in `stages` (node_pre -> edge ->
// node), on the workspace w.  Each output may be null.
static int layer_forward(const pvs_graph *g, const pvs_layer_config *cfg,
                         const pvs_layer_params *p, const float *h_in, const float *x_in,
                         const float *m_prev, float *h_out, float *x_out, float *m_out,
                         float *att_out, float *natt_out, const FwdWorkspace &w, int stages,
                         bool edge_events, NodeStage node, cudaStream_t st) {
    int rc;
    if (stages & PVS_STAGE_NODE_PRE) {
        rc = node_pre_stage(cfg, p, h_in, g->n_nodes, w, st);
        if (rc) return rc;
    }
    if (stages & PVS_STAGE_EDGE) {
        rc = edge_stage(g, cfg, p, x_in, m_prev, x_out, m_out, att_out, w, edge_events, st);
        if (rc) return rc;
    }
    if (!(stages & PVS_STAGE_NODE)) return PVS_OK;
    return node_stage(cfg, p, h_in, h_out, natt_out, g->n_nodes, w, node, st);
}

// Forward recompute for the backward pass: P, Q, M (and the softmax attention
// values + messages, and the GraphNorm pre-activation V with its batch
// statistics).  No h_out / x_out is produced; cfg->stages and the edge events
// do not apply.
int fwd_recompute(const pvs_graph *g, const pvs_layer_config *cfg, const pvs_layer_params *p,
                  const float *h_in, const float *x_in, const float *m_prev, void *ws_base,
                  FwdWorkspace *out, cudaStream_t st) {
    const FwdWorkspace w =
        carve_workspace(ws_base, g->n_nodes, g->n_edges, RECOMPUTE_PITCH, cfg->flags);
    const int rc = layer_forward(g, cfg, p, h_in, x_in, m_prev, nullptr, nullptr, nullptr,
                                 nullptr, nullptr, w, PVS_STAGE_ALL, false, NodeStage::GN_STATS,
                                 st);
    if (rc) return rc;
    *out = w;
    return PVS_OK;
}

}  // namespace pvs

using namespace pvs;

extern "C" {

int pvs_linear_fwd(const float *in, int32_t ld_in, int32_t rows, int32_t ki,
                   const float *w, int32_t ld_w, const float *b, int32_t ko,
                   int32_t act, float *out, int32_t ld_out, void *stream) {
    if (rows < 0 || ki < 1 || ki > 128 || ko < 1 || ko > 128) return PVS_ERR_INVALID_ARG;
    if (rows > 0 && (!in || !w || !out)) return PVS_ERR_INVALID_ARG;
    if (ld_in < ki || ld_w < ki || ld_out < ko) return PVS_ERR_INVALID_ARG;
    return launch_linear(in, ld_in, rows, ki, w, ld_w, b, ko, act, out, ld_out,
                         (cudaStream_t)stream);
}

int pvs_mean_pool_fwd(const float *h, const int32_t *graph_ptr, int32_t n_graphs,
                      int32_t k, float *pooled, void *stream) {
    if (n_graphs < 0 || k < 1) return PVS_ERR_INVALID_ARG;
    if (n_graphs == 0) return PVS_OK;
    if (!h || !graph_ptr || !pooled) return PVS_ERR_INVALID_ARG;
    mean_pool_kernel<<<n_graphs, 256, 0, (cudaStream_t)stream>>>(h, graph_ptr, k, pooled);
    return check_launch();
}

int64_t pvs_egnn_layer_workspace_bytes(int32_t n_nodes, int32_t n_edges,
                                       const pvs_layer_config *cfg) {
    if (!cfg || cfg->k < 1 || cfg->k > PVS_MAX_K_TC_FWD) return -1;
    if (cfg->math < PVS_MATH_FP32 || cfg->math > PVS_MATH_FP16X2) return -1;
    if (cfg->k > PVS_MAX_K && cfg->math == PVS_MATH_FP32) return -1;
    return carve_workspace(nullptr, n_nodes, n_edges, layer_pitch(cfg), cfg->flags).bytes + 256;
}

int pvs_egnn_layer_fwd(const pvs_graph *g, const pvs_layer_config *cfg,
                       const pvs_layer_params *p, const float *h_in,
                       const float *x_in, const float *m_prev, float *h_out,
                       float *x_out, float *m_out, float *att_out,
                       float *natt_out, void *workspace, int64_t workspace_bytes,
                       void *stream) {
    if (!g || !cfg || !p) return PVS_ERR_INVALID_ARG;
    // 65..128: forward only, on the tensor cores (the FFMA kernels are 64 wide)
    if (cfg->k < 1 || cfg->k > PVS_MAX_K_TC_FWD) return PVS_ERR_UNSUPPORTED_K;
    if (cfg->k > PVS_MAX_K && cfg->math == PVS_MATH_FP32) return PVS_ERR_UNSUPPORTED_K;
    if (cfg->math < PVS_MATH_FP32 || cfg->math > PVS_MATH_FP16X2) return PVS_ERR_INVALID_ARG;
    if (cfg->n_edge_classes < 0 || cfg->n_edge_classes > PVS_MAX_EDGE_CLASSES)
        return PVS_ERR_INVALID_ARG;
    if (g->n_nodes < 0 || g->n_edges < 0) return PVS_ERR_INVALID_ARG;
    if (g->n_nodes == 0) return PVS_OK;
    if (cfg->math != PVS_MATH_FP32 && (!g->ptile_last || !g->n_ptiles))
        return PVS_ERR_INVALID_ARG;   // tcgen05 edge kernel: pvs_build_packed_tiles
    if (cfg->math == PVS_MATH_FP32 && (!g->tile_ptr || !g->n_tiles))
        return PVS_ERR_INVALID_ARG;   // FFMA edge kernel: pvs_build_tiles
    if (!g->row_ptr || (g->n_edges > 0 && !g->col))
        return PVS_ERR_INVALID_ARG;
    if (cfg->n_edge_classes > 0 && g->n_edges > 0 && !g->attr) return PVS_ERR_INVALID_ARG;
    if (!h_in || !x_in || !h_out || !workspace) return PVS_ERR_INVALID_ARG;
    if (x_out == x_in) return PVS_ERR_INVALID_ARG;
    if (!p->edge_w1 || !p->edge_b1 || !p->edge_w2 || !p->edge_b2 || !p->node_w1 ||
        !p->node_b1 || !p->node_w2 || !p->node_b2)
        return PVS_ERR_INVALID_ARG;
    const uint32_t f = cfg->flags;
    if ((f & PVS_F_UPDATE_COORDS) && (!p->coord_w1 || !p->coord_b1 || !p->coord_w2 || !x_out))
        return PVS_ERR_INVALID_ARG;
    if ((f & PVS_F_EDGE_ATTENTION) && (!p->att_w || !p->att_b)) return PVS_ERR_INVALID_ARG;
    if ((f & PVS_F_NODE_ATTENTION) && (!p->natt_w || !p->natt_b)) return PVS_ERR_INVALID_ARG;
    if ((f & PVS_F_GRAPHNORM) && (!p->gn_weight || !p->gn_bias || !p->gn_mean_scale))
        return PVS_ERR_INVALID_ARG;
    if ((f & PVS_F_REZERO) && (f & PVS_F_GATED_RESIDUAL)) return PVS_ERR_INVALID_ARG;
    if ((f & (PVS_F_REZERO | PVS_F_GATED_RESIDUAL)) && (f & PVS_F_RESIDUAL) && !p->node_gate)
        return PVS_ERR_INVALID_ARG;
    if (workspace_bytes < pvs_egnn_layer_workspace_bytes(g->n_nodes, g->n_edges, cfg))
        return PVS_ERR_WORKSPACE;

    const int stages = (cfg->stages & PVS_STAGE_ALL) ? (cfg->stages & PVS_STAGE_ALL)
                                                     : PVS_STAGE_ALL;
    const FwdWorkspace w =
        carve_workspace(workspace, g->n_nodes, g->n_edges, layer_pitch(cfg), f);
    return layer_forward(g, cfg, p, h_in, x_in, m_prev, h_out, x_out, m_out, att_out, natt_out,
                         w, stages, true, NodeStage::FULL, (cudaStream_t)stream);
}

}  // extern "C"
