// K1 and friends: radius-graph construction (per-complex cell list -> dst-sorted
// CSR), work-tile partition, caller-order edge_index -> CSR, CSC transpose,
// prune mask.  All integer / fp64-compare work: bit-exact by construction.
//
// Replaces /root/reference/point_vs/preprocessing/preprocessing.py:68-155
// (generate_edges) and the PyG collate offsets (data_loaders.py:517-520).
#include "graph_common.cuh"

namespace pvs {

// ---------------------------------------------------------------------------
// exclusive scan of int32 (three small launches; n is a node count)
// ---------------------------------------------------------------------------
constexpr int SCAN_THREADS = 1024;
constexpr int SCAN_ITEMS = 4;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__global__ void __launch_bounds__(SCAN_THREADS)
scan_local_kernel(const int32_t *__restrict__ in, int n,
                  int32_t *__restrict__ out, int32_t *__restrict__ block_sums) {
    __shared__ int warp_buf[33];
    const int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    int v[SCAN_ITEMS];
    int s = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        v[i] = (base + i < n) ? in[base + i] : 0;
        s += v[i];
    }
    int total;
    int prefix = block_scan_excl(s, &total, warp_buf);
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        if (base + i < n) out[base + i] = prefix;
        prefix += v[i];
    }
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SCAN_THREADS)
scan_sums_kernel(int32_t *__restrict__ block_sums, int nb,
                 int32_t *__restrict__ total_out) {
    __shared__ int warp_buf[33];
    int carry = 0;
    for (int b0 = 0; b0 < nb; b0 += SCAN_THREADS) {
        int i = b0 + threadIdx.x;
        int v = i < nb ? block_sums[i] : 0;
        int total;
        int prefix = block_scan_excl(v, &total, warp_buf);
        if (i < nb) block_sums[i] = carry + prefix;
        carry += total;
    }
    if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(SCAN_THREADS)
scan_add_kernel(int32_t *__restrict__ out, int n,
                const int32_t *__restrict__ block_sums) {
    const int base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_ITEMS;
    const int add = block_sums[blockIdx.x];
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i)
        if (base + i < n) out[base + i] += add;
}

int exclusive_scan(const int32_t *deg, int n, int32_t *row_ptr, void *scratch,
                   cudaStream_t st) {
    if (n == 0) {
        return cuda_call(cudaMemsetAsync(row_ptr, 0, sizeof(int32_t), st));
    }
    int nb = (n + SCAN_TILE - 1) / SCAN_TILE;
    int32_t *sums = (int32_t *)scratch;
    scan_local_kernel<<<nb, SCAN_THREADS, 0, st>>>(deg, n, row_ptr, sums);
    scan_sums_kernel<<<1, SCAN_THREADS, 0, st>>>(sums, nb, row_ptr + n);
    if (nb > 1) scan_add_kernel<<<nb, SCAN_THREADS, 0, st>>>(row_ptr, n, sums);
    return check_launch(nb > 1 ? 3 : 2);
}

// ---------------------------------------------------------------------------
// K1: radius graph.  One CTA per complex.
// ---------------------------------------------------------------------------
constexpr int RG_THREADS = 512;
constexpr int RG_WARPS = RG_THREADS / 32;
constexpr int RG_SPLIT = 4;        // CTAs per complex (each bins all atoms,
                                   // handles a quarter of the destinations;
                                   // 2 and 3 measured slower: 0.217 / 0.242 ms
                                   // vs 0.210 per 128 complexes)
constexpr int RG_MAX_DIM = 16;
constexpr int RG_MAX_CELLS = RG_MAX_DIM * RG_MAX_DIM * RG_MAX_DIM;

struct RgSmem {
    int cell_start[RG_MAX_CELLS + 1];
    int cell_fill[RG_MAX_CELLS];
    double red[6][RG_WARPS];
    double box[6];
    int warp_buf[33];
    int misc[4];
};

static size_t rg_smem_bytes(int max_n, bool with_prefix, bool stage) {
    size_t words = (size_t)(max_n + 31) / 32;
    size_t b = sizeof(RgSmem);
    b += (size_t)max_n * sizeof(int);                 // sorted_idx
    b += (size_t)RG_WARPS * 4 * words * sizeof(int);  // bit masks: 2 lists x 2 half-warps
    b += (size_t)max_n * sizeof(int);                 // prefix_inter (fill + ref_pos)
    (void)with_prefix;
    b = (b + 7) & ~(size_t)7;
    if (stage) b += (size_t)max_n * (3 * sizeof(double) + sizeof(int));  // cell-sorted copy
    return b;
}

template <bool FILL>
__global__ void __launch_bounds__(RG_THREADS)
radius_graph_kernel(const double *__restrict__ coords,
                    const int32_t *__restrict__ bp,
                    const int32_t *__restrict__ complex_ptr, double r_inter,
                    double r_intra, int32_t *__restrict__ deg,
                    int32_t *__restrict__ n_inter_out,
                    const int32_t *__restrict__ n_inter_in,
                    const int32_t *__restrict__ row_ptr,
                    int32_t *__restrict__ col, uint8_t *__restrict__ attr,
                    int32_t *__restrict__ ref_pos, int max_n, int stage,
                    uint32_t *__restrict__ mask_out, int edge_capacity,
                    int32_t *__restrict__ overflow, int split = RG_SPLIT) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    RgSmem &S = *reinterpret_cast<RgSmem *>(smem_raw);
    // `split` CTAs per complex: RG_SPLIT for the warp-per-atom passes, fewer for
    // the thread-per-atom count pass (one thread per atom: 512 atoms a CTA)
    const int cplx = blockIdx.x / split, part = blockIdx.x % split;
    const int n0 = complex_ptr[cplx];
    const int n = complex_ptr[cplx + 1] - n0;
    if (n <= 0 || n > max_n) return;   // host sizes smem from max_n
    const int words = (max_n + 31) / 32;
    int *sorted_idx = reinterpret_cast<int *>(smem_raw + sizeof(RgSmem));
    unsigned *masks = reinterpret_cast<unsigned *>(sorted_idx + max_n);
    int *prefix_inter = reinterpret_cast<int *>(masks + (size_t)RG_WARPS * 4 * words);
    // cell-sorted copy of the coordinates / bp: the neighbour loop then reads
    // contiguous shared-memory ranges instead of chasing sorted_idx into global
    double *scoord = reinterpret_cast<double *>(
        (reinterpret_cast<uintptr_t>(prefix_inter + max_n) + 7) & ~(uintptr_t)7);
    int *sbp = reinterpret_cast<int *>(scoord + 3 * (size_t)max_n);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double *cx = coords + 3 * (size_t)n0;
    const int32_t *cbp = bp + n0;

    // ---- bounding box ----
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (int i = tid; i < n; i += RG_THREADS) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            double v = cx[3 * i + a];
            lo[a] = fmin(lo[a], v);
            hi[a] = fmax(hi[a], v);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fmin(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmax(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
        if (lane == 0) {
            S.red[a][warp] = lo[a];
            S.red[3 + a][warp] = hi[a];
        }
    }
    __syncthreads();
    if (tid < 3) {
        double l = S.red[tid][0], h = S.red[3 + tid][0];
        for (int w = 1; w < RG_WARPS; ++w) {
            l = fmin(l, S.red[tid][w]);
            h = fmax(h, S.red[3 + tid][w]);
        }
        S.box[tid] = l;
        S.box[3 + tid] = h;
    }
    __syncthreads();
    // cell edge >= r_max * (1 + 1e-6): two atoms closer than r_max are at most
    // one cell apart on every axis even after rounding of the cell coordinate.
    const double r_max = fmax(r_inter, r_intra);
    const double cs0 = fmax(r_max * (1.0 + 1e-6), 1e-9);
    int dim[3];
    double cs[3], blo[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        blo[a] = S.box[a];
        double ext = S.box[3 + a] - S.box[a];
        double q = ext / cs0;
        if (q + 1.0 > (double)RG_MAX_DIM) {
            dim[a] = RG_MAX_DIM;
            cs[a] = 1.0 / (ext / RG_MAX_DIM * (1.0 + 1e-6));
        } else {
            dim[a] = (int)q + 1;
            cs[a] = 1.0 / cs0;
        }
    }
    const int ncell = dim[0] * dim[1] * dim[2];

    // ---- counting sort of atoms by cell (x fastest) ----
    for (int c = tid; c < ncell; c += RG_THREADS) {
        S.cell_start[c] = 0;
        S.cell_fill[c] = 0;
    }
    __syncthreads();
    for (int i = tid; i < n; i += RG_THREADS) {
        int c = cell_coord(cx[3 * i], blo[0], cs[0], dim[0]) +
                dim[0] * (cell_coord(cx[3 * i + 1], blo[1], cs[1], dim[1]) +
                          dim[1] * cell_coord(cx[3 * i + 2], blo[2], cs[2], dim[2]));
        atomicAdd(&S.cell_start[c], 1);
    }
    __syncthreads();
    int total = smem_scan_excl(S.cell_start, ncell, S.warp_buf);
    if (tid == 0) S.cell_start[ncell] = total;
    __syncthreads();
    for (int i = tid; i < n; i += RG_THREADS) {
        int c = cell_coord(cx[3 * i], blo[0], cs[0], dim[0]) +
                dim[0] * (cell_coord(cx[3 * i + 1], blo[1], cs[1], dim[1]) +
                          dim[1] * cell_coord(cx[3 * i + 2], blo[2], cs[2], dim[2]));
        int p = S.cell_start[c] + atomicAdd(&S.cell_fill[c], 1);
        sorted_idx[p] = i;
        if (stage) {
            scoord[3 * p] = cx[3 * i];
            scoord[3 * p + 1] = cx[3 * i + 1];
            scoord[3 * p + 2] = cx[3 * i + 2];
            sbp[p] = cbp[i];
        }
    }
    int e_base_c = 0, total_inter_c = 0;
    if (FILL && ref_pos != nullptr) {
        for (int i = tid; i < n; i += RG_THREADS) prefix_inter[i] = n_inter_in[n0 + i];
        __syncthreads();
        total_inter_c = smem_scan_excl(prefix_inter, n, S.warp_buf);
        e_base_c = row_ptr[n0];
    }
    __syncthreads();

    // ---- one warp per destination node ----
    const PairBand band = pair_band(r_inter, r_intra);
    const int nw = (n + 31) / 32;
    // neighbour search of destination atom i by W lanes (lane index l):
    // sets the bits of its inter / intra neighbours in m_inter / m_intra
    auto search = [&](const int i, const int l, const int W, unsigned *m_inter,
                      unsigned *m_intra) {
        const double xi = cx[3 * i], yi = cx[3 * i + 1], zi = cx[3 * i + 2];
        const int bi = cbp[i];
        const int ci0 = cell_coord(xi, blo[0], cs[0], dim[0]);
        const int ci1 = cell_coord(yi, blo[1], cs[1], dim[1]);
        const int ci2 = cell_coord(zi, blo[2], cs[2], dim[2]);
        const int x_lo = max(ci0 - 1, 0), x_hi = min(ci0 + 1, dim[0] - 1);
        for (int dz = -1; dz <= 1; ++dz) {
            int c2 = ci2 + dz;
            if (c2 < 0 || c2 >= dim[2]) continue;
            for (int dy = -1; dy <= 1; ++dy) {
                int c1 = ci1 + dy;
                if (c1 < 0 || c1 >= dim[1]) continue;
                int cb = dim[0] * (c1 + dim[1] * c2);
                int p_end = S.cell_start[cb + x_hi + 1];
                for (int p = S.cell_start[cb + x_lo] + l; p < p_end; p += W) {
                    const int j = sorted_idx[p];
                    double xj, yj, zj;
                    int bj;
                    if (stage) {
                        xj = scoord[3 * p]; yj = scoord[3 * p + 1]; zj = scoord[3 * p + 2];
                        bj = sbp[p];
                    } else {
                        xj = cx[3 * j]; yj = cx[3 * j + 1]; zj = cx[3 * j + 2];
                        bj = cbp[j];
                    }
                    // scipy cdist (preprocessing.py:108), graph_common.cuh
                    bool pos, in_inter, in_intra;
                    pair_test(band, xi, yi, zi, xj, yj, zj, pos, in_inter, in_intra);
                    unsigned bit = 1u << (j & 31);
                    if (pos && in_inter && bj != bi)
                        atomicOr(&m_inter[j >> 5], bit);   // :110-117
                    if (pos && in_intra)
                        atomicOr(&m_intra[j >> 5], bit);   // :119-121
                }
            }
        }
    };
    if (!FILL && mask_out != nullptr) {
        // Round 2 count pass: ONE THREAD per destination atom, atoms taken in
        // cell-sorted order (the 32 atoms of a warp sit in the same or adjacent
        // cells, so they walk nearly the same candidate runs and the shared-
        // memory reads broadcast).  The half-warp version below issued ~4x the
        // warp instructions for the same pair tests (16 lanes share ~12
        // candidates of a run, nine runs per atom, plus mask bookkeeping in
        // shared memory): 186 us per 128 x 1000 atoms, issue-bound.  Each
        // thread sets bits in its atom's PRIVATE mask row in global memory (no
        // atomics; the row lives in L1 while it is written), which the fill
        // pass then only expands -- sorted output without a sort, as before.
        // The CTAs of a complex each run their own counting sort, and the order
        // of the atoms INSIDE a cell depends on the order of their atomics; the
        // cell boundaries do not.  So the sorted positions are split between
        // the CTAs at cell boundaries: part k takes the cells that start in
        // [k n / split, (k + 1) n / split).
        auto part_begin = [&](int k) {
            if (k <= 0) return 0;
            if (k >= split) return n;
            const int target = (int)(((long long)n * k) / split);
            int lo = 0, hi = ncell;          // first cell with cell_start >= target
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (S.cell_start[mid] < target) lo = mid + 1; else hi = mid;
            }
            return S.cell_start[lo];
        };
        const int p_begin = part_begin(part), p_end = part_begin(part + 1);
        for (int p = p_begin + tid; p < p_end; p += RG_THREADS) {
            const int i = sorted_idx[p];
            uint32_t *m_inter = mask_out + (size_t)(n0 + i) * 2 * words;
            uint32_t *m_intra = m_inter + words;   // rows zeroed by the caller
            const double xi = cx[3 * i], yi = cx[3 * i + 1], zi = cx[3 * i + 2];
            const int bi = cbp[i];
            const int ci0 = cell_coord(xi, blo[0], cs[0], dim[0]);
            const int ci1 = cell_coord(yi, blo[1], cs[1], dim[1]);
            const int ci2 = cell_coord(zi, blo[2], cs[2], dim[2]);
            const int x_lo = max(ci0 - 1, 0), x_hi = min(ci0 + 1, dim[0] - 1);
            int n_i = 0, n_a = 0;
            for (int dz = -1; dz <= 1; ++dz) {
                const int c2 = ci2 + dz;
                if (c2 < 0 || c2 >= dim[2]) continue;
                for (int dy = -1; dy <= 1; ++dy) {
                    const int c1 = ci1 + dy;
                    if (c1 < 0 || c1 >= dim[1]) continue;
                    const int cb = dim[0] * (c1 + dim[1] * c2);
                    const int q_end = S.cell_start[cb + x_hi + 1];
                    for (int q = S.cell_start[cb + x_lo]; q < q_end; ++q) {
                        const int j = sorted_idx[q];
                        double xj, yj, zj;
                        int bj;
                        if (stage) {
                            xj = scoord[3 * q]; yj = scoord[3 * q + 1]; zj = scoord[3 * q + 2];
                            bj = sbp[q];
                        } else {
                            xj = cx[3 * j]; yj = cx[3 * j + 1]; zj = cx[3 * j + 2];
                            bj = cbp[j];
                        }
                        // the same test as `search` above
                        bool pos, in_inter, in_intra;
                        pair_test(band, xi, yi, zi, xj, yj, zj, pos, in_inter, in_intra);
                        const unsigned bit = 1u << (j & 31);
                        if (pos && in_inter && bj != bi) {       // :110-117
                            m_inter[j >> 5] |= bit;
                            ++n_i;
                        }
                        if (pos && in_intra) {                   // :119-121
                            m_intra[j >> 5] |= bit;
                            ++n_a;
                        }
                    }
                }
            }
            deg[n0 + i] = n_i + n_a;
            n_inter_out[n0 + i] = n_i;
        }
        return;
    }
    if (!FILL) {
        // count pass without kept masks: a HALF-warp per destination atom (a
        // run of three cells holds ~10 candidates, so 16 lanes are two-thirds
        // busy where 32 were one-third), two atoms per warp
        const int half = lane >> 4, hl = lane & 15;
        unsigned *m_inter = masks + (size_t)(warp * 2 + half) * 2 * words;
        unsigned *m_intra = m_inter + words;
        for (int i0 = 2 * warp + 2 * RG_WARPS * part; i0 < n; i0 += 2 * RG_WARPS * RG_SPLIT) {
            const int i = i0 + half;
            const bool active = i < n;
            for (int w = hl; w < nw; w += 16) {
                m_inter[w] = 0u;
                m_intra[w] = 0u;
            }
            __syncwarp();
            if (active) search(i, hl, 16, m_inter, m_intra);
            __syncwarp();
            int ci = 0, ca = 0;
            for (int w = hl; w < nw; w += 16) {
                ci += __popc(m_inter[w]);
                ca += __popc(m_intra[w]);
            }
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) {     // within the half-warp
                ci += __shfl_xor_sync(0xffffffffu, ci, o);
                ca += __shfl_xor_sync(0xffffffffu, ca, o);
            }
            if (active) {
                if (hl == 0) {
                    deg[n0 + i] = ci + ca;
                    n_inter_out[n0 + i] = ci;
                }
                if (mask_out != nullptr) {   // keep the masks: fill only expands them
                    uint32_t *mo = mask_out + (size_t)(n0 + i) * 2 * words;
                    for (int w = hl; w < nw; w += 16) {
                        mo[w] = m_inter[w];
                        mo[words + w] = m_intra[w];
                    }
                }
            }
            __syncwarp();
        }
        return;
    }
    unsigned *m_inter = masks + (size_t)warp * 2 * words;
    unsigned *m_intra = m_inter + words;
    for (int i = warp + RG_WARPS * part; i < n; i += RG_WARPS * RG_SPLIT) {
        for (int w = lane; w < nw; w += 32) {
            m_inter[w] = 0u;
            m_intra[w] = 0u;
        }
        __syncwarp();
        search(i, lane, 32, m_inter, m_intra);
        const int bi = cbp[i];
        __syncwarp();
        if (!FILL) {
            int ci = 0, ca = 0;
            for (int w = lane; w < nw; w += 32) {
                ci += __popc(m_inter[w]);
                ca += __popc(m_intra[w]);
            }
            ci = warp_sum_int(ci);
            ca = warp_sum_int(ca);
            if (lane == 0) {
                deg[n0 + i] = ci + ca;
                n_inter_out[n0 + i] = ci;
            }
            if (mask_out != nullptr) {   // keep the masks: fill only expands them
                uint32_t *mo = mask_out + (size_t)(n0 + i) * 2 * words;
                for (int w = lane; w < nw; w += 32) {
                    mo[w] = m_inter[w];
                    mo[words + w] = m_intra[w];
                }
            }
        } else {
            const int e_row = row_ptr[n0 + i];
            int run = e_row;
            int pi = 0;
            if (ref_pos != nullptr) pi = prefix_inter[i];
#pragma unroll 1
            for (int pass = 0; pass < 2; ++pass) {
                const unsigned *mk = pass == 0 ? m_inter : m_intra;
                const int pass_base = run;
                for (int w0 = 0; w0 < nw; w0 += 32) {
                    int w = w0 + lane;
                    unsigned bits = w < nw ? mk[w] : 0u;
                    int cnt = __popc(bits);
                    int incl = warp_scan_incl(cnt, lane);
                    int off = run + incl - cnt;
                    while (bits) {
                        int b = __ffs(bits) - 1;
                        bits &= bits - 1;
                        int j = w * 32 + b;
                        int bj = cbp[j];
                        if (off >= edge_capacity) {
                            if (overflow) *overflow = 1;
                            ++off;
                            continue;
                        }
                        col[off] = n0 + j;
                        uint8_t a;
                        if (pass == 0)   // :129-133
                            a = ((bi == 0 && bj == 1) || (bi == 1 && bj == 0)) ? 1 : 0;
                        else             // :135
                            a = (bi == 1 && bj == 1) ? 2 : 0;
                        attr[off] = a;
                        if (ref_pos != nullptr) {
                            int q = off - pass_base;
                            int local_row = e_row - e_base_c;   // edges before node i
                            ref_pos[off] = pass == 0
                                ? e_base_c + pi + q
                                : e_base_c + total_inter_c + (local_row - pi) + q;
                        }
                        ++off;
                    }
                    run += __shfl_sync(0xffffffffu, incl, 31);
                }
            }
        }
        __syncwarp();
    }
}

// fill from the masks stored by the count pass: EIGHT LANES per node (four
// nodes per warp), flat grid.  A lane owns 32 bytes of each 256-byte mask row
// (so a row is one coalesced 256-byte read), counts its bits, takes its offset
// from a 3-step scan inside the 8-lane group and writes its entries.  (One
// warp per node spent 55 us per 128 x 1000 atoms scanning empty words; one
// thread per node 40 us on uncoalesced row reads.)
__global__ void __launch_bounds__(256)
radius_graph_emit1_kernel(const uint32_t *__restrict__ masks, int words,
                          const int32_t *__restrict__ bp,
                          const int32_t *__restrict__ complex_ptr, int n_complexes,
                          int n_nodes, const int32_t *__restrict__ row_ptr,
                          int32_t *__restrict__ col, uint8_t *__restrict__ attr,
                          int edge_capacity, int32_t *__restrict__ overflow) {
    const int lane = threadIdx.x & 31, sub = lane & 7;
    const unsigned gmask = 0xffu << (lane & 24);          // this node's 8 lanes
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;
    if (i >= n_nodes) return;      // whole 8-lane groups leave together
    int lo = 0, hi = n_complexes;     // complex of node i
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (complex_ptr[mid] <= i) lo = mid; else hi = mid;
    }
    const int n0 = complex_ptr[lo];
    const int nw = (complex_ptr[lo + 1] - n0 + 31) / 32;
    const int bi = bp[i];
    int run = row_ptr[i];
    const uint32_t *mk0 = masks + (size_t)i * 2 * words;
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
        const uint32_t *mk = mk0 + pass * words;
        for (int w0 = 0; w0 < nw; w0 += 64) {             // 8 lanes x 8 words
            uint32_t b8[8];
            int cnt = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int w = w0 + 8 * sub + q;
                b8[q] = w < nw ? mk[w] : 0u;
                cnt += __popc(b8[q]);
            }
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
                const int up = __shfl_up_sync(gmask, incl, o, 8);
                if (sub >= o) incl += up;
            }
            int off = run + incl - cnt;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                unsigned bits = b8[q];
                while (bits) {
                    const int b = __ffs(bits) - 1;
                    bits &= bits - 1;
                    const int j = n0 + (w0 + 8 * sub + q) * 32 + b;
                    if (off < edge_capacity) {
                        const int bj = bp[j];
                        col[off] = j;
                        attr[off] = pass == 0
                            ? (((bi == 0 && bj == 1) || (bi == 1 && bj == 0)) ? 1 : 0)
                            : ((bi == 1 && bj == 1) ? 2 : 0);
                    } else if (overflow) {
                        *overflow = 1;
                    }
                    ++off;
                }
            }
            run += __shfl_sync(gmask, incl, 7, 8);
        }
    }
}

// the same with one warp per node (kept for reference / A-B timing)
__global__ void __launch_bounds__(256)
radius_graph_emit_kernel(const uint32_t *__restrict__ masks, int words,
                         const int32_t *__restrict__ bp,
                         const int32_t *__restrict__ complex_ptr, int n_complexes,
                         int n_nodes, const int32_t *__restrict__ row_ptr,
                         int32_t *__restrict__ col, uint8_t *__restrict__ attr,
                         int edge_capacity, int32_t *__restrict__ overflow) {
    const int lane = threadIdx.x & 31;
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (i >= n_nodes) return;
    int lo = 0, hi = n_complexes;     // complex of node i
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (complex_ptr[mid] <= i) lo = mid; else hi = mid;
    }
    const int n0 = complex_ptr[lo];
    const int nw = (complex_ptr[lo + 1] - n0 + 31) / 32;
    const int bi = bp[i];
    int run = row_ptr[i];
    const uint32_t *mk0 = masks + (size_t)i * 2 * words;
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
        const uint32_t *mk = mk0 + pass * words;
        for (int w0 = 0; w0 < nw; w0 += 32) {
            const int w = w0 + lane;
            unsigned bits = w < nw ? mk[w] : 0u;
            const int cnt = __popc(bits);
            const int incl = warp_scan_incl(cnt, lane);
            int off = run + incl - cnt;
            while (bits) {
                const int b = __ffs(bits) - 1;
                bits &= bits - 1;
                const int j = n0 + w * 32 + b;
                if (off < edge_capacity) {
                    const int bj = bp[j];
                    col[off] = j;
                    attr[off] = pass == 0
                        ? (((bi == 0 && bj == 1) || (bi == 1 && bj == 0)) ? 1 : 0)
                        : ((bi == 1 && bj == 1) ? 2 : 0);
                } else if (overflow) {
                    *overflow = 1;
                }
                ++off;
            }
            run += __shfl_sync(0xffffffffu, incl, 31);
        }
    }
}

// ---------------------------------------------------------------------------
// prune mask: component reachable from the first inter edge's row
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
prune_mask_kernel(const int32_t *__restrict__ row_ptr,
                  const int32_t *__restrict__ col,
                  const int32_t *__restrict__ n_inter,
                  const int32_t *__restrict__ complex_ptr,
                  uint8_t *__restrict__ keep) {
    __shared__ int start;
    const int n0 = complex_ptr[blockIdx.x];
    const int n = complex_ptr[blockIdx.x + 1] - n0;
    if (n <= 0) return;
    if (threadIdx.x == 0) start = 0x7fffffff;
    __syncthreads();
    int first = 0x7fffffff;
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        if (n_inter[n0 + i] > 0) { first = i; break; }
    if (first != 0x7fffffff) atomicMin(&start, first);
    __syncthreads();
    const int s = start;
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        keep[n0 + i] = (s == 0x7fffffff || i == s) ? 1 : 0;
    if (s == 0x7fffffff) return;   // no inter edge: reference keeps everything
    __syncthreads();
    for (;;) {
        int changed = 0;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            if (keep[n0 + i]) continue;
            for (int e = row_ptr[n0 + i]; e < row_ptr[n0 + i + 1]; ++e) {
                if (keep[col[e]]) {
                    keep[n0 + i] = 1;
                    changed = 1;
                    break;
                }
            }
        }
        if (!__syncthreads_or(changed)) break;
    }
}

// ---------------------------------------------------------------------------
// work tiles
// ---------------------------------------------------------------------------
constexpr int TILE_CHUNK = 256;   // nodes walked serially by one thread

__global__ void __launch_bounds__(256)
tiles_walk_kernel(const int32_t *__restrict__ row_ptr, int n_nodes,
                  int32_t *__restrict__ tmp, int32_t *__restrict__ chunk_count) {
    __shared__ int rp[TILE_CHUNK + 1];
    const int c0 = blockIdx.x * TILE_CHUNK;
    const int cn = min(TILE_CHUNK, n_nodes - c0);
    for (int i = threadIdx.x; i <= cn; i += blockDim.x) rp[i] = row_ptr[c0 + i];
    __syncthreads();
    if (threadIdx.x == 0) {
        int count = 0;
        int start = 0;
        while (start < cn) {
            tmp[c0 + count++] = c0 + start;
            int end = start + 1;   // a tile always holds at least one node
            while (end < cn && end - start < PVS_TILE_NODES &&
                   rp[end + 1] - rp[start] <= PVS_TILE_EDGES)
                ++end;
            start = end;
        }
        chunk_count[blockIdx.x] = count;
    }
}

__global__ void __launch_bounds__(256)
tiles_compact_kernel(const int32_t *__restrict__ tmp,
                     const int32_t *__restrict__ chunk_count,
                     const int32_t *__restrict__ chunk_off, int n_nodes,
                     int n_chunks, int32_t *__restrict__ tile_ptr,
                     int32_t *__restrict__ n_tiles) {
    const int c0 = blockIdx.x * TILE_CHUNK;
    const int cnt = chunk_count[blockIdx.x];
    const int off = chunk_off[blockIdx.x];
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) tile_ptr[off + i] = tmp[c0 + i];
    if (blockIdx.x == n_chunks - 1 && threadIdx.x == 0) {
        tile_ptr[off + cnt] = n_nodes;
        *n_tiles = off + cnt;
    }
}

// ---------------------------------------------------------------------------
// group edges by an integer key (row for CSR, col for CSC), stable
// ---------------------------------------------------------------------------
template <typename KeyT>
__global__ void key_count_kernel(const KeyT *__restrict__ keys, int64_t n_edges,
                                 int n_nodes, int32_t *__restrict__ deg,
                                 int32_t *__restrict__ bad,
                                 const int32_t *__restrict__ n_valid = nullptr) {
    // n_valid: device-side count of the keys actually present (a capacity-
    // bounded edge list is only filled up to row_ptr[n_nodes])
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_edges || (n_valid && e >= *n_valid)) return;
    int64_t k = (int64_t)keys[e];
    if (k < 0 || k >= n_nodes) {
        if (bad) *bad = 1;
        return;
    }
    atomicAdd(&deg[k], 1);
}

template <typename KeyT>
__global__ void key_place_kernel(const KeyT *__restrict__ keys, int64_t n_edges,
                                 int n_nodes, const int32_t *__restrict__ ptr,
                                 int32_t *__restrict__ cursor,
                                 int32_t *__restrict__ perm,
                                 const int32_t *__restrict__ n_valid = nullptr) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_edges || (n_valid && e >= *n_valid)) return;
    int64_t k = (int64_t)keys[e];
    if (k < 0 || k >= n_nodes) return;
    int p = atomicAdd(&cursor[k], 1);
    perm[ptr[k] + p] = (int32_t)e;
}

// symmetric graph: the edge arriving at j from i = col[p] (p in row j) is the
// entry of row i whose column is j.  One warp per node j, a lane per entry of
// its row; rows are short (~15), so the search is a plain scan.
__global__ void csc_symmetric_kernel(const int32_t *__restrict__ row_ptr,
                                     const int32_t *__restrict__ col, int n_nodes,
                                     int32_t *__restrict__ csc_eid,
                                     int32_t *__restrict__ asymmetric) {
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= n_nodes) return;
    const int lane = threadIdx.x & 31;
    const int lo = row_ptr[j], hi = row_ptr[j + 1];
    for (int p = lo + lane; p < hi; p += 32) {
        const int i = col[p];
        // a pair can be listed twice (once as an inter-, once as an intra-
        // molecular edge when both cut-offs admit it): the r-th i in row j
        // pairs with the r-th j in row i
        int rank = 0;
        for (int q = lo; q < p; ++q) rank += col[q] == i;
        int found = -1;
        if (i >= 0 && i < n_nodes) {
            const int qlo = row_ptr[i], qhi = row_ptr[i + 1];
            for (int q = qlo; q < qhi; ++q)
                if (col[q] == j && rank-- == 0) { found = q; break; }
        }
        if (found < 0) {
            found = p;
            if (asymmetric) *asymmetric = 1;
        }
        csc_eid[p] = found;
    }
}

// restore the caller's order inside every group (=> stable sort by key)
__global__ void segment_sort_kernel(const int32_t *__restrict__ ptr, int n_nodes,
                                    int32_t *__restrict__ perm) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    const int lo = ptr[i], hi = ptr[i + 1];
    for (int a = lo + 1; a < hi; ++a) {
        int v = perm[a];
        int b = a - 1;
        while (b >= lo && perm[b] > v) {
            perm[b + 1] = perm[b];
            --b;
        }
        perm[b + 1] = v;
    }
}

__global__ void csr_gather_kernel(const int64_t *__restrict__ edge_col,
                                  const int64_t *__restrict__ onehot,
                                  int n_classes, const int32_t *__restrict__ perm,
                                  const int32_t *__restrict__ n_valid,
                                  int64_t n_edges, int n_nodes,
                                  int32_t *__restrict__ col,
                                  uint8_t *__restrict__ attr,
                                  int32_t *__restrict__ bad) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // edges with an out-of-range row were never placed: slots past the valid
    // count hold no permutation entry
    if (p >= n_edges || p >= *n_valid) return;
    const int e = perm[p];
    int64_t c = edge_col[e];
    if (c < 0 || c >= n_nodes) {
        if (bad) *bad = 1;
        c = 0;
    }
    col[p] = (int32_t)c;
    if (attr != nullptr) {
        int cls = 0;
        if (onehot != nullptr)
            for (int d = 0; d < n_classes; ++d)
                if (onehot[(int64_t)e * n_classes + d] != 0) cls = d;
        attr[p] = (uint8_t)cls;
    }
}

__global__ void batch_to_ptr_kernel(const int64_t *__restrict__ batch, int n_nodes,
                                    int n_graphs, int32_t *__restrict__ ptr) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_nodes) return;
    int64_t prev = i == 0 ? -1 : batch[i - 1];
    int64_t cur = i == n_nodes ? (int64_t)n_graphs : batch[i];
    if (cur > n_graphs) cur = n_graphs;
    for (int64_t g = prev + 1; g <= cur; ++g)
        if (g >= 0 && g <= n_graphs) ptr[g] = i;
}

// After a capacity-bounded fill: no consumer may index past col/attr, so the
// offsets are cut at the capacity (a no-op unless *overflow was raised).
__global__ void clamp_row_ptr_kernel(int32_t *row_ptr, int n, int cap) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && row_ptr[i] > cap) row_ptr[i] = cap;
}

int clamp_row_ptr(int32_t *row_ptr, int n_nodes, int cap, cudaStream_t st) {
    clamp_row_ptr_kernel<<<(n_nodes + 1 + 255) / 256, 256, 0, st>>>(row_ptr, n_nodes + 1, cap);
    return check_launch();
}

}  // namespace pvs

using namespace pvs;

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

int64_t pvs_radius_graph_mask_bytes(int32_t n_nodes, int32_t max_complex_nodes) {
    const int64_t words = ((int64_t)max_complex_nodes + 31) / 32;
    return align_up((int64_t)n_nodes * 2 * words * 4, 256);
}

int64_t pvs_scan_scratch_bytes(int32_t n) {
    int64_t nb = ((int64_t)n + SCAN_TILE - 1) / SCAN_TILE + 1;
    return align_up(nb * (int64_t)sizeof(int32_t), 256);
}

int pvs_exclusive_scan(const int32_t *deg, int32_t n, int32_t *row_ptr,
                       void *scratch, void *stream) {
    if (n < 0 || row_ptr == nullptr || (n > 0 && (deg == nullptr || scratch == nullptr)))
        return PVS_ERR_INVALID_ARG;
    return exclusive_scan(deg, n, row_ptr, scratch, (cudaStream_t)stream);
}

static int rg_check(const double *coords, const int32_t *bp,
                    const int32_t *complex_ptr, int32_t n_complexes,
                    int32_t n_nodes, int32_t max_n, double r1, double r2) {
    if (n_complexes < 0 || n_nodes < 0 || max_n < 0) return PVS_ERR_INVALID_ARG;
    if (!(r1 >= 0.0) || !(r2 >= 0.0)) return PVS_ERR_INVALID_ARG;
    if (n_complexes > 0 && complex_ptr == nullptr) return PVS_ERR_INVALID_ARG;
    if (n_nodes > 0 && (coords == nullptr || bp == nullptr)) return PVS_ERR_INVALID_ARG;
    return PVS_OK;
}

int pvs_radius_graph_count(const double *coords, const int32_t *bp,
                           const int32_t *complex_ptr, int32_t n_complexes,
                           int32_t n_nodes, int32_t max_complex_nodes,
                           double inter_radius, double intra_radius,
                           int32_t *deg, int32_t *n_inter, int32_t *row_ptr,
                           uint32_t *mask_scratch, void *scratch, void *stream) {
    int rc = rg_check(coords, bp, complex_ptr, n_complexes, n_nodes,
                      max_complex_nodes, inter_radius, intra_radius);
    if (rc) return rc;
    if (row_ptr == nullptr || (n_nodes > 0 && (!deg || !n_inter || !scratch)))
        return PVS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (n_nodes > 0 && n_complexes > 0) {
        int stage = 1;
        size_t smem = rg_smem_bytes(max_complex_nodes, false, true);
        if (smem > (size_t)max_optin_smem()) {
            stage = 0;
            smem = rg_smem_bytes(max_complex_nodes, false, false);
        }
        if (smem > (size_t)max_optin_smem()) return PVS_ERR_TOO_LARGE;
        rc = ensure_smem(radius_graph_kernel<false>, smem);
        if (rc) return rc;
        if (mask_scratch != nullptr) {
            // the thread-per-atom count pass ORs bits into zeroed private rows
            rc = cuda_call(cudaMemsetAsync(
                mask_scratch, 0,
                (size_t)pvs_radius_graph_mask_bytes(n_nodes, max_complex_nodes), st));
            if (rc) return rc;
        }
        // thread-per-atom count pass (masks kept): one CTA per 512 atoms of the
        // largest complex; warp-per-atom pass: RG_SPLIT CTAs per complex
        int split = RG_SPLIT;
        if (mask_scratch != nullptr) {
            split = (max_complex_nodes + RG_THREADS - 1) / RG_THREADS;
            split = split < 1 ? 1 : (split > 8 ? 8 : split);
        }
        radius_graph_kernel<false><<<n_complexes * split, RG_THREADS, smem, st>>>(
            coords, bp, complex_ptr, inter_radius, intra_radius, deg, n_inter,
            nullptr, nullptr, nullptr, nullptr, nullptr, max_complex_nodes, stage,
            mask_scratch, 0, nullptr, split);
        rc = check_launch();
        if (rc) return rc;
    }
    return exclusive_scan(deg, n_nodes, row_ptr, scratch, st);
}

// Edge-packed tiles: tile t owns edges [128 t, min(128 t + 128, E)); last[t] is
// the node that holds its last edge (for E = 0 the single tile spans no edge and
// last[0] = n_nodes - 1).  One thread per tile: binary search in row_ptr.
__global__ void packed_tiles_kernel(const int32_t *__restrict__ row_ptr, int n_nodes, int cap,
                                    int32_t *__restrict__ last, int32_t *__restrict__ n_ptiles) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int E = row_ptr[n_nodes];
    int T = (E + PVS_TILE_EDGES - 1) / PVS_TILE_EDGES;
    if (T < 1) T = 1;
    if (T > cap) T = cap;
    if (t == 0) *n_ptiles = T;
    if (t >= T) return;
    if (E == 0) { last[t] = n_nodes > 0 ? n_nodes - 1 : 0; return; }
    const int e = min((t + 1) * PVS_TILE_EDGES, E) - 1;   // last edge of the tile
    // largest node i with row_ptr[i] <= e
    int lo = 0, hi = n_nodes;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (row_ptr[mid] <= e) lo = mid; else hi = mid;
    }
    last[t] = lo;
}

int pvs_radius_graph_fill(const double *coords, const int32_t *bp,
                          const int32_t *complex_ptr, int32_t n_complexes,
                          int32_t n_nodes, int32_t max_complex_nodes,
                          double inter_radius, double intra_radius,
                          const int32_t *n_inter, int32_t *row_ptr,
                          const uint32_t *mask_scratch, int32_t edge_capacity,
                          int32_t *col, uint8_t *attr, int32_t *ref_pos,
                          int32_t *overflow, void *stream) {
    int rc = rg_check(coords, bp, complex_ptr, n_complexes, n_nodes,
                      max_complex_nodes, inter_radius, intra_radius);
    if (rc) return rc;
    if (n_nodes == 0 || n_complexes == 0) return PVS_OK;
    if (!n_inter || !row_ptr || !col || !attr || edge_capacity < 0) return PVS_ERR_INVALID_ARG;
    if (mask_scratch != nullptr && ref_pos == nullptr) {
        const int words = (max_complex_nodes + 31) / 32;
        radius_graph_emit1_kernel<<<(n_nodes + 31) / 32, 256, 0, (cudaStream_t)stream>>>(
            mask_scratch, words, bp, complex_ptr, n_complexes, n_nodes, row_ptr, col, attr,
            edge_capacity, overflow);
        rc = check_launch();
        if (rc) return rc;
        return clamp_row_ptr(row_ptr, n_nodes, edge_capacity, (cudaStream_t)stream);
    }
    int stage = 1;
    size_t smem = rg_smem_bytes(max_complex_nodes, ref_pos != nullptr, true);
    if (smem > (size_t)max_optin_smem()) {
        stage = 0;
        smem = rg_smem_bytes(max_complex_nodes, ref_pos != nullptr, false);
    }
    if (smem > (size_t)max_optin_smem()) return PVS_ERR_TOO_LARGE;
    rc = ensure_smem(radius_graph_kernel<true>, smem);
    if (rc) return rc;
    radius_graph_kernel<true><<<n_complexes * RG_SPLIT, RG_THREADS, smem,
                                (cudaStream_t)stream>>>(
        coords, bp, complex_ptr, inter_radius, intra_radius, nullptr, nullptr,
        n_inter, row_ptr, col, attr, ref_pos, max_complex_nodes, stage, nullptr,
        edge_capacity, overflow);
    rc = check_launch();
    if (rc) return rc;
    return clamp_row_ptr(row_ptr, n_nodes, edge_capacity, (cudaStream_t)stream);
}

int pvs_prune_mask(const int32_t *row_ptr, const int32_t *col,
                   const int32_t *n_inter, const int32_t *complex_ptr,
                   int32_t n_complexes, int32_t n_nodes, uint8_t *keep,
                   void *stream) {
    if (n_complexes < 0 || n_nodes < 0) return PVS_ERR_INVALID_ARG;
    if (n_complexes == 0 || n_nodes == 0) return PVS_OK;
    if (!row_ptr || !n_inter || !complex_ptr || !keep) return PVS_ERR_INVALID_ARG;
    prune_mask_kernel<<<n_complexes, 256, 0, (cudaStream_t)stream>>>(
        row_ptr, col, n_inter, complex_ptr, keep);
    return check_launch();
}

int32_t pvs_packed_tiles_capacity(int32_t n_edges) {
    return (int32_t)((int64_t)n_edges / PVS_TILE_EDGES + 2);
}

int pvs_build_packed_tiles(const int32_t *row_ptr, int32_t n_nodes, int32_t n_edges,
                           int32_t *ptile_last, int32_t *n_ptiles, void *stream) {
    if (n_nodes < 0 || n_edges < 0 || !row_ptr || !ptile_last || !n_ptiles)
        return PVS_ERR_INVALID_ARG;
    const int cap = pvs_packed_tiles_capacity(n_edges);
    packed_tiles_kernel<<<(cap + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        row_ptr, n_nodes, cap, ptile_last, n_ptiles);
    return check_launch();
}

int32_t pvs_tiles_capacity(int32_t n_nodes, int32_t n_edges) {
    int64_t chunks = ((int64_t)n_nodes + TILE_CHUNK - 1) / TILE_CHUNK;
    int64_t cap = (int64_t)n_edges / (PVS_TILE_EDGES / 2) +
                  (int64_t)n_nodes / PVS_TILE_NODES + 2 * chunks + 2;
    if (cap > n_nodes) cap = n_nodes;   // never more tiles than nodes
    return (int32_t)(cap < 1 ? 1 : cap);
}

int64_t pvs_tiles_scratch_bytes(int32_t n_nodes) {
    int64_t chunks = ((int64_t)n_nodes + TILE_CHUNK - 1) / TILE_CHUNK;
    return align_up((int64_t)n_nodes * 4, 256) +
           2 * align_up((chunks + 1) * 4, 256) +
           pvs_scan_scratch_bytes((int32_t)chunks);
}

int pvs_build_tiles(const int32_t *row_ptr, int32_t n_nodes, int32_t *tile_ptr,
                    int32_t *n_tiles, void *scratch, void *stream) {
    if (n_nodes < 0 || !tile_ptr || !n_tiles) return PVS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (n_nodes == 0) {
        int rc = cuda_call(cudaMemsetAsync(n_tiles, 0, sizeof(int32_t), st));
        if (rc) return rc;
        return cuda_call(cudaMemsetAsync(tile_ptr, 0, sizeof(int32_t), st));
    }
    if (!row_ptr || !scratch) return PVS_ERR_INVALID_ARG;
    int chunks = (n_nodes + TILE_CHUNK - 1) / TILE_CHUNK;
    char *p = (char *)scratch;
    int32_t *tmp = (int32_t *)p;
    p += align_up((int64_t)n_nodes * 4, 256);
    int32_t *cnt = (int32_t *)p;
    p += align_up(((int64_t)chunks + 1) * 4, 256);
    int32_t *off = (int32_t *)p;
    p += align_up(((int64_t)chunks + 1) * 4, 256);
    tiles_walk_kernel<<<chunks, 256, 0, st>>>(row_ptr, n_nodes, tmp, cnt);
    g_launches += 1;
    int rc = exclusive_scan(cnt, chunks, off, p, st);
    if (rc) return rc;
    tiles_compact_kernel<<<chunks, 256, 0, st>>>(tmp, cnt, off, n_nodes, chunks,
                                                 tile_ptr, n_tiles);
    return check_launch();
}

int pvs_edge_index_to_csr(const int64_t *edge_index, int64_t n_edges,
                          const int64_t *edge_attr_onehot, int32_t n_classes,
                          int32_t n_nodes, int32_t *deg, int32_t *row_ptr,
                          int32_t *col, uint8_t *attr, int32_t *perm,
                          int32_t *bad_index, void *scratch, void *stream) {
    if (n_edges < 0 || n_nodes < 0 || n_classes < 0 ||
        n_classes > PVS_MAX_EDGE_CLASSES || n_edges > 0x7fffffffLL)
        return PVS_ERR_INVALID_ARG;
    if (!row_ptr || (n_nodes > 0 && (!deg || !scratch))) return PVS_ERR_INVALID_ARG;
    if (n_edges > 0 && (!edge_index || !col || !perm)) return PVS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if (n_nodes > 0) {
        rc = cuda_call(cudaMemsetAsync(deg, 0, (size_t)n_nodes * 4, st));
        if (rc) return rc;
    }
    int32_t *cursor = (int32_t *)scratch;
    void *scan_scratch = (char *)scratch + align_up((int64_t)n_nodes * 4, 256);
    const int T = 256;
    const unsigned nb = (unsigned)((n_edges + T - 1) / T);
    if (n_edges > 0) {
        key_count_kernel<int64_t><<<nb, T, 0, st>>>(edge_index, n_edges, n_nodes,
                                                   deg, bad_index);
        g_launches += 1;
    }
    rc = exclusive_scan(deg, n_nodes, row_ptr, scan_scratch, st);
    if (rc) return rc;
    if (n_edges > 0 && n_nodes > 0) {
        rc = cuda_call(cudaMemsetAsync(cursor, 0, (size_t)n_nodes * 4, st));
        if (rc) return rc;
        key_place_kernel<int64_t><<<nb, T, 0, st>>>(edge_index, n_edges, n_nodes,
                                                   row_ptr, cursor, perm);
        segment_sort_kernel<<<(n_nodes + T - 1) / T, T, 0, st>>>(row_ptr, n_nodes,
                                                               perm);
        csr_gather_kernel<<<nb, T, 0, st>>>(edge_index + n_edges,
                                            edge_attr_onehot, n_classes, perm,
                                            row_ptr + n_nodes, n_edges, n_nodes, col, attr,
                                            bad_index);
        g_launches += 3;
    }
    return check_launch(0);
}

int pvs_csr_transpose(const pvs_graph *g, int32_t *csc_ptr, int32_t *csc_eid,
                      void *scratch, void *stream) {
    if (!g || !csc_ptr || g->n_nodes < 0 || g->n_edges < 0) return PVS_ERR_INVALID_ARG;
    if (g->n_nodes > 0 && !scratch) return PVS_ERR_INVALID_ARG;
    if (g->n_edges > 0 && (!g->col || !csc_eid)) return PVS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int n = g->n_nodes;
    const int64_t E = g->n_edges;
    // g->n_edges may be the CAPACITY of a graph built without a host read-back
    // of its edge count; row_ptr[n] is the number of edges actually present
    const int32_t *n_valid = g->row_ptr ? g->row_ptr + n : nullptr;
    // scratch: deg[n] | cursor[n] | scan scratch
    int32_t *deg = (int32_t *)scratch;
    int32_t *cursor = (int32_t *)((char *)scratch + align_up((int64_t)n * 4, 256));
    void *scan_scratch = (char *)cursor + align_up((int64_t)n * 4, 256);
    int rc;
    if (n > 0) {
        rc = cuda_call(cudaMemsetAsync(scratch, 0, 2 * align_up((int64_t)n * 4, 256), st));
        if (rc) return rc;
    }
    const int T = 256;
    const unsigned nb = (unsigned)((E + T - 1) / T);
    if (E > 0)
        key_count_kernel<int32_t><<<nb, T, 0, st>>>(g->col, E, n, deg, nullptr, n_valid);
    if (E > 0) g_launches += 1;
    rc = exclusive_scan(deg, n, csc_ptr, scan_scratch, st);
    if (rc) return rc;
    if (E > 0 && n > 0) {
        key_place_kernel<int32_t><<<nb, T, 0, st>>>(g->col, E, n, csc_ptr, cursor,
                                                   csc_eid, n_valid);
        segment_sort_kernel<<<(n + T - 1) / T, T, 0, st>>>(csc_ptr, n, csc_eid);
        g_launches += 2;
    }
    return check_launch(0);
}

int pvs_csr_transpose_symmetric(const pvs_graph *g, int32_t *csc_eid, int32_t *asymmetric,
                                void *stream) {
    if (!g || g->n_nodes < 0 || g->n_edges < 0) return PVS_ERR_INVALID_ARG;
    if (g->n_nodes == 0 || g->n_edges == 0) return PVS_OK;
    if (!g->row_ptr || !g->col || !csc_eid) return PVS_ERR_INVALID_ARG;
    const int warps_per_block = 8;
    csc_symmetric_kernel<<<(g->n_nodes + warps_per_block - 1) / warps_per_block,
                           32 * warps_per_block, 0, (cudaStream_t)stream>>>(
        g->row_ptr, g->col, g->n_nodes, csc_eid, asymmetric);
    return check_launch();
}

int pvs_batch_to_ptr(const int64_t *batch, int32_t n_nodes, int32_t n_graphs,
                     int32_t *graph_ptr, void *stream) {
    if (n_nodes < 0 || n_graphs < 0 || !graph_ptr) return PVS_ERR_INVALID_ARG;
    if (n_nodes > 0 && !batch) return PVS_ERR_INVALID_ARG;
    const int T = 256;
    batch_to_ptr_kernel<<<(n_nodes + 1 + T - 1) / T, T, 0, (cudaStream_t)stream>>>(
        batch, n_nodes, n_graphs, graph_ptr);
    return check_launch();
}

}  // extern "C"
