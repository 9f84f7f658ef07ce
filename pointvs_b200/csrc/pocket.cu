// K1p: radius graph of ligand poses against resident receptors.
//
// Replaces /root/reference/point_vs/preprocessing/preprocessing.py:68-155
// (generate_edges) for the complexes K0 assembles from resident receptors
// (data_loaders.py:259-309), and produces what K1 (graph.cu) would produce on
// them, byte for byte.
//
// In a pocket screen nearly all pairs K1 tests are receptor-receptor pairs,
// and they are the same for every pose.  So, once per pocket:
//   pocket_cells_kernel : a cell list of each receptor's emitted atoms;
//   pocket_rr_kernel    : the receptor-receptor CSR at intra_radius.
// Per batch, one group of CTAs per pose:
//   ligand rows   : a warp per ligand atom searches the resident cell list
//                   (kept receptor atoms only) and tests the other ligand
//                   atoms;
//   receptor rows : a thread per kept receptor atom tests the ligand atoms
//                   and copies its cached receptor-receptor row, dropping the
//                   atoms the pose's crop did not keep.
// A kept receptor atom j becomes node n_lig + (kept atoms before j): a prefix
// popcount of the pose's keep bits.  Within a row: inter edges by column
// (attr 1), then intra edges by column (attr 0, receptor-receptor attr 2).
#include <algorithm>

#include "graph_common.cuh"

namespace pvs {

constexpr int PK_MAX_CELLS = PVS_POCKET_MAX_DIM * PVS_POCKET_MAX_DIM * PVS_POCKET_MAX_DIM;
constexpr int PK_BUILD_THREADS = 1024;
constexpr int PK_RR_THREADS = 256;
constexpr int PG_THREADS = 256;
constexpr int PG_WARPS = PG_THREADS / 32;
constexpr int PG_ATOMS_PER_CTA = 256;   // receptor atoms per CTA of a pose
constexpr int PG_MAX_SPLIT = 8;         // CTAs per pose

// views into pvs_pocket.cells
struct PocketCells {
    double *geom;         // [R][6]: box low corner xyz, 1 / cell edge xyz
    int32_t *dims;        // [R][4]: cells per axis xyz, -
    int32_t *cell_start;  // [R][PK_MAX_CELLS + 1], relative to rec_ptr[r]
    int32_t *cell_fill;   // [R][PK_MAX_CELLS]: build scratch, not resident
    int32_t *cell_atom;   // [A]: receptor r's emitted atoms, by cell, at
                          //      [rec_ptr[r], rec_ptr[r] + emitted), as the
                          //      index inside the receptor
    double *cell_xyz;     // [A][3]: their coordinates, same order
};

// build scratch: cell_fill [R][PK_MAX_CELLS] | receptor-receptor degrees [A] |
// scan scratch
static int64_t build_scratch_layout(void *base, int n_rec, int n_atoms, int32_t **cell_fill,
                                    int32_t **rr_deg, void **scan) {
    char *p = (char *)base;
    const int64_t a = align_up((int64_t)n_rec * PK_MAX_CELLS * 4, 256);
    const int64_t b = align_up((int64_t)n_atoms * 4, 256);
    if (p) {
        *cell_fill = (int32_t *)p;
        *rr_deg = (int32_t *)(p + a);
        *scan = p + a + b;
    }
    return a + b + pvs_scan_scratch_bytes(n_atoms);
}

static int64_t cells_layout(void *base, int n_rec, int n_atoms, PocketCells *c) {
    char *p = (char *)base;
    int64_t off = 0;
    auto take = [&](int64_t bytes) {
        char *q = p ? p + off : nullptr;
        off += align_up(bytes, 256);
        return q;
    };
    PocketCells v;
    v.geom = (double *)take((int64_t)n_rec * 6 * 8);
    v.dims = (int32_t *)take((int64_t)n_rec * 4 * 4);
    v.cell_start = (int32_t *)take((int64_t)n_rec * (PK_MAX_CELLS + 1) * 4);
    v.cell_fill = nullptr;
    v.cell_atom = (int32_t *)take((int64_t)n_atoms * 4);
    v.cell_xyz = (double *)take((int64_t)n_atoms * 3 * 8);
    if (c) *c = v;
    return off;
}

// ---------------------------------------------------------------------------
// build: one CTA per receptor bins its emitted atoms
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(PK_BUILD_THREADS)
pocket_cells_kernel(const double *__restrict__ xyz, const uint8_t *__restrict__ emit,
                    const int32_t *__restrict__ rec_ptr, double r_max, PocketCells c) {
    __shared__ double red[6][PK_BUILD_THREADS / 32];
    __shared__ double box[6];
    __shared__ int warp_buf[33];
    const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r0 = rec_ptr[r], n = rec_ptr[r + 1] - r0;
    const double *rx = xyz + 3 * (size_t)r0;
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (int i = tid; i < n; i += PK_BUILD_THREADS) {
        if (!emit[r0 + i]) continue;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            lo[a] = fmin(lo[a], rx[3 * i + a]);
            hi[a] = fmax(hi[a], rx[3 * i + a]);
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
            red[a][warp] = lo[a];
            red[3 + a][warp] = hi[a];
        }
    }
    __syncthreads();
    if (tid < 3) {
        double l = red[tid][0], h = red[3 + tid][0];
        for (int w = 1; w < PK_BUILD_THREADS / 32; ++w) {
            l = fmin(l, red[tid][w]);
            h = fmax(h, red[3 + tid][w]);
        }
        if (l > h) l = h = 0.0;   // no emitted atom: one empty cell
        box[tid] = l;
        box[3 + tid] = h;
    }
    __syncthreads();
    // cell edge >= r_max * (1 + 1e-6): cs0 when (int)(ext / cs0) + 1 cells of
    // that edge fit PVS_POCKET_MAX_DIM, else ext / PVS_POCKET_MAX_DIM * (1 + 1e-6),
    // which is then >= cs0 * (1 + 1e-6).  Never smaller than cs0, so two atoms
    // closer than r_max are at most one cell apart on every axis.
    const double cs0 = fmax(r_max * (1.0 + 1e-6), 1e-9);
    int dim[3];
    double inv[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double ext = box[3 + a] - box[a];
        const double q = ext / cs0;
        if (q >= (double)PVS_POCKET_MAX_DIM) {
            dim[a] = PVS_POCKET_MAX_DIM;
            inv[a] = 1.0 / (ext / PVS_POCKET_MAX_DIM * (1.0 + 1e-6));
        } else {
            dim[a] = (int)q + 1;
            inv[a] = 1.0 / cs0;
        }
    }
    const int ncell = dim[0] * dim[1] * dim[2];
    if (tid == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            c.geom[6 * r + a] = box[a];
            c.geom[6 * r + 3 + a] = inv[a];
            c.dims[4 * r + a] = dim[a];
        }
    }
    int32_t *cs = c.cell_start + (size_t)r * (PK_MAX_CELLS + 1);
    int32_t *cf = c.cell_fill + (size_t)r * PK_MAX_CELLS;
    for (int i = tid; i < ncell; i += PK_BUILD_THREADS) {
        cs[i] = 0;
        cf[i] = 0;
    }
    __syncthreads();
    auto cell_of = [&](int i) {
        return cell_coord(rx[3 * i], box[0], inv[0], dim[0]) +
               dim[0] * (cell_coord(rx[3 * i + 1], box[1], inv[1], dim[1]) +
                         dim[1] * cell_coord(rx[3 * i + 2], box[2], inv[2], dim[2]));
    };
    for (int i = tid; i < n; i += PK_BUILD_THREADS)
        if (emit[r0 + i]) atomicAdd(&cs[cell_of(i)], 1);
    __syncthreads();
    const int total = smem_scan_excl(cs, ncell, warp_buf);
    if (tid == 0) cs[ncell] = total;
    __syncthreads();
    for (int i = tid; i < n; i += PK_BUILD_THREADS) {
        if (!emit[r0 + i]) continue;
        const int cell = cell_of(i);
        const int p = r0 + cs[cell] + atomicAdd(&cf[cell], 1);
        c.cell_atom[p] = i;
        c.cell_xyz[3 * (size_t)p] = rx[3 * i];
        c.cell_xyz[3 * (size_t)p + 1] = rx[3 * i + 1];
        c.cell_xyz[3 * (size_t)p + 2] = rx[3 * i + 2];
    }
}

// Visit the cell-list positions q (relative to rec_ptr[r]) of receptor r's
// emitted atoms in the 27 cells around (x, y, z), lanes l, l + W, ...
template <typename F>
__device__ __forceinline__ void pocket_search(const PocketCells &c, int r, double x, double y,
                                              double z, int l, int W, F &&visit) {
    const double *g = c.geom + 6 * r;
    const int32_t *d = c.dims + 4 * r;
    const int32_t *cs = c.cell_start + (size_t)r * (PK_MAX_CELLS + 1);
    const int d0 = d[0], d1 = d[1], d2 = d[2];
    const int ci0 = cell_coord(x, g[0], g[3], d0);
    const int ci1 = cell_coord(y, g[1], g[4], d1);
    const int ci2 = cell_coord(z, g[2], g[5], d2);
    const int x_lo = max(ci0 - 1, 0), x_hi = min(ci0 + 1, d0 - 1);
#pragma unroll 1
    for (int dz = -1; dz <= 1; ++dz) {
        const int c2 = ci2 + dz;
        if (c2 < 0 || c2 >= d2) continue;
#pragma unroll 1
        for (int dy = -1; dy <= 1; ++dy) {
            const int c1 = ci1 + dy;
            if (c1 < 0 || c1 >= d1) continue;
            const int cb = d0 * (c1 + d1 * c2);
            const int q_end = cs[cb + x_hi + 1];
            for (int q = cs[cb + x_lo] + l; q < q_end; q += W) visit(q);
        }
    }
}

// receptor-receptor CSR: a thread per receptor atom (grid.x = receptor)
template <bool FILL>
__global__ void __launch_bounds__(PK_RR_THREADS)
pocket_rr_kernel(const double *__restrict__ xyz, const uint8_t *__restrict__ emit,
                 const int32_t *__restrict__ rec_ptr, const PairBand band, PocketCells c,
                 int32_t *__restrict__ rr, int32_t *__restrict__ rr_col) {
    const int r = blockIdx.x;
    const int r0 = rec_ptr[r], n = rec_ptr[r + 1] - r0;
    const int i = blockIdx.y * PK_RR_THREADS + threadIdx.x;
    if (i >= n) return;
    if (!emit[r0 + i]) {
        if (!FILL) rr[r0 + i] = 0;   // count pass: rr = degrees
        return;
    }
    const double xi = xyz[3 * (size_t)(r0 + i)], yi = xyz[3 * (size_t)(r0 + i) + 1],
                 zi = xyz[3 * (size_t)(r0 + i) + 2];
    int32_t *row = FILL ? rr_col + rr[r0 + i] : nullptr;   // fill pass: rr = row_ptr
    const double *cxyz = c.cell_xyz + 3 * (size_t)r0;
    const int32_t *catom = c.cell_atom + r0;
    int cnt = 0;
    pocket_search(c, r, xi, yi, zi, 0, 1, [&](int q) {
        bool pos, in_inter, in_intra;
        pair_test(band, xi, yi, zi, cxyz[3 * q], cxyz[3 * q + 1], cxyz[3 * q + 2], pos,
                  in_inter, in_intra);
        if (pos && in_intra) {
            if (FILL) row[cnt] = catom[q];
            ++cnt;
        }
    });
    if (!FILL) {
        rr[r0 + i] = cnt;
    } else {
        // file order inside the row (rows are short: insertion sort)
        for (int a = 1; a < cnt; ++a) {
            const int v = row[a];
            int b = a - 1;
            while (b >= 0 && row[b] > v) {
                row[b + 1] = row[b];
                --b;
            }
            row[b + 1] = v;
        }
    }
}

// ---------------------------------------------------------------------------
// per batch: gridDim.y = `split` CTAs per pose
// ---------------------------------------------------------------------------
// CTAs of a pose's receptor rows: one per PG_ATOMS_PER_CTA kept atoms, at
// least one, at most PG_MAX_SPLIT
__host__ __device__ __forceinline__ int pg_split_of(int atoms) {
    const int s = (atoms + PG_ATOMS_PER_CTA - 1) / PG_ATOMS_PER_CTA;
    return s < 1 ? 1 : (s > PG_MAX_SPLIT ? PG_MAX_SPLIT : s);
}

// position of the set bit of rank k (0-based) in m; k < __popc(m)
__device__ __forceinline__ int nth_set_bit(uint32_t m, int k) {
    int p = 0;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const int c = __popc(m & ((1u << s) - 1u));
        if (k >= c) {
            k -= c;
            m >>= s;
            p += s;
        }
    }
    return p;
}

static size_t pg_smem_bytes(int max_lig, int mask_words) {
    return (size_t)(3 * max_lig + 6) * sizeof(double) +
           (size_t)(2 + 2 * PG_WARPS) * mask_words * sizeof(uint32_t) + 33 * sizeof(int);
}

template <bool FILL, bool LIG_ROWS>
__global__ void __launch_bounds__(PG_THREADS)
pocket_graph_kernel(PocketCells c, const double *__restrict__ rec_xyz,
                    const int32_t *__restrict__ rec_ptr, const int32_t *__restrict__ rr_ptr,
                    const int32_t *__restrict__ rr_col, const double *__restrict__ coords,
                    const int32_t *__restrict__ complex_ptr, const uint32_t *__restrict__ mask,
                    int mask_words, const int32_t *__restrict__ lig_count, int max_lig,
                    const int32_t *__restrict__ rec_of_pose, const PairBand band, int32_t *__restrict__ deg, int32_t *__restrict__ n_inter,
                    const int32_t *__restrict__ row_ptr, int32_t *__restrict__ col,
                    uint8_t *__restrict__ attr, int edge_capacity,
                    int32_t *__restrict__ overflow) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int split = gridDim.y;
    const int b = blockIdx.x, part = blockIdx.y;   // split = gridDim.y
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n0 = complex_ptr[b], n = complex_ptr[b + 1] - n0;
    if (n <= 0) return;
    const int nl = lig_count[b];
    if (nl < 0 || nl > max_lig || nl > n) {
        // outside the caller's bound: the pose gets no edges, and the fill
        // reports it through *overflow (2)
        if (!FILL)
            for (int i = part * PG_THREADS + tid; i < n; i += split * PG_THREADS) {
                deg[n0 + i] = 0;
                n_inter[n0 + i] = 0;
            }
        else if (overflow && part == 0 && tid == 0)
            *overflow = 2;
        return;
    }
    const int rid = rec_of_pose ? rec_of_pose[b] : 0;
    const int r0 = rec_ptr[rid], nr = min(rec_ptr[rid + 1] - r0, mask_words * 32);
    const int words = (nr + 31) / 32;
    double *lx = reinterpret_cast<double *>(smem_raw);
    double *ly = lx + max_lig, *lz = ly + max_lig;
    double *lbox = lz + max_lig;   // ligand box grown by the larger radius
    uint32_t *mw = reinterpret_cast<uint32_t *>(lbox + 6);   // keep bits
    int *wp = reinterpret_cast<int *>(mw + mask_words);          // kept before word
    uint32_t *wmask = reinterpret_cast<uint32_t *>(wp + mask_words);
    int *warp_buf = reinterpret_cast<int *>(wmask + 2 * PG_WARPS * mask_words);

    for (int i = tid; i < nl; i += PG_THREADS) {
        lx[i] = coords[3 * (size_t)(n0 + i)];
        ly[i] = coords[3 * (size_t)(n0 + i) + 1];
        lz[i] = coords[3 * (size_t)(n0 + i) + 2];
    }
    const uint32_t *mrow = mask + (size_t)b * mask_words;
    for (int w = tid; w < words; w += PG_THREADS) {
        // no bit at or above nr: kept atom t always lands on an atom j < nr
        const uint32_t v = mrow[w] & (nr - 32 * w >= 32 ? ~0u : (1u << (nr - 32 * w)) - 1u);
        mw[w] = v;
        wp[w] = __popc(v);
    }
    __syncthreads();
    if (warp == 0) {
        // a receptor atom outside this box has no ligand neighbour:
        // |dx| >= r (1 + 1e-6) rules the pair out whatever the rounding of d2
        double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
        for (int k = lane; k < nl; k += 32) {
            lo[0] = fmin(lo[0], lx[k]); hi[0] = fmax(hi[0], lx[k]);
            lo[1] = fmin(lo[1], ly[k]); hi[1] = fmax(hi[1], ly[k]);
            lo[2] = fmin(lo[2], lz[k]); hi[2] = fmax(hi[2], lz[k]);
        }
        const double grow = fmax(band.r_inter, band.r_intra) * (1.0 + 1e-6) + 1e-9;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                lo[a] = fmin(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
                hi[a] = fmax(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
            }
            if (lane == 0) {
                lbox[a] = lo[a] - grow;
                lbox[3 + a] = hi[a] + grow;
            }
        }
    }
    const int kept_total = smem_scan_excl(wp, words, warp_buf);   // its barriers also publish lbox

    auto kept = [&](int j) { return (mw[j >> 5] >> (j & 31)) & 1u; };
    auto node = [&](int j) {   // complex-local node of kept receptor atom j
        return nl + wp[j >> 5] + __popc(mw[j >> 5] & ((1u << (j & 31)) - 1u));
    };
    auto put = [&](int off, int c_, uint8_t a) {
        if (off < edge_capacity) {
            col[off] = c_;
            attr[off] = a;
        } else if (overflow) {
            *overflow = 1;
        }
    };

    // ---- receptor rows: a thread per kept receptor atom of this CTA's slice ----
    auto receptor_rows = [&]() {
        // the pose's kept atoms t = 0 .. n - nl - 1 are nodes nl + t; the pose
        // uses as many of the grid's CTAs as its kept count needs
        const int n_kept = min(n - nl, kept_total);
        const int used = pg_split_of(n_kept);
        if (part >= used) return;
        const int t_lo = (int)(((long long)n_kept * part) / used);
        const int t_hi = (int)(((long long)n_kept * (part + 1)) / used);
        for (int t = t_lo + tid; t < t_hi; t += PG_THREADS) {
            // kept atom t: the last word with wp[w] <= t, then the bit of rank
            // t - wp[w] inside it
            int w_lo = 0, w_hi = words;   // wp[w_lo] <= t < wp[w_hi], wp[words] = kept_total
            while (w_hi - w_lo > 1) {
                const int mid = (w_lo + w_hi) >> 1;
                if (wp[mid] <= t) w_lo = mid; else w_hi = mid;
            }
            const int j = w_lo * 32 + nth_set_bit(mw[w_lo], t - wp[w_lo]);
            const int row = n0 + nl + t;
            const double xj = rec_xyz[3 * (size_t)(r0 + j)], yj = rec_xyz[3 * (size_t)(r0 + j) + 1],
                         zj = rec_xyz[3 * (size_t)(r0 + j) + 2];
            const bool near = nl > 0 && xj > lbox[0] && xj < lbox[3] && yj > lbox[1] &&
                              yj < lbox[4] && zj > lbox[2] && zj < lbox[5];
            const int e_lo = rr_ptr[r0 + j], e_hi = rr_ptr[r0 + j + 1];
            if (!FILL) {
                int li = 0, la = 0, rk = 0;
                if (near)
                    for (int k = 0; k < nl; ++k) {
                        bool pos, in_inter, in_intra;
                        pair_test(band, xj, yj, zj, lx[k], ly[k], lz[k], pos, in_inter, in_intra);
                        li += (pos && in_inter) ? 1 : 0;
                        la += (pos && in_intra) ? 1 : 0;
                    }
                for (int e = e_lo; e < e_hi; ++e) rk += kept(rr_col[e]) ? 1 : 0;
                deg[row] = li + la + rk;
                n_inter[row] = li;
            } else {
                int off = row_ptr[row];
                if (near) {
    #pragma unroll 1
                    for (int pass = 0; pass < 2; ++pass)
                        for (int k = 0; k < nl; ++k) {
                            bool pos, in_inter, in_intra;
                            pair_test(band, xj, yj, zj, lx[k], ly[k], lz[k], pos, in_inter,
                                      in_intra);
                            if (pos && (pass == 0 ? in_inter : in_intra))
                                put(off++, n0 + k, pass == 0 ? 1 : 0);
                        }
                }
                for (int e = e_lo; e < e_hi; ++e) {
                    const int jj = rr_col[e];
                    if (kept(jj)) put(off++, n0 + node(jj), 2);
                }
            }
        }
    };
    // ---- ligand rows: a warp per ligand atom ----
    auto ligand_rows = [&]() {
        uint32_t *m_inter = wmask + (size_t)warp * 2 * mask_words;
        uint32_t *m_intra = m_inter + mask_words;
        for (int i = part * PG_WARPS + warp; i < nl; i += split * PG_WARPS) {
            for (int w = lane; w < words; w += 32) {
                m_inter[w] = 0u;
                m_intra[w] = 0u;
            }
            __syncwarp();
            // the query point is re-read from shared memory inside the visit:
            // kept in registers across the pair test's sqrt subroutine, it spilled
            pocket_search(c, rid, lx[i], ly[i], lz[i], lane, 32, [&](int q) {
                const int j = c.cell_atom[r0 + q];
                if (j >= nr || !kept(j)) return;
                const double *pj = c.cell_xyz + 3 * (size_t)(r0 + q);
                bool pos, in_inter, in_intra;
                pair_test(band, lx[i], ly[i], lz[i], pj[0], pj[1], pj[2], pos, in_inter,
                          in_intra);
                const unsigned bit = 1u << (j & 31);
                if (pos && in_inter) atomicOr(&m_inter[j >> 5], bit);   // :110-117
                if (pos && in_intra) atomicOr(&m_intra[j >> 5], bit);   // :119-121
            });
            __syncwarp();
            const double xi = lx[i], yi = ly[i], zi = lz[i];
            if (!FILL) {
                int ci = 0, ca = 0;
                for (int w = lane; w < words; w += 32) {
                    ci += __popc(m_inter[w]);
                    ca += __popc(m_intra[w]);
                }
                for (int k = lane; k < nl; k += 32) {   // ligand-ligand: intra only
                    bool pos, in_inter, in_intra;
                    pair_test(band, xi, yi, zi, lx[k], ly[k], lz[k], pos, in_inter, in_intra);
                    ca += (pos && in_intra) ? 1 : 0;
                }
                ci = warp_sum_int(ci);
                ca = warp_sum_int(ca);
                if (lane == 0) {
                    deg[n0 + i] = ci + ca;
                    n_inter[n0 + i] = ci;
                }
            } else {
                int run = row_ptr[n0 + i];
                // set bits of a mask in ascending j -> receptor columns
                auto emit_mask = [&](const uint32_t *mk, uint8_t a) {
                    for (int w0 = 0; w0 < words; w0 += 32) {
                        const int w = w0 + lane;
                        unsigned bits = w < words ? mk[w] : 0u;
                        const int cnt = __popc(bits);
                        const int incl = warp_scan_incl(cnt, lane);
                        int off = run + incl - cnt;
                        while (bits) {
                            const int j = w * 32 + __ffs(bits) - 1;
                            bits &= bits - 1;
                            put(off++, n0 + node(j), a);
                        }
                        run += __shfl_sync(0xffffffffu, incl, 31);
                    }
                };
                emit_mask(m_inter, 1);
                for (int k0 = 0; k0 < nl; k0 += 32) {   // ligand-ligand, ascending
                    const int k = k0 + lane;
                    bool hit = false;
                    if (k < nl) {
                        bool pos, in_inter, in_intra;
                        pair_test(band, xi, yi, zi, lx[k], ly[k], lz[k], pos, in_inter, in_intra);
                        hit = pos && in_intra;
                    }
                    const unsigned bal = __ballot_sync(0xffffffffu, hit);
                    if (hit) put(run + __popc(bal & ((1u << lane) - 1u)), n0 + k, 0);
                    run += __popc(bal);
                }
                emit_mask(m_intra, 0);
            }
            __syncwarp();
        }
    };
    // Separate launches for the two independent halves: together in one
    // kernel, the values live across the pair test's sqrt subroutine did not
    // all fit the registers the call leaves alone (spills).
    if (LIG_ROWS)
        ligand_rows();
    else
        receptor_rows();
}

// ---------------------------------------------------------------------------
// compose: part k of a pocket of several receptors, copied from a built
// pocket.  Cell positions are relative to rec_ptr[r] and rr_col holds indices
// inside the receptor, so only rr_ptr moves: by the edges of the parts before
// (out.rr_ptr[a_off], written by part k - 1's launch; 0 for the first part).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pocket_compose_kernel(PocketCells src, const int32_t *__restrict__ src_rr_ptr,
                      const int32_t *__restrict__ src_rr_col, int n_rec, int n_atoms,
                      PocketCells dst, int32_t *__restrict__ dst_rr_ptr,
                      int32_t *__restrict__ dst_rr_col, int r_off, int a_off, bool first) {
    const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    const int32_t e_off = first ? 0 : dst_rr_ptr[a_off];
    for (int64_t i = i0; i < 6 * n_rec; i += step) dst.geom[6 * (int64_t)r_off + i] = src.geom[i];
    for (int64_t i = i0; i < 4 * n_rec; i += step) dst.dims[4 * (int64_t)r_off + i] = src.dims[i];
    const int64_t n_cs = (int64_t)n_rec * (PK_MAX_CELLS + 1);
    for (int64_t i = i0; i < n_cs; i += step)
        dst.cell_start[(int64_t)r_off * (PK_MAX_CELLS + 1) + i] = src.cell_start[i];
    for (int64_t i = i0; i < n_atoms; i += step) {
        dst.cell_atom[a_off + i] = src.cell_atom[i];
        dst.cell_xyz[3 * (a_off + i)] = src.cell_xyz[3 * i];
        dst.cell_xyz[3 * (a_off + i) + 1] = src.cell_xyz[3 * i + 1];
        dst.cell_xyz[3 * (a_off + i) + 2] = src.cell_xyz[3 * i + 2];
    }
    // entry a_off is the previous part's end (or 0): write 1 .. n_atoms
    if (first && i0 == 0) dst_rr_ptr[0] = 0;
    for (int64_t i = i0 + 1; i <= n_atoms; i += step)
        dst_rr_ptr[a_off + i] = src_rr_ptr[i] + e_off;
    const int32_t n_e = src_rr_ptr[n_atoms];
    for (int64_t e = i0; e < n_e; e += step) dst_rr_col[e_off + e] = src_rr_col[e];
}

}  // namespace pvs

using namespace pvs;

static int pocket_check(const pvs_pocket *p) {
    if (!p || p->n_receptors < 0 || p->n_atoms < 0 || p->max_atoms < 0)
        return PVS_ERR_INVALID_ARG;
    if (!(p->inter_radius >= 0.0) || !(p->intra_radius >= 0.0)) return PVS_ERR_INVALID_ARG;
    if (p->n_receptors > 0 && !p->rec_ptr) return PVS_ERR_INVALID_ARG;
    if (p->n_atoms > 0 && (!p->xyz || !p->emit || !p->cells || !p->rr_ptr))
        return PVS_ERR_INVALID_ARG;
    if (p->max_atoms > p->n_atoms) return PVS_ERR_INVALID_ARG;
    if (p->max_atoms > PVS_POCKET_MAX_REC_ATOMS) return PVS_ERR_TOO_LARGE;
    return PVS_OK;
}

static int pose_check(const pvs_pocket *p, const double *coords, const int32_t *complex_ptr,
                      int32_t n_poses, int32_t n_nodes, const uint32_t *mask,
                      int32_t mask_words, const int32_t *lig_count, int32_t max_lig,
                      double r_inter, double r_intra) {
    int rc = pocket_check(p);
    if (rc) return rc;
    if (n_poses < 0 || n_nodes < 0 || mask_words < 0 || max_lig < 0) return PVS_ERR_INVALID_ARG;
    if (!(r_inter >= 0.0) || !(r_intra >= 0.0)) return PVS_ERR_INVALID_ARG;
    // the cached receptor-receptor rows and the cell size hold for the
    // pocket's own radii only
    if (r_inter != p->inter_radius || r_intra != p->intra_radius) return PVS_ERR_INVALID_ARG;
    if (n_poses > 0 && (!complex_ptr || !mask || !lig_count || p->n_receptors < 1))
        return PVS_ERR_INVALID_ARG;
    if (n_nodes > 0 && !coords) return PVS_ERR_INVALID_ARG;
    if ((int64_t)mask_words * 32 < p->max_atoms) return PVS_ERR_INVALID_ARG;
    if (p->n_atoms > 0 && !p->rr_col) return PVS_ERR_INVALID_ARG;
    if (max_lig > PVS_POCKET_MAX_LIG_ATOMS) return PVS_ERR_TOO_LARGE;
    if (mask_words > PVS_POCKET_MAX_REC_ATOMS / 32) return PVS_ERR_TOO_LARGE;
    return PVS_OK;
}

template <bool FILL>
static int pg_launch(const pvs_pocket *p, const double *coords, const int32_t *complex_ptr,
                     int32_t n_poses, const uint32_t *mask, int32_t mask_words,
                     const int32_t *lig_count, int32_t max_lig, const int32_t *rec_of_pose,
                     double r_inter, double r_intra, int32_t *deg, int32_t *n_inter,
                     const int32_t *row_ptr, int32_t edge_capacity, int32_t *col,
                     uint8_t *attr, int32_t *overflow, cudaStream_t st) {
    const size_t smem = pg_smem_bytes(max_lig > 0 ? max_lig : 1, mask_words);
    if (smem > (size_t)max_optin_smem()) return PVS_ERR_TOO_LARGE;
    int rc = ensure_smem(pocket_graph_kernel<FILL, true>, smem);
    if (rc) return rc;
    rc = ensure_smem(pocket_graph_kernel<FILL, false>, smem);
    if (rc) return rc;
    PocketCells c;
    cells_layout(p->cells, p->n_receptors, p->n_atoms, &c);
    // receptor rows: enough CTAs for a pose that keeps the largest receptor
    // whole; each pose runs on pg_split_of(its kept count) of them and the
    // rest return at once.  Ligand rows: no more CTAs than the largest ligand
    // has warps' worth of atoms
    const dim3 grid(n_poses, pg_split_of(p->max_atoms));
    const int ml = max_lig > 0 ? max_lig : 1;
    const dim3 grid_lig(n_poses, std::min<int>(grid.y, (ml + PG_WARPS - 1) / PG_WARPS));
    const PairBand band = pair_band(r_inter, r_intra);
    pocket_graph_kernel<FILL, true><<<grid_lig, PG_THREADS, smem, st>>>(
        c, p->xyz, p->rec_ptr, p->rr_ptr, p->rr_col, coords, complex_ptr, mask, mask_words,
        lig_count, ml, rec_of_pose, band, deg, n_inter, row_ptr, col, attr, edge_capacity,
        overflow);
    pocket_graph_kernel<FILL, false><<<grid, PG_THREADS, smem, st>>>(
        c, p->xyz, p->rec_ptr, p->rr_ptr, p->rr_col, coords, complex_ptr, mask, mask_words,
        lig_count, ml, rec_of_pose, band, deg, n_inter, row_ptr, col, attr, edge_capacity,
        overflow);
    return check_launch(2);
}

extern "C" {

int64_t pvs_pocket_cells_bytes(int32_t n_receptors, int32_t n_atoms) {
    if (n_receptors < 0 || n_atoms < 0) return -1;
    return cells_layout(nullptr, n_receptors, n_atoms, nullptr);
}

int64_t pvs_pocket_build_scratch_bytes(int32_t n_receptors, int32_t n_atoms) {
    if (n_receptors < 0 || n_atoms < 0) return -1;
    return build_scratch_layout(nullptr, n_receptors, n_atoms, nullptr, nullptr, nullptr);
}

int pvs_pocket_build_count(const pvs_pocket *pocket, void *scratch, void *stream) {
    int rc = pocket_check(pocket);
    if (rc) return rc;
    if (!pocket->rr_ptr || ((pocket->n_atoms > 0 || pocket->n_receptors > 0) && !scratch))
        return PVS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const pvs_pocket &p = *pocket;
    int32_t *rr_deg = nullptr;
    void *scan = nullptr;
    PocketCells c;
    cells_layout(p.cells, p.n_receptors, p.n_atoms, &c);
    build_scratch_layout(scratch, p.n_receptors, p.n_atoms, &c.cell_fill, &rr_deg, &scan);
    if (p.n_atoms > 0 && p.n_receptors > 0) {
        pocket_cells_kernel<<<p.n_receptors, PK_BUILD_THREADS, 0, st>>>(
            p.xyz, p.emit, p.rec_ptr, fmax(p.inter_radius, p.intra_radius), c);
        rc = check_launch();
        if (rc) return rc;
        if (p.max_atoms > 0) {
            dim3 grid(p.n_receptors, (p.max_atoms + PK_RR_THREADS - 1) / PK_RR_THREADS);
            pocket_rr_kernel<false><<<grid, PK_RR_THREADS, 0, st>>>(
                p.xyz, p.emit, p.rec_ptr, pair_band(p.inter_radius, p.intra_radius), c, rr_deg,
                nullptr);
            rc = check_launch();
            if (rc) return rc;
        }
    }
    return exclusive_scan(rr_deg, p.n_atoms, p.rr_ptr, scan, st);
}

int pvs_pocket_build_fill(const pvs_pocket *pocket, void *stream) {
    int rc = pocket_check(pocket);
    if (rc) return rc;
    if (pocket->n_atoms > 0 && !pocket->rr_col) return PVS_ERR_INVALID_ARG;
    const pvs_pocket &p = *pocket;
    if (p.n_atoms == 0 || p.n_receptors == 0 || p.max_atoms == 0) return PVS_OK;
    PocketCells c;
    cells_layout(p.cells, p.n_receptors, p.n_atoms, &c);
    dim3 grid(p.n_receptors, (p.max_atoms + PK_RR_THREADS - 1) / PK_RR_THREADS);
    pocket_rr_kernel<true><<<grid, PK_RR_THREADS, 0, (cudaStream_t)stream>>>(
        p.xyz, p.emit, p.rec_ptr, pair_band(p.inter_radius, p.intra_radius), c, p.rr_ptr,
        p.rr_col);
    return check_launch();
}

int pvs_pocket_compose(const pvs_pocket *const *parts, int32_t n_parts, const pvs_pocket *out,
                       void *stream) {
    int rc = pocket_check(out);
    if (rc) return rc;
    if (n_parts < 1 || !parts) return PVS_ERR_INVALID_ARG;
    int64_t n_rec = 0, n_atoms = 0;
    int max_atoms = 0;
    for (int k = 0; k < n_parts; ++k) {
        const pvs_pocket *q = parts[k];
        rc = pocket_check(q);
        if (rc) return rc;
        if (q->inter_radius != out->inter_radius || q->intra_radius != out->intra_radius)
            return PVS_ERR_INVALID_ARG;
        if (q->n_atoms > 0 && (!q->rr_col || !q->cells)) return PVS_ERR_INVALID_ARG;
        n_rec += q->n_receptors;
        n_atoms += q->n_atoms;
        max_atoms = std::max(max_atoms, (int)q->max_atoms);
    }
    if (n_rec != out->n_receptors || n_atoms != out->n_atoms || max_atoms != out->max_atoms)
        return PVS_ERR_INVALID_ARG;
    if (!out->rr_ptr || (out->n_atoms > 0 && (!out->rr_col || !out->cells)))
        return PVS_ERR_INVALID_ARG;
    if (!out->cells) return out->n_receptors > 0 ? PVS_ERR_INVALID_ARG : PVS_OK;
    PocketCells dst;
    cells_layout(out->cells, out->n_receptors, out->n_atoms, &dst);
    int r_off = 0, a_off = 0;
    for (int k = 0; k < n_parts; ++k) {
        const pvs_pocket *q = parts[k];
        PocketCells src;
        cells_layout(q->cells, q->n_receptors, q->n_atoms, &src);
        const int64_t work = std::max<int64_t>((int64_t)q->n_receptors * (PK_MAX_CELLS + 1),
                                               (int64_t)q->n_atoms * 8);
        const int grid = (int)std::min<int64_t>(std::max<int64_t>((work + 255) / 256, 1), 1024);
        pocket_compose_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
            src, q->rr_ptr, q->rr_col, q->n_receptors, q->n_atoms, dst, out->rr_ptr, out->rr_col,
            r_off, a_off, k == 0);
        rc = check_launch();
        if (rc) return rc;
        r_off += q->n_receptors;
        a_off += q->n_atoms;
    }
    return PVS_OK;
}

int pvs_pocket_graph_count(const pvs_pocket *pocket, const double *coords,
                           const int32_t *complex_ptr, int32_t n_poses, int32_t n_nodes,
                           const uint32_t *mask, int32_t mask_words, const int32_t *lig_count,
                           int32_t max_ligand_atoms, const int32_t *rec_of_pose,
                           double inter_radius, double intra_radius, int32_t *deg,
                           int32_t *n_inter, int32_t *row_ptr, void *scratch, void *stream) {
    int rc = pose_check(pocket, coords, complex_ptr, n_poses, n_nodes, mask, mask_words,
                        lig_count, max_ligand_atoms, inter_radius, intra_radius);
    if (rc) return rc;
    if (!row_ptr || (n_nodes > 0 && (!deg || !n_inter || !scratch))) return PVS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (n_nodes > 0 && n_poses > 0) {
        rc = pg_launch<false>(pocket, coords, complex_ptr, n_poses, mask, mask_words, lig_count,
                              max_ligand_atoms, rec_of_pose, inter_radius, intra_radius, deg,
                              n_inter, nullptr, 0, nullptr, nullptr, nullptr, st);
        if (rc) return rc;
    }
    return exclusive_scan(deg, n_nodes, row_ptr, scratch, st);
}

int pvs_pocket_graph_fill(const pvs_pocket *pocket, const double *coords,
                          const int32_t *complex_ptr, int32_t n_poses, int32_t n_nodes,
                          const uint32_t *mask, int32_t mask_words, const int32_t *lig_count,
                          int32_t max_ligand_atoms, const int32_t *rec_of_pose,
                          double inter_radius, double intra_radius, int32_t *row_ptr,
                          int32_t edge_capacity, int32_t *col, uint8_t *attr,
                          int32_t *overflow, void *stream) {
    int rc = pose_check(pocket, coords, complex_ptr, n_poses, n_nodes, mask, mask_words,
                        lig_count, max_ligand_atoms, inter_radius, intra_radius);
    if (rc) return rc;
    if (n_nodes == 0 || n_poses == 0) return PVS_OK;
    if (!row_ptr || !col || !attr || edge_capacity < 0) return PVS_ERR_INVALID_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    rc = pg_launch<true>(pocket, coords, complex_ptr, n_poses, mask, mask_words, lig_count,
                         max_ligand_atoms, rec_of_pose, inter_radius, intra_radius, nullptr,
                         nullptr, row_ptr, edge_capacity, col, attr, overflow, st);
    if (rc) return rc;
    return clamp_row_ptr(row_ptr, n_nodes, edge_capacity, st);
}

}  // extern "C"
