// Pieces of K1 shared with K1p (pocket.cu): block scans, the cell coordinate
// and the pair predicate.  Both graph builders must decide every pair the same
// way, so the predicate lives here once.
#pragma once
#include "pvs_common.cuh"

namespace pvs {

// exclusive scan of one value per thread across the block; returns prefix,
// writes the block total to *total (all threads see it after the call).
__device__ inline int block_scan_excl(int v, int *total, int *warp_buf) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarps = (blockDim.x + 31) >> 5;
    int incl = warp_scan_incl(v, lane);
    if (lane == 31) warp_buf[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = lane < nwarps ? warp_buf[lane] : 0;
        int wi = warp_scan_incl(w, lane);
        warp_buf[lane] = wi - w;
        if (lane == 31) warp_buf[32] = wi;
    }
    __syncthreads();
    int prefix = warp_buf[warp] + incl - v;
    *total = warp_buf[32];
    __syncthreads();
    return prefix;
}

// in-place exclusive scan of an array of any length (shared or global memory)
__device__ inline int smem_scan_excl(int *data, int n, int *warp_buf) {
    const int T = blockDim.x;
    const int per = (n + T - 1) / T;
    const int lo = min(n, (int)threadIdx.x * per), hi = min(n, lo + per);
    int s = 0;
    for (int i = lo; i < hi; ++i) s += data[i];
    int total;
    int prefix = block_scan_excl(s, &total, warp_buf);
    for (int i = lo; i < hi; ++i) {
        int v = data[i];
        data[i] = prefix;
        prefix += v;
    }
    __syncthreads();
    return total;
}

// cell index along one axis; `inv` = 1 / cell edge.  Monotone in v, and the same
// expression bins the atoms and locates the query, so neighbours within r_max
// (< cell edge / (1 + 1e-6)) are never more than one cell apart.
__device__ __forceinline__ int cell_coord(double v, double lo, double inv, int dim) {
    int c = (int)floor(__dmul_rn(__dsub_rn(v, lo), inv));
    return max(0, min(dim - 1, c));
}

// The two cut-offs with the +-1e-15 relative band around r^2 inside which the
// rounded sqrt decides (see pair_test).
struct PairBand {
    double r_inter, r_intra;
    double inter_lo, inter_hi, intra_lo, intra_hi, pos_hi;
};

__host__ __device__ __forceinline__ PairBand pair_band(double r_inter, double r_intra) {
    PairBand b;
    b.r_inter = r_inter;
    b.r_intra = r_intra;
    b.inter_lo = r_inter * r_inter * (1.0 - 1e-15);
    b.inter_hi = r_inter * r_inter * (1.0 + 1e-15);
    b.intra_lo = r_intra * r_intra * (1.0 - 1e-15);
    b.intra_hi = r_intra * r_intra * (1.0 + 1e-15);
    b.pos_hi = 1e-14 * (1.0 + 1e-15);
    return b;
}

// The distance test of generate_edges (preprocessing.py:108-121) for the pair
// (i, j): pos = d > 1e-7, in_inter = d < r_inter, in_intra = d < r_intra with
// d the scipy cdist value sqrt((dx*dx + dy*dy) + dz*dz), no FMA contraction.
// Swapping i and j negates dx, dy, dz exactly, so the test is symmetric.
__device__ __forceinline__ void pair_test(const PairBand &b, double xi, double yi, double zi,
                                          double xj, double yj, double zj, bool &pos,
                                          bool &in_inter, bool &in_intra) {
    const double ddx = __dsub_rn(xi, xj);
    const double ddy = __dsub_rn(yi, yj);
    const double ddz = __dsub_rn(zi, zj);
    const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy)),
                                __dmul_rn(ddz, ddz));
    // The reference compares the ROUNDED sqrt with the radius.  Outside a
    // +-1e-15 relative band around r^2 the outcome is decided by d2 alone
    // (sqrt is monotone and correctly rounded); only inside the band is the
    // sqrt evaluated.
    if (d2 > b.pos_hi && (d2 < b.inter_lo || d2 > b.inter_hi) &&
        (d2 < b.intra_lo || d2 > b.intra_hi)) {
        pos = true;
        in_inter = d2 < b.inter_lo;
        in_intra = d2 < b.intra_lo;
    } else {
        const double d = __dsqrt_rn(d2);
        pos = d > 1e-7;
        in_inter = d < b.r_inter;
        in_intra = d < b.r_intra;
    }
}

// graph.cu: row_ptr[0..n] = exclusive scan of deg (2-3 launches), and the cut
// of row_ptr at the edge capacity after a capacity-bounded fill (1 launch)
int exclusive_scan(const int32_t *deg, int n, int32_t *row_ptr, void *scratch,
                   cudaStream_t st);
int clamp_row_ptr(int32_t *row_ptr, int n_nodes, int cap, cudaStream_t st);

}  // namespace pvs
