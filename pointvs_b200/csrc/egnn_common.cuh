// Argument block shared by the FFMA and tcgen05 edge kernels.
#pragma once
#include "pvs_common.cuh"

namespace pvs {

constexpr int TE = PVS_TILE_EDGES;
constexpr int TN = PVS_TILE_NODES;

struct EdgeArgs {
    // graph
    const int32_t *row_ptr, *col, *tile_ptr, *n_tiles;
    const uint8_t *attr;
    // edge-packed tiles (tcgen05 kernel only): see pvs_graph
    const int32_t *ptile_last, *n_ptiles;
    int n_nodes;
    float *Mpart;            // [n_ptiles_cap][2][KP] partial message sums of split nodes
    float *xpart;            // [n_ptiles_cap][2][4]  partial coordinate sums
    // activations
    const float *P, *Q;      // [N][KP], KP = 64 (k <= 64 in the tcgen05 modes) or 128
    const float *x_in;       // [N][3]
    const float *m_prev;     // [E][k] or null
    float *M;                // [N][KP]
    float *x_out;            // [N][3] or null
    float *m_out;            // [E][ld_m] or null
    int ld_m;
    float *att_out;          // [E] or null (softmax mode: raw logits)
    // params
    const float *edge_w1, *edge_w2, *edge_b2, *coord_w1, *coord_b1, *coord_w2;
    const float *att_w, *att_b, *edge_gate;
    int k, in_e, n_classes;
    uint32_t flags;
    int att_act;
};

// columns of edge_mlp.0.weight: h_i and h_j (perm-invariant: h_i alone), the
// squared distance and the one-hot edge class
inline int edge_in_width(const pvs_layer_config *cfg) {
    const int k = cfg->k;
    return ((cfg->flags & PVS_F_PERM_INVARIANT) ? k : 2 * k) + 1 + cfg->n_edge_classes;
}

// launches the tcgen05 edge kernel (egnn_edge_tc.cu); mode = pvs_math
int launch_edge_tc(const EdgeArgs &a, int n_ptiles_cap, int mode, cudaStream_t st);
// bf16x3 variant with 8-warp groups and the segment-reduce on the tensor core
// (egnn_edge_tc8.cu); launch_edge_tc dispatches to it when PVS_EDGE_TC8 says so
int launch_edge_tc8(const EdgeArgs &a, int n_ptiles_cap, cudaStream_t st);
// out = act(in . W^T + b) (w_in_major: out = in . W); accumulate: out += ...
int launch_linear(const float *in, int ld_in, int rows, int ki, const float *w,
                  int ld_w, const float *b, int ko, int act, float *out,
                  int ld_out, cudaStream_t st, int w_in_major = 0,
                  int accumulate = 0);
int persistent_grid(int work_items, int blocks_per_sm);

// per-layer forward workspace (egnn_fwd.cu)
struct FwdWorkspace {
    float *P, *Q, *M, *V, *m_ws, *z_ws, *gn_partial, *gn_shift, *gn_a, *gn_b;
    float *gn_mean, *gn_invstd;
    float *Mpart, *xpart;    // split-node partials of the edge-packed tiles
    int kp;                  // pitch of P, Q, M, V and m_ws
    int64_t bytes;
};
int64_t fwd_recompute_bytes(int n, int e, uint32_t flags);
int fwd_recompute(const pvs_graph *g, const pvs_layer_config *cfg, const pvs_layer_params *p,
                  const float *h_in, const float *x_in, const float *m_prev, void *ws_base,
                  FwdWorkspace *out, cudaStream_t st);
// P, Q, M of a layer as pvs_egnn_layer_fwd left them in its workspace
FwdWorkspace fwd_saved(const void *saved_workspace, int n, int e, const pvs_layer_config *cfg);
// tensor-core node stages (egnn_node_tc.cu); mode = PVS_MATH_BF16X3 / BF16
// K3: d_h[N][k] += dP[N][64] . W1a + dQ[N][64] . W1b on tcgen05 (bf16x3)
int launch_dgrad_pq_tc(const float *dP, const float *dQ, const float *edge_w1, float *d_h,
                       int n_nodes, int k, int in_e, cudaStream_t st);
int launch_node_pre_tc(const float *h, const float *edge_w1, const float *edge_b1, float *P,
                       float *Q, int n_nodes, int k, int in_e, int perm, int mode,
                       cudaStream_t st);
int launch_node_tc(const float *h_in, const float *M, float *h_out, float *natt_out,
                   const pvs_layer_params *p, int n_nodes, int k, uint32_t flags, int att_act,
                   int mode, cudaStream_t st, int phase = 0, float *V = nullptr,
                   const float *gn_a = nullptr, const float *gn_b = nullptr);
// the same two stages at 65 <= k <= 128 (egnn_wide_tc.cu): P, Q, M, V at pitch
// 128; launch_node_pre_tc / launch_node_tc dispatch to them when k > 64
int launch_wide_node_pre_tc(const float *h, const float *edge_w1, const float *edge_b1, float *P,
                            float *Q, int n_nodes, int k, int in_e, int perm, int mode,
                            cudaStream_t st);
int launch_wide_node_tc(const float *h_in, const float *M, float *h_out, float *natt_out,
                        const pvs_layer_params *p, int n_nodes, int k, uint32_t flags,
                        int att_act, int mode, cudaStream_t st, int phase, float *V,
                        const float *gn_a, const float *gn_b);

}  // namespace pvs
