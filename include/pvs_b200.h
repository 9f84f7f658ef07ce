/*
 * pvs_b200.h -- C ABI of the B200-native PointVS EGNN hot path.
 *
 * The reference (jscant/PointVS) is pure Python/PyTorch and has no FFI of its
 * own; each entry point below names the reference function it replaces
 * (file:line under /root/reference).  The host-side mirror of the reference's
 * Python API (pointvs_b200/*.py) binds these with ctypes; INTEGRATION.md shows
 * the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns and allocates all outputs and workspaces;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as
 *     void*), never synchronises and keeps no mutable global state;
 *   - the return value is a pvs_status (0 = ok).  Argument errors are
 *     reported before anything is launched; launch errors come back as
 *     PVS_ERR_CUDA (pvs_last_cuda_error() has the cudaError_t);
 *   - feature matrices are row-major fp32; parameters are passed in the
 *     layout nn.Linear stores them ([out][in], row-major), so a PyTorch
 *     state_dict is usable without re-packing.
 */
#ifndef PVS_B200_H
#define PVS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PVS_VERSION 100 /* 0.1.0 */

typedef enum pvs_status {
    PVS_OK = 0,
    PVS_ERR_INVALID_ARG = 1,   /* null pointer, negative size, bad enum */
    PVS_ERR_UNSUPPORTED_K = 2, /* hidden width outside 1..PVS_MAX_K (forward in a
                                  tensor-core math mode: 1..PVS_MAX_K_TC_FWD) */
    PVS_ERR_TOO_LARGE = 3,     /* one complex does not fit the cell-list smem */
    PVS_ERR_CUDA = 4,          /* a CUDA call failed: pvs_last_cuda_error() */
    PVS_ERR_WORKSPACE = 5,     /* workspace smaller than *_workspace_bytes */
    PVS_ERR_UNSUPPORTED = 6    /* valid request the kernels do not cover yet */
} pvs_status;

#define PVS_MAX_K 64          /* widest hidden size (--channels) every path supports */
#define PVS_MAX_K_TC_FWD 128  /* widest hidden size of the forward in the tensor-core
                                 math modes (bf16x3 / fp16x2 / bf16); the backward,
                                 the stacked training calls and fp32 stop at PVS_MAX_K */
#define PVS_MAX_EDGE_CLASSES 8
#define PVS_TILE_EDGES 128    /* edges per work tile (one tcgen05 M=128 tile) */
#define PVS_TILE_NODES 128    /* node cap per work tile */

/* capability bits returned by pvs_capabilities() */
#define PVS_CAP_FWD_FP32 1u      /* FFMA forward                              */
#define PVS_CAP_FWD_TCGEN05 2u   /* tcgen05 edge-MLP tiles (bf16x3 / bf16)    */
#define PVS_CAP_BWD_FP32 4u      /* backward kernels                          */
#define PVS_CAP_FWD_FP16X2 8u    /* PVS_MATH_FP16X2 edge kernel               */
#define PVS_CAP_CROP 16u         /* K0: pvs_crop_count / pvs_crop_fill        */
#define PVS_CAP_FWD_WIDE_K 32u   /* forward at 65..PVS_MAX_K_TC_FWD (tcgen05)  */
#define PVS_CAP_POCKET 64u       /* K1p: pvs_pocket_build_* / pvs_pocket_graph_* */

/* pvs_layer_config.flags -- EGNNLayer.__init__ (egnn_satorras.py:26-46) */
#define PVS_F_RESIDUAL 0x001u
#define PVS_F_EDGE_RESIDUAL 0x002u
#define PVS_F_EDGE_ATTENTION 0x004u
#define PVS_F_NORMALIZE 0x008u
#define PVS_F_TANH 0x010u
#define PVS_F_GRAPHNORM 0x020u
#define PVS_F_UPDATE_COORDS 0x040u
#define PVS_F_PERM_INVARIANT 0x080u
#define PVS_F_NODE_ATTENTION 0x100u
#define PVS_F_GATED_RESIDUAL 0x200u
#define PVS_F_REZERO 0x400u
#define PVS_F_SOFTMAX_ATTENTION 0x800u

/* attention / head activations (egnn_satorras.py:66-73) */
typedef enum pvs_act {
    PVS_ACT_NONE = 0,
    PVS_ACT_SIGMOID = 1,
    PVS_ACT_TANH = 2,
    PVS_ACT_RELU = 3,
    PVS_ACT_SILU = 4,
    PVS_ACT_SOFTPLUS = 5
} pvs_act;

/* arithmetic used for the two per-edge 64x64 contractions */
typedef enum pvs_math {
    PVS_MATH_FP32 = 0,   /* FFMA, fp32 throughout                            */
    PVS_MATH_BF16X3 = 1, /* tcgen05, error-compensated bf16 split (fp32-class) */
    PVS_MATH_BF16 = 2,   /* tcgen05, single bf16 pass (fast mode)            */
    PVS_MATH_FP16X2 = 3  /* tcgen05, fp32-class: the per-edge GEMMs take the
                            activations as one fp16 tile and the weights as
                            fp16 hi + lo (A.Bhi + A.Blo); the per-node GEMMs
                            run as BF16X3.  Activations saturate at +-65504. */
} pvs_math;

/* Destination-sorted CSR of one packed batch plus its work-tile partition. */
typedef struct pvs_graph {
    int32_t n_nodes;
    int32_t n_edges;
    const int32_t *row_ptr;  /* [n_nodes+1] edges of node i (the RECEIVER,
                                edge_index[0]) are [row_ptr[i], row_ptr[i+1]) */
    const int32_t *col;      /* [n_edges] neighbour j (edge_index[1])         */
    const uint8_t *attr;     /* [n_edges] edge class (argmax of the one-hot
                                edge_attr) or NULL when edges_in_d == 0       */
    const int32_t *tile_ptr; /* [n_tiles+1] node boundaries of work tiles     */
    const int32_t *n_tiles;  /* device scalar written by pvs_build_tiles      */
    int32_t n_tiles_cap;     /* capacity of tile_ptr minus one                */
    /* Edge-packed tiles (pvs_build_packed_tiles), used by the tcgen05 edge
     * kernel (math != PVS_MATH_FP32): tile t owns edges [128 t, 128 t + 128),
     * ptile_last[t] = node that holds its last edge.  A node whose edges
     * cross a tile boundary is reduced through per-tile partial slots and a
     * fixed-order fix-up pass.  NULL: math = PVS_MATH_FP32 only.            */
    const int32_t *ptile_last; /* [n_ptiles_cap]                              */
    const int32_t *n_ptiles;   /* device scalar = max(1, ceil(E / 128))       */
    int32_t n_ptiles_cap;
} pvs_graph;

typedef struct pvs_layer_config {
    int32_t k;              /* hidden_nf == input_nf == output_nf            */
    int32_t n_edge_classes; /* edges_in_d (3 in every PointVS model, or 0)   */
    uint32_t flags;         /* PVS_F_*                                        */
    int32_t att_act;        /* pvs_act for att_mlp / node_att_mlp            */
    int32_t math;           /* pvs_math                                       */
    int32_t stages;         /* PVS_STAGE_* mask; 0 = all.  Lets a profiler put
                               events between the three launches of a layer;
                               the workspace carries state between calls.     */
    void *ev_edge_begin;    /* optional cudaEvent_t pair recorded on `stream`  */
    void *ev_edge_end;      /* around the edge stage (NULL = none): lets a     */
                            /* caller time the dominant kernel with no extra   */
                            /* host work inside a step                          */
    const void *saved_fwd_workspace; /* pvs_egnn_layer_bwd only (NULL = recompute):
                               the workspace pvs_egnn_layer_fwd was given for this
                               layer, same inputs, parameters and math, contents
                               untouched since.  The backward then reads P, Q and
                               M from it instead of re-running the node_pre and
                               edge stages (tensor-core modes without softmax
                               attention / GraphNorm; ignored otherwise).       */
} pvs_layer_config;

#define PVS_STAGE_NODE_PRE 1 /* P = h W1a^T + b1, Q = h W1b^T                 */
#define PVS_STAGE_EDGE 2     /* edge MLP, attention, coordinate + message reduce */
#define PVS_STAGE_NODE 4     /* node MLP, node attention, residual            */
#define PVS_STAGE_ALL 7

/* Parameters of one EGNNLayer in state_dict layout (egnn_satorras.py:76-121).
 * Unused blocks are NULL. */
typedef struct pvs_layer_params {
    const float *edge_w1;  /* edge_mlp.0.weight [k][in_e], in_e =
                              (perm_invariant ? k : 2k) + 1 + n_edge_classes */
    const float *edge_b1;  /* edge_mlp.0.bias   [k]     */
    const float *edge_w2;  /* edge_mlp.2.weight [k][k]  */
    const float *edge_b2;  /* edge_mlp.2.bias   [k]     */
    const float *coord_w1; /* coord_mlp.0.weight [k][k] */
    const float *coord_b1; /* coord_mlp.0.bias   [k]    */
    const float *coord_w2; /* coord_mlp.2.weight [1][k] (no bias) */
    const float *att_w;    /* att_mlp.0.weight   [1][k] */
    const float *att_b;    /* att_mlp.0.bias     [1]    */
    const float *node_w1;  /* node_mlp.0.weight  [k][2k] */
    const float *node_b1;  /* node_mlp.0.bias    [k]    */
    const float *gn_weight;     /* node_mlp.1.weight     [k] (GraphNorm)     */
    const float *gn_bias;       /* node_mlp.1.bias       [k]                 */
    const float *gn_mean_scale; /* node_mlp.1.mean_scale [k]                 */
    const float *node_w2;  /* node_mlp.3.weight  [k][k] */
    const float *node_b2;  /* node_mlp.3.bias    [k]    */
    const float *natt_w;   /* node_att_mlp.0.weight [1][k] */
    const float *natt_b;   /* node_att_mlp.0.bias   [1]    */
    const float *edge_gate; /* edge_gate_parameter [1] */
    const float *node_gate; /* node_gate_parameter [1] */
} pvs_layer_params;

/* Gradients of pvs_layer_params: same members, same shapes, accumulated into
 * (+=); NULL members are skipped. */
typedef struct pvs_layer_grads {
    float *edge_w1, *edge_b1, *edge_w2, *edge_b2;
    float *coord_w1, *coord_b1, *coord_w2;
    float *att_w, *att_b;
    float *node_w1, *node_b1;
    float *gn_weight, *gn_bias, *gn_mean_scale;
    float *node_w2, *node_b2;
    float *natt_w, *natt_b;
    float *edge_gate, *node_gate;
} pvs_layer_grads;

int pvs_version(void);
uint32_t pvs_capabilities(void);
const char *pvs_status_string(int status);
int pvs_last_cuda_error(void);
/* kernels launched by this library (all host threads) since load */
int64_t pvs_launch_count(void);

/* ---- K1: radius graph --------------------------------------------------
 * Replaces generate_edges (point_vs/preprocessing/preprocessing.py:68-155)
 * for a packed batch of complexes.  Per-complex cell list; fp64 distances
 * sqrt((dx*dx+dy*dy)+dz*dz) without FMA contraction, tests d < radius and
 * d > 1e-7 exactly as :108-121.  Output is the destination-sorted CSR of
 * the reference edge list: within a row, the inter-molecular edges in
 * ascending col, then the intra list in ascending col (the stable sort by
 * row of the reference's [inter | intra] output).
 *
 * Two passes so the caller can size col/attr:
 *   count: deg[N] = edges per node, n_inter[N] = of which inter edges,
 *          row_ptr[N+1] = exclusive scan of deg (row_ptr[N] = total edges).
 *          If mask_scratch != NULL (pvs_radius_graph_mask_bytes) the per-node
 *          neighbour bit masks are kept there and `fill` only expands them
 *          (no second neighbour search).
 *   fill:  col / attr, and optionally ref_pos[E] = index of each CSR edge in
 *          the reference's (PyG-collated) edge order.  edge_capacity = size of
 *          col/attr in edges: a caller that wants NO host sync between the
 *          passes allocates an upper bound instead of reading row_ptr[N];
 *          edges beyond the capacity are dropped, *overflow (device int,
 *          may be NULL) is set non-zero and row_ptr is cut at the capacity
 *          so that no consumer of the CSR indexes past col/attr.
 * coords: fp64 [N][3]; bp: int32 [N] (0 ligand, 1 receptor; :106);
 * complex_ptr: int32 [B+1] node offsets.  scratch: pvs_scan_scratch_bytes(N). */
int64_t pvs_radius_graph_mask_bytes(int32_t n_nodes, int32_t max_complex_nodes);
int pvs_radius_graph_count(const double *coords, const int32_t *bp,
                           const int32_t *complex_ptr, int32_t n_complexes,
                           int32_t n_nodes, int32_t max_complex_nodes,
                           double inter_radius, double intra_radius,
                           int32_t *deg, int32_t *n_inter, int32_t *row_ptr,
                           uint32_t *mask_scratch, void *scratch, void *stream);
int pvs_radius_graph_fill(const double *coords, const int32_t *bp,
                          const int32_t *complex_ptr, int32_t n_complexes,
                          int32_t n_nodes, int32_t max_complex_nodes,
                          double inter_radius, double intra_radius,
                          const int32_t *n_inter, int32_t *row_ptr,
                          const uint32_t *mask_scratch, int32_t edge_capacity,
                          int32_t *col, uint8_t *attr, int32_t *ref_pos,
                          int32_t *overflow, void *stream);
/* Connected-component mask for `prune` (preprocessing.py:144-153): keep[i]=1
 * iff node i is reachable from the row of its complex's first inter edge
 * (or every node of a complex that has no inter edge). */
int pvs_prune_mask(const int32_t *row_ptr, const int32_t *col,
                   const int32_t *n_inter, const int32_t *complex_ptr,
                   int32_t n_complexes, int32_t n_nodes, uint8_t *keep,
                   void *stream);

/* ---- K0: receptor crop + atom typing in front of K1 (row N2) ---------------
 * Replaces: make_box(relative_to_ligand=True) + the hydrogen filter + atom
 *           typing + make_bit_vector of PointCloudDataset.parquets_to_inputs
 *           (preprocessing/data_loaders.py:259-309, preprocessing.py:165-239)
 *           for a batch of poses whose receptors are resident on the device.
 * lig_xyz fp64 [L][3], lig_emit u8 [L] (0 = atom only takes part in the box
 * test, e.g. a filtered hydrogen), lig_ptr int32 [B+1]; rec_xyz / rec_emit
 * likewise for the concatenated receptors, rec_ptr int32 [R+1], rec_of_pose
 * int32 [B] (NULL = receptor 0 for every pose).  mask: B * mask_words uint32
 * keep-bits, mask_words >= ceil(largest receptor / 32).  counts[b] = atoms of
 * complex b (emitted ligand atoms + kept receptor atoms); the caller scans
 * them into complex_ptr (pvs_exclusive_scan) and calls pvs_crop_fill, which
 * writes each complex as [ligand atoms; kept receptor atoms] in file order:
 * coords fp64 [N][3], bp int32 [N] (0/1), feats fp32 [N][F] with F =
 * n_atom_types + 1 (compact) or 2 * n_atom_types.  *_code int16: the atom
 * `types` value the reference would one-hot (receptor codes already shifted
 * by n_atom_types). */
int pvs_crop_count(const double *lig_xyz, const uint8_t *lig_emit,
                   const int32_t *lig_ptr, int32_t n_poses,
                   const double *rec_xyz, const uint8_t *rec_emit,
                   const int32_t *rec_ptr, const int32_t *rec_of_pose,
                   int32_t mask_words, double radius, uint32_t *mask,
                   int32_t *counts, void *stream);
int pvs_crop_fill(const double *lig_xyz, const uint8_t *lig_emit,
                  const int16_t *lig_code, const int32_t *lig_ptr,
                  int32_t n_poses, const double *rec_xyz,
                  const int16_t *rec_code, const int32_t *rec_ptr,
                  const int32_t *rec_of_pose, const uint32_t *mask,
                  int32_t mask_words, const int32_t *complex_ptr,
                  int32_t n_atom_types, int32_t compact, double *coords,
                  int32_t *bp, float *feats, void *stream);

/* ---- K1p: radius graph of ligand poses against resident receptors ----------
 * Replaces: generate_edges (preprocessing/preprocessing.py:68-155) for the
 *           complexes K0 assembles (data_loaders.py:259-309) when many poses
 *           share a receptor.  The receptor-receptor part of every such graph
 *           is the same, so it is searched once per pocket; per batch only
 *           ligand-ligand and ligand-receptor pairs are tested.
 * Output: exactly pvs_radius_graph_count / _fill's (deg, n_inter, row_ptr,
 * col, attr, edge_capacity / overflow semantics) on the same K0 complexes,
 * byte for byte: the same fp64 pair test, the same within-row order.
 *
 * A pocket is the receptors in K0's form (xyz fp64 [A][3], emit u8 [A],
 * rec_ptr int32 [R+1]; they stay resident and K0 reads the same arrays)
 * plus, in caller-allocated device memory:
 *   cells  pvs_pocket_cells_bytes(R, A) bytes (about 128 KB per receptor
 *          plus 28 B per atom): a cell list of each receptor's emitted
 *          atoms (cell edge >= max radius, at most PVS_POCKET_MAX_DIM cells
 *          per axis, larger cells beyond);
 *   rr_ptr int32 [A+1], rr_col int32 [rr_ptr[A]]: CSR of the receptor-
 *          receptor pairs within intra_radius over emitted atoms, rows in
 *          concatenated atom order, columns the atom's index inside its own
 *          receptor, ascending (file order).
 * Build, once per pocket: pvs_pocket_build_count (cell list, rr_ptr; scratch
 * pvs_pocket_build_scratch_bytes(R, A), free after the call), a host read
 * of rr_ptr[A] to size rr_col, then pvs_pocket_build_fill.  A receptor of
 * more than PVS_POCKET_MAX_REC_ATOMS atoms returns PVS_ERR_TOO_LARGE.
 *
 * Per batch, after K0 (pvs_crop_count / pvs_crop_fill):
 *   coords, complex_ptr: K0's assembled complexes; mask / mask_words: K0's
 *   keep bits (mask_words * 32 >= pocket->max_atoms); lig_count int32 [B]:
 *   emitted ligand atoms of each pose, all <= max_ligand_atoms <=
 *   PVS_POCKET_MAX_LIG_ATOMS (above: PVS_ERR_TOO_LARGE; a pose whose count
 *   exceeds max_ligand_atoms gets no edges, and the fill sets *overflow to
 *   2); rec_of_pose int32 [B] or NULL.
 *   The radii must be the pocket's own (else PVS_ERR_INVALID_ARG).
 *   scratch: pvs_scan_scratch_bytes(n_nodes) (no more: the receptor rows of
 *   a pose walk only its kept atoms, located from the keep bits in shared
 *   memory, on as many CTAs as its kept count needs).
 *
 * Compose: pvs_pocket_compose fills `out`, a pocket of the receptors of
 * parts[0], parts[1], ... in that order, from those built pockets by device
 * copies, without searching any receptor again.  The caller gives `out` its
 * concatenated xyz / emit / rec_ptr, sizes (n_receptors, n_atoms, max_atoms:
 * the sums and the largest), the parts' radii, and cells, rr_ptr and rr_col
 * sized for it (rr_col: the sum of the parts' rr_ptr[n_atoms]). */
#define PVS_POCKET_MAX_LIG_ATOMS 256    /* emitted ligand atoms per pose      */
#define PVS_POCKET_MAX_REC_ATOMS 65536  /* atoms per receptor                 */
#define PVS_POCKET_MAX_DIM 32           /* cells per axis of a receptor grid  */

typedef struct pvs_pocket {
    int32_t n_receptors;
    int32_t n_atoms;        /* rec_ptr[n_receptors] */
    int32_t max_atoms;      /* atoms of the largest receptor */
    double inter_radius;    /* the radii the pocket is built for */
    double intra_radius;
    const double *xyz;      /* [n_atoms][3] */
    const uint8_t *emit;    /* [n_atoms] */
    const int32_t *rec_ptr; /* [n_receptors + 1] */
    void *cells;            /* pvs_pocket_cells_bytes(n_receptors, n_atoms) */
    int32_t *rr_ptr;        /* [n_atoms + 1] */
    int32_t *rr_col;        /* [rr_ptr[n_atoms]] (build_fill and per batch) */
} pvs_pocket;

int64_t pvs_pocket_cells_bytes(int32_t n_receptors, int32_t n_atoms);
int64_t pvs_pocket_build_scratch_bytes(int32_t n_receptors, int32_t n_atoms);
int pvs_pocket_build_count(const pvs_pocket *pocket, void *scratch, void *stream);
int pvs_pocket_build_fill(const pvs_pocket *pocket, void *stream);
int pvs_pocket_compose(const pvs_pocket *const *parts, int32_t n_parts,
                       const pvs_pocket *out, void *stream);
int pvs_pocket_graph_count(const pvs_pocket *pocket, const double *coords,
                           const int32_t *complex_ptr, int32_t n_poses,
                           int32_t n_nodes, const uint32_t *mask,
                           int32_t mask_words, const int32_t *lig_count,
                           int32_t max_ligand_atoms,
                           const int32_t *rec_of_pose, double inter_radius,
                           double intra_radius, int32_t *deg, int32_t *n_inter,
                           int32_t *row_ptr, void *scratch, void *stream);
int pvs_pocket_graph_fill(const pvs_pocket *pocket, const double *coords,
                          const int32_t *complex_ptr, int32_t n_poses,
                          int32_t n_nodes, const uint32_t *mask,
                          int32_t mask_words, const int32_t *lig_count,
                          int32_t max_ligand_atoms, const int32_t *rec_of_pose,
                          double inter_radius, double intra_radius,
                          int32_t *row_ptr, int32_t edge_capacity,
                          int32_t *col, uint8_t *attr, int32_t *overflow,
                          void *stream);

int64_t pvs_scan_scratch_bytes(int32_t n);
/* row_ptr[0..n] = exclusive scan of deg[0..n-1] */
int pvs_exclusive_scan(const int32_t *deg, int32_t n, int32_t *row_ptr,
                       void *scratch, void *stream);

/* Greedy partition of the node range into work tiles: consecutive nodes
 * whose edges total <= PVS_TILE_EDGES (a node with more edges gets a tile of
 * its own) and at most PVS_TILE_NODES nodes.  tile_ptr needs
 * pvs_tiles_capacity(n_nodes, n_edges)+1 ints; scratch the same amount of
 * ints again + pvs_scan_scratch_bytes of that. */
int32_t pvs_tiles_capacity(int32_t n_nodes, int32_t n_edges);
int64_t pvs_tiles_scratch_bytes(int32_t n_nodes);
int pvs_build_tiles(const int32_t *row_ptr, int32_t n_nodes, int32_t *tile_ptr,
                    int32_t *n_tiles, void *scratch, void *stream);

/* Edge-packed tile partition (see pvs_graph).  ptile_last needs
 * pvs_packed_tiles_capacity(n_edges) ints; n_edges may be an upper bound (a
 * capacity-bounded CSR): the true count is read from row_ptr[n_nodes]. */
int32_t pvs_packed_tiles_capacity(int32_t n_edges);
int pvs_build_packed_tiles(const int32_t *row_ptr, int32_t n_nodes,
                           int32_t n_edges, int32_t *ptile_last,
                           int32_t *n_ptiles, void *stream);

/* Arbitrary-order edge_index (PyG [2][E] int64, edge_attr one-hot int64
 * [E][n_classes] or NULL) -> destination-sorted CSR, stable in the caller's
 * order.  perm[p] = caller's edge index stored at CSR slot p.  For callers
 * that bring their own graph (attribution, reference data loaders;
 * pnn_geometric_base.py:55-58).  bad_index (device int) is set non-zero if
 * any index is outside [0, n_nodes).  scratch: n_nodes ints +
 * pvs_scan_scratch_bytes(n_nodes). */
int pvs_edge_index_to_csr(const int64_t *edge_index, int64_t n_edges,
                          const int64_t *edge_attr_onehot, int32_t n_classes,
                          int32_t n_nodes, int32_t *deg, int32_t *row_ptr,
                          int32_t *col, uint8_t *attr, int32_t *perm,
                          int32_t *bad_index, void *scratch, void *stream);

/* batch [N] int64 non-decreasing -> graph_ptr [B+1]
 * (pnn_geometric_base.py:27 derives B = max(batch)+1) */
int pvs_batch_to_ptr(const int64_t *batch, int32_t n_nodes, int32_t n_graphs,
                     int32_t *graph_ptr, void *stream);

/* ---- dense helpers ------------------------------------------------------
 * out[r][0..ko) = act(in[r][0..ki) . W[ko][ki]^T + b).  Embedding
 * (PygLinearPass, pnn_geometric_base.py:83-94), heads
 * (egnn_satorras.py:304-317, egnn_multitask.py:141-146).  ki, ko <= 128. */
int pvs_linear_fwd(const float *in, int32_t ld_in, int32_t rows, int32_t ki,
                   const float *w, int32_t ld_w, const float *b, int32_t ko,
                   int32_t act, float *out, int32_t ld_out, void *stream);
/* Backward of pvs_linear_fwd (recomputes the pre-activation):
 *   g = d_out * act'(in.W^T + b);  d_in = g . W;  d_w += g^T . in;
 *   d_b += column sums of g.  d_in / d_w / d_b may be NULL.  ko <= 64. */
int64_t pvs_linear_bwd_workspace_bytes(int32_t rows, int32_t ki, int32_t ko);
int pvs_linear_bwd(const float *in, int32_t ld_in, int32_t rows, int32_t ki,
                   const float *w, int32_t ld_w, const float *b, int32_t ko,
                   int32_t act, const float *d_out, int32_t ld_dout,
                   float *d_in, int32_t ld_din, float *d_w, int32_t ld_dw,
                   float *d_b, void *workspace, int64_t workspace_bytes,
                   void *stream);

/* global_mean_pool (pnn_geometric_base.py:29-33): pooled[b] = mean of h rows
 * [graph_ptr[b], graph_ptr[b+1]) (0 for an empty graph). */
int pvs_mean_pool_fwd(const float *h, const int32_t *graph_ptr,
                      int32_t n_graphs, int32_t k, float *pooled, void *stream);

int pvs_mean_pool_bwd(const float *d_pooled, const int32_t *graph_ptr,
                      int32_t n_graphs, int32_t k, float *d_h, void *stream);

/* ---- K2: one EGNN layer, forward ----------------------------------------
 * Replaces EGNNLayer.forward (egnn_satorras.py:189-206 and :123-187).
 *   h_in [N][k], x_in [N][3] -> h_out [N][k], x_out [N][3] (x_out may not
 *   alias x_in; the Python wrapper copies back to keep the reference's
 *   in-place `coord += agg`, :174).
 *   m_prev [E][k] (CSR order) or NULL: previous layer's messages, read only
 *   with PVS_F_EDGE_RESIDUAL.  m_out [E][k], att_out [E], natt_out [N] are
 *   optional outputs (NULL to skip) in CSR order.
 * workspace: pvs_egnn_layer_workspace_bytes(). */
int64_t pvs_egnn_layer_workspace_bytes(int32_t n_nodes, int32_t n_edges,
                                       const pvs_layer_config *cfg);
int pvs_egnn_layer_fwd(const pvs_graph *graph, const pvs_layer_config *cfg,
                       const pvs_layer_params *params, const float *h_in,
                       const float *x_in, const float *m_prev, float *h_out,
                       float *x_out, float *m_out, float *att_out,
                       float *natt_out, void *workspace,
                       int64_t workspace_bytes, void *stream);

/* ---- whole-model scoring pass ----------------------------------------------
 * SartorrasEGNN.forward / MultitaskSatorrasEGNN.forward
 * (pnn_geometric_base.py:24-41, egnn_multitask.py:150-166) in ONE call:
 * embedding Linear -> n_layers x pvs_egnn_layer_fwd -> mean pool -> head
 * (up to 3 Linear layers with fused activations).  Same kernels and the same
 * results as issuing the per-layer calls; it exists so that a scoring step
 * costs one host call instead of ~40 (the Python launch path was the
 * bottleneck at ~4 ms of GPU work per step).  No side channels, no autograd.
 *   feats [N][dim_input] (pitch ld_feats), x_in [N][3], graph_ptr [B+1].
 *   scores [B][head[n_head-1].ko]; x_out [N][3] (final coordinates, may be
 *   NULL or == x_in for the reference's in-place update); h_out [N][k] or NULL. */
typedef struct pvs_head_layer {
    const float *w;   /* [ko][ki] */
    const float *b;   /* [ko] or NULL */
    int32_t ki, ko;
    int32_t act;      /* pvs_act applied after this Linear */
} pvs_head_layer;

typedef struct pvs_model_desc {
    int32_t n_layers, k, dim_input, n_head;
    const float *embed_w;                  /* layers.0.m.weight [k][dim_input] */
    const float *embed_b;                  /* layers.0.m.bias   [k]            */
    const pvs_layer_config *layer_cfg;     /* [n_layers] */
    const pvs_layer_params *layer_params;  /* [n_layers] */
    const pvs_head_layer *head;            /* [n_head], n_head <= 3 */
} pvs_model_desc;

int64_t pvs_egnn_model_workspace_bytes(int32_t n_nodes, int32_t n_edges,
                                       int32_t n_graphs,
                                       const pvs_model_desc *model);
int pvs_egnn_model_fwd(const pvs_graph *graph, const pvs_model_desc *model,
                       const float *feats, int32_t ld_feats, const float *x_in,
                       const int32_t *graph_ptr, int32_t n_graphs,
                       float *scores, float *x_out, float *h_out,
                       void *workspace, int64_t workspace_bytes, void *stream);

/* ---- K3: one EGNN layer, backward ---------------------------------------
 * Autograd of pvs_egnn_layer_fwd (SURVEY.md 9.2; PyTorch autograd of
 * egnn_satorras.py:123-206 in the reference).  Recomputes the layer from
 * (h_in, x_in, m_prev) instead of saving per-edge activations.
 *   csc_ptr/csc_eid: the same edges grouped by neighbour (pvs_csr_transpose):
 *   the scatter over `col` becomes a second atomics-free segment reduce.
 *   d_h_out [N][k], d_x_out [N][3] (NULL = zero), d_m_out [E][k] (NULL =
 *   zero): gradients of the layer outputs, CSR order.
 *   d_h_in [N][k], d_x_in [N][3] are overwritten; d_m_prev [E][k] is
 *   overwritten when the layer has an edge residual and m_prev != NULL.
 *   Parameter gradients are ACCUMULATED into `grads` (NULL members skipped).
 * GraphNorm (batch-wide statistics) and softmax attention are differentiated
 * too. */
int pvs_csr_transpose(const pvs_graph *graph, int32_t *csc_ptr,
                      int32_t *csc_eid, void *scratch, void *stream);
/* Same grouping for a SYMMETRIC graph (every radius graph of K1: i-j is an
 * edge iff j-i is): the edges arriving at node j are the reverses of row j,
 * so csc_ptr == row_ptr and csc_eid[p] = position of j in the row of col[p]
 * (of its r-th occurrence for the r-th occurrence of col[p] in row j: a pair
 * within both cut-offs is listed twice); one pass, no counting sort.  *asymmetric (device, may be NULL) is set to 1
 * if some edge has no reverse (the entry then refers to the edge itself). */
int pvs_csr_transpose_symmetric(const pvs_graph *graph, int32_t *csc_eid,
                                int32_t *asymmetric, void *stream);
int64_t pvs_egnn_layer_bwd_workspace_bytes(int32_t n_nodes, int32_t n_edges,
                                           const pvs_layer_config *cfg);
int pvs_egnn_layer_bwd(const pvs_graph *graph, const int32_t *csc_ptr,
                       const int32_t *csc_eid, const pvs_layer_config *cfg,
                       const pvs_layer_params *params, const float *h_in,
                       const float *x_in, const float *m_prev,
                       const float *d_h_out, const float *d_x_out,
                       const float *d_m_out, float *d_h_in, float *d_x_in,
                       float *d_m_prev, const pvs_layer_grads *grads,
                       void *workspace, int64_t workspace_bytes, void *stream);

/* ---- Training through the whole stack of EGNN layers: one call each way ----
 * The layer loop of get_embeddings (egnn_satorras.py:319-329) and its autograd,
 * issued from C so that a training step costs two library calls instead of two
 * per layer (for hosts slower than the ~350 kernel launches of a step; on the
 * B200 box the per-layer calls are as fast).  Layers without edge residual
 * only; no side channels.
 *   H [L+1][N][k]: H[0] = input features (caller), H[l+1] = output of layer l.
 *   X [L+1][N][3]: likewise for the coordinates (copied through a layer that
 *   does not update them).
 *   layer_ws: L slices of pvs_egnn_stack_layer_ws_stride() bytes, one forward
 *   workspace per layer, KEPT until the backward (its P, Q, M are reused).
 * pvs_egnn_stack_bwd walks the layers in reverse through pvs_egnn_layer_bwd:
 * d_h_out / d_x_out are the gradients of H[L] / X[L] (d_x_out NULL = the final
 * coordinates are not consumed), d_h_in / d_x_in those of H[0] / X[0];
 * parameter gradients are accumulated into grads[l]. */
int64_t pvs_egnn_stack_layer_ws_stride(int32_t n_nodes, int32_t n_edges,
                                       int32_t n_layers,
                                       const pvs_layer_config *cfgs);
int pvs_egnn_stack_fwd(const pvs_graph *graph, int32_t n_layers,
                       const pvs_layer_config *cfgs,
                       const pvs_layer_params *params, float *H, float *X,
                       void *layer_ws, int64_t layer_ws_stride, void *stream);
int64_t pvs_egnn_stack_bwd_workspace_bytes(int32_t n_nodes, int32_t n_edges,
                                           int32_t n_layers,
                                           const pvs_layer_config *cfgs);
int pvs_egnn_stack_bwd(const pvs_graph *graph, const int32_t *csc_ptr,
                       const int32_t *csc_eid, int32_t n_layers,
                       const pvs_layer_config *cfgs,
                       const pvs_layer_params *params,
                       const pvs_layer_grads *grads, const float *H,
                       const float *X, const void *layer_ws,
                       int64_t layer_ws_stride, const float *d_h_out,
                       const float *d_x_out, float *d_h_in, float *d_x_in,
                       void *workspace, int64_t workspace_bytes, void *stream);


#ifdef __cplusplus
}
#endif
#endif /* PVS_B200_H */
