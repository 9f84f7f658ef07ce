// Whole-model scoring pass: one C call per step (pvs_egnn_model_fwd).
// Composition only -- every kernel is launched through the same code paths as
// the per-layer entry points.
#include <cstdlib>

#include "egnn_common.cuh"
#include "egnn_bwd_common.cuh"

using namespace pvs;

namespace {

struct ModelWs {
    float *h[2], *x[2], *m[2], *pooled, *head_tmp[2];
    void *layer_ws;
    int64_t layer_ws_bytes;
    int64_t bytes;
};

bool any_edge_residual(const pvs_model_desc *md) {
    for (int l = 0; l < md->n_layers; ++l)
        if (md->layer_cfg[l].flags & PVS_F_EDGE_RESIDUAL) return true;
    return false;
}

ModelWs carve_model(void *base, int n, int e, int b, const pvs_model_desc *md) {
    ModelWs w{};
    char *p = (char *)base;
    auto take = [&](int64_t bytes) {
        void *r = p;
        p += align_up(bytes, 256);
        return r;
    };
    const int k = md->k;
    for (int i = 0; i < 2; ++i) w.h[i] = (float *)take((int64_t)n * k * 4);
    for (int i = 0; i < 2; ++i) w.x[i] = (float *)take((int64_t)n * 3 * 4);
    if (any_edge_residual(md))
        for (int i = 0; i < 2; ++i) w.m[i] = (float *)take((int64_t)e * k * 4);
    w.pooled = (float *)take((int64_t)b * k * 4);
    for (int i = 0; i < 2; ++i) w.head_tmp[i] = (float *)take((int64_t)b * 128 * 4);
    int64_t lw = 0;
    for (int l = 0; l < md->n_layers; ++l) {
        int64_t v = pvs_egnn_layer_workspace_bytes(n, e, &md->layer_cfg[l]);
        if (v > lw) lw = v;
    }
    w.layer_ws_bytes = lw;
    w.layer_ws = take(lw);
    w.bytes = p - (char *)base;
    return w;
}

int check_desc(const pvs_model_desc *md) {
    if (!md || md->n_layers < 0 || md->n_head < 1 || md->n_head > 3) return PVS_ERR_INVALID_ARG;
    if (md->k < 1 || md->k > PVS_MAX_K_TC_FWD) return PVS_ERR_UNSUPPORTED_K;
    if (md->dim_input < 1 || md->dim_input > 128) return PVS_ERR_INVALID_ARG;
    if (!md->embed_w || !md->head || (md->n_layers > 0 && (!md->layer_cfg || !md->layer_params)))
        return PVS_ERR_INVALID_ARG;
    for (int l = 0; l < md->n_layers; ++l) {
        if (md->layer_cfg[l].k != md->k) return PVS_ERR_INVALID_ARG;
        if (md->k > PVS_MAX_K && md->layer_cfg[l].math == PVS_MATH_FP32)
            return PVS_ERR_UNSUPPORTED_K;   // 65..128 runs on the tensor cores only
    }
    for (int i = 0; i < md->n_head; ++i) {
        const pvs_head_layer &hl = md->head[i];
        if (!hl.w || hl.ki < 1 || hl.ki > 128 || hl.ko < 1 || hl.ko > 128) return PVS_ERR_INVALID_ARG;
    }
    if (md->head[0].ki != md->k) return PVS_ERR_INVALID_ARG;
    return PVS_OK;
}

}  // namespace

extern "C" {

int64_t pvs_egnn_model_workspace_bytes(int32_t n_nodes, int32_t n_edges, int32_t n_graphs,
                                       const pvs_model_desc *md) {
    if (check_desc(md) != PVS_OK || n_nodes < 0 || n_edges < 0 || n_graphs < 0) return -1;
    return carve_model(nullptr, n_nodes, n_edges, n_graphs, md).bytes + 256;
}

int pvs_egnn_model_fwd(const pvs_graph *g, const pvs_model_desc *md, const float *feats,
                       int32_t ld_feats, const float *x_in, const int32_t *graph_ptr,
                       int32_t n_graphs, float *scores, float *x_out, float *h_out,
                       void *workspace, int64_t workspace_bytes, void *stream) {
    int rc = check_desc(md);
    if (rc) return rc;
    if (!g || g->n_nodes < 0 || g->n_edges < 0 || n_graphs < 0) return PVS_ERR_INVALID_ARG;
    if (g->n_nodes == 0 || n_graphs == 0) return PVS_OK;
    if (!feats || !x_in || !graph_ptr || !scores || !workspace || ld_feats < md->dim_input)
        return PVS_ERR_INVALID_ARG;
    if (workspace_bytes < pvs_egnn_model_workspace_bytes(g->n_nodes, g->n_edges, n_graphs, md))
        return PVS_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int n = g->n_nodes, k = md->k;
    ModelWs w = carve_model((void *)align_up((int64_t)(uintptr_t)workspace, 256), n, g->n_edges,
                            n_graphs, md);
    // embedding (PygLinearPass)
    rc = launch_linear(feats, ld_feats, n, md->dim_input, md->embed_w, md->dim_input,
                       md->embed_b, k, PVS_ACT_NONE, w.h[0], k, st);
    if (rc) return rc;
    const float *h_cur = w.h[0];
    const float *x_cur = x_in;
    const float *m_cur = nullptr;
    int hb = 0, xb = 0, mb = 0;
    // from here to the end of the layer loop the tcgen05 kernels are launched
    // with programmatic stream serialization: each one's prologue runs under
    // the tail of the one before (pvs_common.cuh).  Every kernel of the chain
    // waits for its predecessor before touching its data, and none of them
    // writes what a prologue reads (weights, graph structure).
    ChainScope chain_scope;
    for (int l = 0; l < md->n_layers; ++l) {
        const pvs_layer_config &cfg = md->layer_cfg[l];
        const bool coords = cfg.flags & PVS_F_UPDATE_COORDS;
        const bool next_eres = l + 1 < md->n_layers &&
                               (md->layer_cfg[l + 1].flags & PVS_F_EDGE_RESIDUAL);
        float *h_next = w.h[hb ^ 1];
        float *x_next = coords ? w.x[xb] : nullptr;
        float *m_next = next_eres ? w.m[mb] : nullptr;
        rc = pvs_egnn_layer_fwd(g, &cfg, &md->layer_params[l], h_cur, x_cur,
                                (cfg.flags & PVS_F_EDGE_RESIDUAL) ? m_cur : nullptr, h_next,
                                x_next, m_next, nullptr, nullptr, w.layer_ws, w.layer_ws_bytes,
                                stream);
        if (rc) return rc;
        h_cur = h_next; hb ^= 1;
        if (coords) { x_cur = x_next; xb ^= 1; }
        m_cur = m_next;
        if (next_eres) mb ^= 1;
    }
    if (h_out) {
        rc = cuda_call(cudaMemcpyAsync(h_out, h_cur, (size_t)n * k * 4, cudaMemcpyDeviceToDevice, st));
        if (rc) return rc;
    }
    if (x_out && x_out != x_cur) {
        rc = cuda_call(cudaMemcpyAsync(x_out, x_cur, (size_t)n * 3 * 4, cudaMemcpyDeviceToDevice, st));
        if (rc) return rc;
    }
    rc = pvs_mean_pool_fwd(h_cur, graph_ptr, n_graphs, k, w.pooled, stream);
    if (rc) return rc;
    const float *in = w.pooled;
    for (int i = 0; i < md->n_head; ++i) {
        const pvs_head_layer &hl = md->head[i];
        float *out = (i == md->n_head - 1) ? scores : w.head_tmp[i & 1];
        rc = launch_linear(in, hl.ki, n_graphs, hl.ki, hl.w, hl.ki, hl.b, hl.ko, hl.act, out,
                           hl.ko, st);
        if (rc) return rc;
        in = out;
    }
    return PVS_OK;
}


/* ---- training through the whole stack of EGNN layers, one call each way ---- */

static int64_t stack_layer_ws_stride(int32_t n_nodes, int32_t n_edges, int32_t n_layers,
                                     const pvs_layer_config *cfgs) {
    int64_t lw = 0;
    for (int l = 0; l < n_layers; ++l) {
        const int64_t v = pvs_egnn_layer_workspace_bytes(n_nodes, n_edges, &cfgs[l]);
        if (v < 0) return -1;
        if (v > lw) lw = v;
    }
    return align_up(lw, 256);
}

int64_t pvs_egnn_stack_layer_ws_stride(int32_t n_nodes, int32_t n_edges, int32_t n_layers,
                                       const pvs_layer_config *cfgs) {
    if (!cfgs || n_layers < 1 || n_nodes < 0 || n_edges < 0) return -1;
    return stack_layer_ws_stride(n_nodes, n_edges, n_layers, cfgs);
}

int pvs_egnn_stack_fwd(const pvs_graph *g, int32_t n_layers, const pvs_layer_config *cfgs,
                       const pvs_layer_params *params, float *H, float *X, void *layer_ws,
                       int64_t layer_ws_stride, void *stream) {
    if (!g || !cfgs || !params || !H || !X || !layer_ws || n_layers < 1)
        return PVS_ERR_INVALID_ARG;
    const int n = g->n_nodes;
    if (n <= 0) return PVS_OK;
    const int k = cfgs[0].k;
    if (k > PVS_MAX_K) return PVS_ERR_UNSUPPORTED_K;   // training path: 64 wide
    if (layer_ws_stride < stack_layer_ws_stride(n, g->n_edges, n_layers, cfgs))
        return PVS_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    ChainScope chain_scope;      // as in pvs_egnn_model_fwd
    for (int l = 0; l < n_layers; ++l) {
        if (cfgs[l].k != k) return PVS_ERR_INVALID_ARG;
        if (cfgs[l].flags & PVS_F_EDGE_RESIDUAL) return PVS_ERR_INVALID_ARG;   // per-layer path
        const bool coords = cfgs[l].flags & PVS_F_UPDATE_COORDS;
        const float *h_in = H + (size_t)l * n * k;
        float *h_out = H + (size_t)(l + 1) * n * k;
        const float *x_in = X + (size_t)l * n * 3;
        float *x_out = X + (size_t)(l + 1) * n * 3;
        int rc = pvs_egnn_layer_fwd(g, &cfgs[l], &params[l], h_in, x_in, nullptr, h_out,
                                    coords ? x_out : nullptr, nullptr, nullptr, nullptr,
                                    (char *)layer_ws + (size_t)l * layer_ws_stride,
                                    layer_ws_stride, stream);
        if (rc) return rc;
        if (!coords) {
            rc = cuda_call(cudaMemcpyAsync(x_out, x_in, (size_t)n * 3 * 4,
                                           cudaMemcpyDeviceToDevice, st));
            if (rc) return rc;
        }
    }
    return PVS_OK;
}

int64_t pvs_egnn_stack_bwd_workspace_bytes(int32_t n_nodes, int32_t n_edges, int32_t n_layers,
                                           const pvs_layer_config *cfgs) {
    if (!cfgs || n_layers < 1 || n_nodes < 0 || n_edges < 0) return -1;
    int64_t lw = 0;
    for (int l = 0; l < n_layers; ++l) {
        const int64_t v = pvs_egnn_layer_bwd_workspace_bytes(n_nodes, n_edges, &cfgs[l]);
        if (v < 0) return -1;
        if (v > lw) lw = v;
    }
    const int k = cfgs[0].k;
    // two layer workspaces: layer l's gradient reductions still read theirs on
    // the side stream while layer l - 1 runs in the other one
    return 2 * align_up(lw, 256) + 2 * align_up((int64_t)n_nodes * k * 4, 256) +
           2 * align_up((int64_t)n_nodes * 3 * 4, 256) + 256;
}

int pvs_egnn_stack_bwd(const pvs_graph *g, const int32_t *csc_ptr, const int32_t *csc_eid,
                       int32_t n_layers, const pvs_layer_config *cfgs,
                       const pvs_layer_params *params, const pvs_layer_grads *grads,
                       const float *H, const float *X, const void *layer_ws,
                       int64_t layer_ws_stride, const float *d_h_out, const float *d_x_out,
                       float *d_h_in, float *d_x_in, void *workspace, int64_t workspace_bytes,
                       void *stream) {
    if (!g || !cfgs || !params || !grads || !H || !X || !d_h_out || !d_h_in || !d_x_in ||
        !workspace || n_layers < 1)
        return PVS_ERR_INVALID_ARG;
    for (int l = 0; l < n_layers; ++l)
        if (cfgs[l].k < 1 || cfgs[l].k > PVS_MAX_K) return PVS_ERR_UNSUPPORTED_K;
    const int n = g->n_nodes;
    if (n <= 0) return PVS_OK;
    if (workspace_bytes < pvs_egnn_stack_bwd_workspace_bytes(n, g->n_edges, n_layers, cfgs))
        return PVS_ERR_WORKSPACE;
    const int k = cfgs[0].k;
    char *p = (char *)align_up((int64_t)(uintptr_t)workspace, 256);
    float *dh[2], *dx[2];
    for (int i = 0; i < 2; ++i) { dh[i] = (float *)p; p += align_up((int64_t)n * k * 4, 256); }
    for (int i = 0; i < 2; ++i) { dx[i] = (float *)p; p += align_up((int64_t)n * 3 * 4, 256); }
    const int64_t lws_bytes = ((workspace_bytes - (p - (char *)workspace)) / 2) & ~(int64_t)255;
    void *lws[2] = {p, p + lws_bytes};
    cudaStream_t st = (cudaStream_t)stream;
    // Side stream for the reductions into the parameter gradients (per-CTA
    // partials of the edge kernel, the grouped weight gradients): nothing later
    // in the backward reads them, so they run beside the next layer's node and
    // edge kernels.  Each layer uses the workspace the layer before the
    // previous one has finished with (ev_done), and everything is joined to the
    // caller's stream at the end.  PVS_NO_BWD_SIDE=1 keeps one stream.
    static const bool no_side = getenv("PVS_NO_BWD_SIDE") != nullptr;
    struct SideRes {
        BwdSide s{};
        cudaEvent_t ev_done[2]{};
        bool ok = false;
        SideRes() {
            ok = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) == cudaSuccess &&
                 cudaEventCreateWithFlags(&s.ev_a, cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&s.ev_b, cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&ev_done[0], cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&ev_done[1], cudaEventDisableTiming) == cudaSuccess;
        }
    };
    static thread_local SideRes *res[16] = {};      // per device of this host thread
    SideRes *sr = nullptr;
    int dev = 0;
    if (!no_side && n_layers > 1 && cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 16) {
        if (!res[dev]) res[dev] = new SideRes();
        if (res[dev]->ok) sr = res[dev];
    }
    bool pending[2] = {false, false};
    const float *dh_cur = d_h_out, *dx_cur = d_x_out;
    int rc = PVS_OK;
    for (int l = n_layers - 1; l >= 0 && rc == PVS_OK; --l) {
        pvs_layer_config cfg = cfgs[l];
        if (layer_ws != nullptr)
            cfg.saved_fwd_workspace = (const char *)layer_ws + (size_t)l * layer_ws_stride;
        float *dh_next = l == 0 ? d_h_in : dh[l & 1];
        float *dx_next = l == 0 ? d_x_in : dx[l & 1];
        const int par = l & 1;
        if (sr && pending[par]) {        // the reductions that read this workspace
            cudaStreamWaitEvent(st, sr->ev_done[par], 0);
            pending[par] = false;
        }
        g_bwd_side = sr ? &sr->s : nullptr;
        rc = pvs_egnn_layer_bwd(g, csc_ptr, csc_eid, &cfg, &params[l],
                                H + (size_t)l * n * k, X + (size_t)l * n * 3, nullptr,
                                dh_cur, dx_cur, nullptr, dh_next, dx_next, nullptr,
                                &grads[l], lws[sr ? par : 0], lws_bytes, stream);
        g_bwd_side = nullptr;
        if (sr) {
            cudaEventRecord(sr->ev_done[par], sr->s.stream);
            pending[par] = true;
        }
        dh_cur = dh_next;
        dx_cur = dx_next;
    }
    if (sr)
        for (int par = 0; par < 2; ++par)
            if (pending[par]) cudaStreamWaitEvent(st, sr->ev_done[par], 0);
    return rc;
}

}  // extern "C"
