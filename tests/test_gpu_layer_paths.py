"""Two equivalences of the per-layer C ABI, bit for bit.

- pvs_egnn_layer_fwd issued as three staged calls (node_pre, edge, node) on
  one workspace gives what one call gives.
- pvs_egnn_layer_bwd reading P, Q and M from the forward's own workspace
  (saved_fwd_workspace) gives what its recompute gives: the forward and the
  backward must agree on where the workspace keeps them."""
import ctypes as C

import pytest
import torch

from tests import gpu_helpers as gh

pytestmark = pytest.mark.gpu

WIDTHS = {'fp32': (16, 32, 48, 64), 'bf16x3': (32, 64, 96, 128),
          'fp16x2': (32, 64, 96, 128), 'bf16': (32, 64, 96, 128)}
# layer options -> (EGNNLayer flags, caller asks for the edge messages)
OPTIONS = {
    'plain': (dict(update_coords=False), False),
    'graphnorm': (dict(graphnorm=True, update_coords=False), False),
    'softmax': (dict(edge_attention=True, softmax_attention=True), False),
    'softmax_m_out': (dict(edge_attention=True, softmax_attention=True), True),
    'node_attention': (dict(node_attention=True, update_coords=False), False),
    'edge_residual': (dict(edge_residual=True, edge_attention=True), True),
    'coords': (dict(update_coords=True, normalize=True, tanh=True), False),
}


@pytest.fixture(scope='module')
def graph():
    return gh.synthetic_graph(700, 3, 400, 25, ragged=True)


def _setup(graph, k, math, option, seed=0):
    from pointvs_b200 import EGNNLayer
    flags, want_m = OPTIONS[option]
    torch.manual_seed(seed)
    layer = EGNNLayer(k, k, k, edges_in_d=3, math=math, **flags).cuda()
    with torch.no_grad():
        for p in layer.parameters():    # GraphNorm's affine off its 1 / 0 init
            p.add_(0.05 * torch.randn_like(p))
        layer.coord_mlp[2].weight.mul_(1000.0)
    csr = graph.pvs_csr
    gen = torch.Generator().manual_seed(seed + 1)
    h = torch.randn(csr.n_nodes, k, generator=gen).cuda()
    m_prev = torch.randn(csr.n_edges, k, generator=gen).cuda() \
        if layer.edge_residual else None
    return layer, csr, h, graph.pos.contiguous(), m_prev, want_m


def _forward(layer, csr, h, x, m_prev, want_m, stage_calls):
    from pointvs_b200 import _cabi
    from pointvs_b200._cabi import check, ptr, stream
    lib = _cabi.lib()
    n, e, k = csr.n_nodes, csr.n_edges, layer.hidden_nf
    cfg = layer.c_config()
    pstruct = layer.c_params(layer.param_list())
    g = csr.c_struct()
    z = dict(dtype=torch.float32, device='cuda')
    out = {'h': torch.zeros(n, k, **z),
           'x': torch.zeros(n, 3, **z) if layer.use_coords else None,
           'm': torch.zeros(e, k, **z) if want_m else None,
           'att': torch.zeros(e, **z) if layer.edge_attention else None,
           'natt': torch.zeros(n, **z) if layer.node_attention else None}
    nbytes = int(lib.pvs_egnn_layer_workspace_bytes(n, e, C.byref(cfg)))
    ws = torch.zeros(nbytes, dtype=torch.uint8, device='cuda')
    for stages in stage_calls:
        cfg.stages = stages
        check(lib.pvs_egnn_layer_fwd(
            C.byref(g), C.byref(cfg), C.byref(pstruct), ptr(h), ptr(x), ptr(m_prev),
            ptr(out['h']), ptr(out['x']), ptr(out['m']), ptr(out['att']),
            ptr(out['natt']), ptr(ws), C.c_int64(nbytes), stream()), 'pvs_egnn_layer_fwd')
    torch.cuda.synchronize()
    return out, ws


CASES = [(math, k, option) for math, ks in WIDTHS.items() for k in ks for option in OPTIONS]


@pytest.mark.parametrize('math,k,option', CASES)
def test_staged_calls_equal_one_call(graph, math, k, option):
    layer, csr, h, x, m_prev, want_m = _setup(graph, k, math, option)
    whole, _ = _forward(layer, csr, h, x, m_prev, want_m, (0,))
    staged, _ = _forward(layer, csr, h, x, m_prev, want_m, (1, 2, 4))
    assert whole['h'].abs().sum() > 0
    for name, t in whole.items():
        if t is not None:
            assert torch.equal(t, staged[name]), name


def _backward(layer, csr, h, x, m_prev, saved_ws, seed=2):
    from pointvs_b200 import _cabi
    from pointvs_b200._cabi import check, ptr, stream
    lib = _cabi.lib()
    n, e, k = csr.n_nodes, csr.n_edges, layer.hidden_nf
    cfg = layer.c_config()
    cfg.saved_fwd_workspace = ptr(saved_ws)
    params = layer.param_list()
    pstruct = layer.c_params(params)
    grads = [None if p is None else torch.zeros_like(p) for p in params]
    gstruct = _cabi.LayerGrads(*[ptr(t) for t in grads])
    gen = torch.Generator().manual_seed(seed)
    d_h_out = torch.randn(n, k, generator=gen).cuda()
    d_x_out = torch.randn(n, 3, generator=gen).cuda() if layer.use_coords else None
    d_m_out = torch.randn(e, k, generator=gen).cuda() if layer.edge_residual else None
    d_h_in = torch.zeros(n, k, device='cuda')
    d_x_in = torch.zeros(n, 3, device='cuda')
    d_m_prev = torch.zeros(e, k, device='cuda') if m_prev is not None else None
    csc_ptr, csc_eid = csr.csc()
    g = csr.c_struct()
    nbytes = int(lib.pvs_egnn_layer_bwd_workspace_bytes(n, e, C.byref(cfg)))
    ws = torch.zeros(nbytes, dtype=torch.uint8, device='cuda')
    launches = lib.pvs_launch_count()
    check(lib.pvs_egnn_layer_bwd(
        C.byref(g), ptr(csc_ptr), ptr(csc_eid), C.byref(cfg), C.byref(pstruct), ptr(h),
        ptr(x), ptr(m_prev), ptr(d_h_out), ptr(d_x_out), ptr(d_m_out), ptr(d_h_in),
        ptr(d_x_in), ptr(d_m_prev), C.byref(gstruct), ptr(ws), C.c_int64(nbytes), stream()),
        'pvs_egnn_layer_bwd')
    torch.cuda.synchronize()
    launches = lib.pvs_launch_count() - launches
    outs = {'d_h_in': d_h_in, 'd_x_in': d_x_in, 'd_m_prev': d_m_prev}
    outs.update((name, t) for name, t in zip(_cabi.GRAD_FIELDS, grads))
    return outs, launches


# the backward reads the forward's workspace in the tensor-core modes at k <= 64
# without softmax attention or GraphNorm
SAVED_CASES = [(math, k, option) for math in ('bf16x3', 'fp16x2', 'bf16') for k in (32, 64)
               for option in ('plain', 'node_attention', 'edge_residual', 'coords')]


@pytest.mark.parametrize('math,k,option', SAVED_CASES)
def test_saved_forward_workspace_equals_recompute(graph, math, k, option):
    layer, csr, h, x, m_prev, want_m = _setup(graph, k, math, option)
    _, fwd_ws = _forward(layer, csr, h, x, m_prev, want_m, (0,))
    recomputed, n_recompute = _backward(layer, csr, h, x, m_prev, None)
    saved, n_saved = _backward(layer, csr, h, x, m_prev, fwd_ws)
    assert n_saved < n_recompute      # the node_pre and edge stages were skipped
    assert recomputed['d_h_in'].abs().sum() > 0
    for name, t in recomputed.items():
        if t is not None:
            assert torch.equal(t, saved[name]), name
