"""Host-side mirror of the reference's EGNN model API, running on the CUDA
C-ABI (include/pvs_b200.h).

Same class names, constructor/`build_net`/`forward`/`get_embeddings`
signatures, state_dict keys and side channels as
/root/reference/point_vs/models/geometric/{egnn_satorras,egnn_multitask,
pnn_geometric_base}.py, so checkpoints and callers carry over unchanged.  The
nn.Modules below only HOLD parameters (in the reference's layout and init
order); all arithmetic happens in the kernels.  There is no PyTorch fallback:
without the built library, or on CPU tensors, forward raises.
"""
import ctypes as C
import os

import torch
from torch import nn

from . import _cabi
from ._cabi import check, lib, ptr, stream
from .base import PointNeuralNetworkBase, DEVICE
from .graph import CSRGraph, csr_from_edge_index, dropout_adj


class GraphNorm(nn.Module):
    """Parameter holder with PyG GraphNorm's state_dict keys
    (node_mlp.1.{weight,bias,mean_scale}); applied inside the node kernel."""

    def __init__(self, in_channels, eps=1e-5):
        super().__init__()
        self.in_channels, self.eps = in_channels, eps
        self.weight = nn.Parameter(torch.ones(in_channels))
        self.bias = nn.Parameter(torch.zeros(in_channels))
        self.mean_scale = nn.Parameter(torch.ones(in_channels))


_ATT_MODULES = {'sigmoid': nn.Sigmoid, 'tanh': nn.Tanh, 'relu': nn.ReLU,
                'silu': nn.SiLU}

# (data_ptr, shape, version) of the last edge_index seen -> its CSR.  The
# reference passes the same `edges` tensor to every layer
# (egnn_satorras.py:325-328); one sort serves the whole stack.
_CSR_CACHE = {}


def _csr_for(edge_index, edge_attr, n_nodes):
    key = (edge_index.data_ptr(), tuple(edge_index.shape), edge_index._version,
           None if edge_attr is None else
           (edge_attr.data_ptr(), edge_attr._version), n_nodes,
           str(edge_index.device))
    hit = _CSR_CACHE.get(key)
    if hit is not None:
        return hit
    if len(_CSR_CACHE) > 8:
        _CSR_CACHE.clear()
    g = csr_from_edge_index(edge_index, edge_attr, n_nodes)
    if int(g._bad.item()):
        raise IndexError('edge_index holds node ids outside [0, n_nodes)')
    # hold the tensors so the cache key (a raw address) stays valid
    g._key_refs = (edge_index, edge_attr)
    _CSR_CACHE[key] = g
    return g


# Optional profiler hook: an object with begin(stage)/end(stage) that records
# CUDA events around each stage of a layer (see bench.py).  None = one call.
STAGE_TIMER = None


def _width_error(k, fp32):
    """Why the library refused hidden width k."""
    if _cabi.MAX_K < k <= _cabi.MAX_K_TC_FWD and fp32:
        return (f'hidden width k={k}: hidden width 65..128 needs a tensor-core '
                "math mode (set_math('bf16x3'), 'fp16x2' or 'bf16')")
    return (f'unsupported hidden width k={k} (1..{_cabi.MAX_K}; '
            f'{_cabi.MAX_K + 1}..{_cabi.MAX_K_TC_FWD} for scoring in a '
            'tensor-core math mode)')


def _workspace(layer_cfg, n_nodes, n_edges, device):
    nbytes = int(lib().pvs_egnn_layer_workspace_bytes(
        n_nodes, n_edges, C.byref(layer_cfg)))
    if nbytes < 0:
        raise _cabi.PvsError(_width_error(
            layer_cfg.k, layer_cfg.math == _cabi.MATH['fp32']))
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


class _EGNNLayerFn(torch.autograd.Function):
    """One fused EGNN layer.  forward -> pvs_egnn_layer_fwd; backward ->
    pvs_egnn_layer_bwd (recomputes the layer from the saved inputs)."""

    @staticmethod
    def forward(ctx, layer, csr, want_m, want_side, h, x, m_prev, *params):
        # outputs nobody consumes (the last layer's coordinates) reach
        # backward as None, so their parameters get no gradient -- as under
        # the reference's autograd
        ctx.set_materialize_grads(False)
        cfg = layer.c_config()
        n, e, k = csr.n_nodes, csr.n_edges, layer.hidden_nf
        dev = h.device
        h = h.contiguous()
        x = x.contiguous()
        m_prev = None if m_prev is None else m_prev.contiguous()
        pstruct = layer.c_params(params)
        h_out = torch.empty_like(h)
        x_out = torch.empty_like(x) if layer.use_coords else None
        m_out = torch.empty((e, k), dtype=torch.float32, device=dev) \
            if want_m else None
        att = torch.empty((e,), dtype=torch.float32, device=dev) \
            if (want_side and layer.edge_attention) else None
        natt = torch.empty((n,), dtype=torch.float32, device=dev) \
            if (want_side and layer.node_attention) else None
        ws = _workspace(cfg, n, e, dev)
        tc = layer.math != 'fp32'
        g = csr.c_struct(node_tiles=not tc, packed_tiles=tc)
        timer = STAGE_TIMER
        split = timer is not None and getattr(timer, 'split_stages', True)
        if timer is not None and not split:
            # pre-created CUDA events recorded by the library around the edge
            # stage: no extra host work inside the step
            cfg.ev_edge_begin, cfg.ev_edge_end = timer.next_edge_events()
        with torch.cuda.device(dev):
            # a splitting stage timer (bench.py, outside the headline timing)
            # issues the three stages as separate calls with events between
            for stages in ((1, 2, 4) if split else (0,)):
                cfg.stages = stages
                if split:
                    timer.begin(stages)
                check(lib().pvs_egnn_layer_fwd(
                    C.byref(g), C.byref(cfg), C.byref(pstruct), ptr(h), ptr(x),
                    ptr(m_prev), ptr(h_out), ptr(x_out), ptr(m_out), ptr(att),
                    ptr(natt), ptr(ws), C.c_int64(ws.numel()), stream()),
                    'pvs_egnn_layer_fwd')
                if split:
                    timer.end(stages)
        ctx.layer, ctx.csr = layer, csr
        # training: keep this layer's workspace (P, Q, M: 768 B per node) so
        # the backward need not re-run the node_pre and edge stages
        ctx.fwd_ws = ws if (any(ctx.needs_input_grad) and not split) else None
        ctx.fwd_math = layer.math
        ctx.save_for_backward(h, x, m_prev, *params)
        ctx.mark_non_differentiable(*[t for t in (att, natt) if t is not None])
        if x_out is None:
            x_out = x
        return h_out, x_out, m_out, att, natt

    @staticmethod
    def backward(ctx, d_h, d_x, d_m, _d_att, _d_natt):
        from .backward import egnn_layer_backward
        return egnn_layer_backward(ctx, d_h, d_x, d_m)


class _EGNNStackFn(torch.autograd.Function):
    """All EGNN layers of a model in ONE library call each way
    (pvs_egnn_stack_fwd / pvs_egnn_stack_bwd): the training counterpart of the
    fused scoring pass.  Used by get_embeddings when gradients are wanted and
    no layer needs edge messages or side channels, and PVS_STACK_TRAIN=1."""

    @staticmethod
    def forward(ctx, layers, csr, h, x, *params):
        ctx.set_materialize_grads(False)
        L = len(layers)
        n, e, k = csr.n_nodes, csr.n_edges, layers[0].hidden_nf
        dev = h.device
        cfgs = (_cabi.LayerConfig * L)()
        pstructs = (_cabi.LayerParams * L)()
        per = len(_cabi.PARAM_FIELDS)
        keep = []
        for i, layer in enumerate(layers):
            cfgs[i] = layer.c_config()
            ps = params[i * per:(i + 1) * per]
            det = [None if p is None else p.detach().contiguous() for p in ps]
            keep.append(det)
            pstructs[i] = _cabi.LayerParams(*[ptr(p) for p in det])
        H = torch.empty((L + 1, n, k), dtype=torch.float32, device=dev)
        X = torch.empty((L + 1, n, 3), dtype=torch.float32, device=dev)
        H[0].copy_(h)
        X[0].copy_(x)
        stride = int(lib().pvs_egnn_stack_layer_ws_stride(n, e, L, cfgs))
        if stride < 0:
            raise _cabi.PvsError('unsupported layer configuration for the '
                                 'stacked training pass')
        ws = torch.empty(max(1, L * stride), dtype=torch.uint8, device=dev)
        tc = layers[0].math != 'fp32'
        g = csr.c_struct(node_tiles=True, packed_tiles=tc)
        with torch.cuda.device(dev):
            check(lib().pvs_egnn_stack_fwd(
                C.byref(g), L, cfgs, pstructs, ptr(H), ptr(X), ptr(ws),
                C.c_int64(stride), stream()), 'pvs_egnn_stack_fwd')
        ctx.layers, ctx.csr, ctx.stride = layers, csr, stride
        ctx.H, ctx.X, ctx.ws = H, X, ws
        ctx.math = layers[0].math
        ctx.save_for_backward(*[p for p in params if p is not None])
        ctx.param_mask = [p is not None for p in params]
        return H[L], X[L]

    @staticmethod
    def backward(ctx, d_h, d_x):
        from . import backward as _bw
        return _bw.egnn_stack_backward(ctx, d_h, d_x)


class _StackPlan:
    """Everything the lean training pass needs again on every step while the
    layers' parameters stay where they are: the struct arrays of
    pvs_egnn_stack_fwd / _bwd, and (per gradient arena) the gradient pointer
    block.  Cached on the model, keyed on the parameters' storage addresses."""

    def __init__(self, layers):
        self.layers = tuple(layers)
        L = len(self.layers)
        self.params = [p for layer in self.layers for p in layer.param_list()]
        self.key = self.make_key(self.params, self.layers)
        self.cfgs = (_cabi.LayerConfig * L)()
        self.pstructs = (_cabi.LayerParams * L)()
        for i, layer in enumerate(self.layers):
            self.cfgs[i] = layer.c_config()
            self.pstructs[i] = layer.c_params(layer.param_list())
        self.anchor = next((p for p in self.params
                            if p is not None and p.requires_grad), None)
        self.grad_plans = {}

    @staticmethod
    def make_key(params, layers):
        return (tuple(0 if p is None else p.data_ptr() for p in params),
                tuple(p is not None and p.requires_grad for p in params),
                tuple((l.math, l.c_flags()) for l in layers))

    @classmethod
    def of(cls, model, layers):
        plan = model.__dict__.get('_stack_plan')
        if plan is not None and len(plan.layers) == len(layers) and all(
                a is b for a, b in zip(plan.layers, layers)):
            # the Parameter objects of a module survive `.to()` / state-dict
            # loads (only their storage moves), so the cached list is checked
            # instead of walking the modules again
            if cls.make_key(plan.params, layers) == plan.key:
                return plan
        plan = cls(layers)
        model.__dict__['_stack_plan'] = plan
        return plan


class _EGNNStackLeanFn(torch.autograd.Function):
    """The stacked training pass for models trained through `backprop()`:
    only h and x (and one anchor parameter, so that the outputs require
    grad) are autograd inputs.  Parameter gradients never travel through
    autograd: the backward kernels write them into the model's gradient arena
    (parallel.GradArena), or -- outside `backprop()` -- they are accumulated
    into `p.grad` by hand, as AccumulateGrad would.  Host time per step: two
    library calls instead of sixteen Functions with 27 inputs each."""

    @staticmethod
    def forward(ctx, plan, csr, h, x, _anchor):
        ctx.set_materialize_grads(False)
        layers = plan.layers
        L = len(layers)
        n, e, k = csr.n_nodes, csr.n_edges, layers[0].hidden_nf
        dev = h.device
        H = torch.empty((L + 1, n, k), dtype=torch.float32, device=dev)
        X = torch.empty((L + 1, n, 3), dtype=torch.float32, device=dev)
        H[0].copy_(h)
        X[0].copy_(x)
        stride = int(lib().pvs_egnn_stack_layer_ws_stride(n, e, L, plan.cfgs))
        if stride < 0:
            raise _cabi.PvsError('unsupported layer configuration for the '
                                 'stacked training pass')
        ws = torch.empty(max(1, L * stride), dtype=torch.uint8, device=dev)
        tc = layers[0].math != 'fp32'
        g = csr.c_struct(node_tiles=True, packed_tiles=tc)
        with torch.cuda.device(dev):
            check(lib().pvs_egnn_stack_fwd(
                C.byref(g), L, plan.cfgs, plan.pstructs, ptr(H), ptr(X), ptr(ws),
                C.c_int64(stride), stream()), 'pvs_egnn_stack_fwd')
        ctx.plan, ctx.csr, ctx.stride = plan, csr, stride
        ctx.H, ctx.X, ctx.ws = H, X, ws
        return H[L], X[L]

    @staticmethod
    def backward(ctx, d_h, d_x):
        from . import backward as _bw
        return _bw.egnn_stack_backward_lean(ctx, d_h, d_x)


class EGNNLayer(nn.Module):
    """Mirror of EGNNLayer (egnn_satorras.py:23-206)."""
    # pylint: disable = R, W, C

    def __init__(self, input_nf, output_nf, hidden_nf, edges_in_d=0,
                 act_fn=nn.SiLU(), residual=True, edge_residual=False,
                 edge_attention=False, normalize=False, tanh=False,
                 graphnorm=False, update_coords=True,
                 permutation_invariance=False, node_attention=False,
                 attention_activation_fn='sigmoid', gated_residual=False,
                 rezero=False, softmax_attention=False, math='fp32'):
        assert not (gated_residual and rezero), \
            'gated_residual and rezero are incompatible'
        super().__init__()
        if not (input_nf == output_nf == hidden_nf):
            raise NotImplementedError(
                'the fused kernels need input_nf == hidden_nf == output_nf '
                '(every PointVS model builds EGNNLayer(k, k, k))')
        if not isinstance(act_fn, nn.SiLU):
            raise NotImplementedError(
                'EGNN activation is SiLU in every PointVS model '
                '(--activation never reaches EGNN)')
        input_edge = input_nf if permutation_invariance else input_nf * 2
        self.gated_residual, self.rezero = gated_residual, rezero
        self.residual, self.edge_residual = residual, edge_residual
        self.edge_attention, self.normalize, self.tanh = \
            edge_attention, normalize, tanh
        self.epsilon = 1e-8
        self.use_coords = update_coords
        self.permutation_invariance = permutation_invariance
        self.node_attention = node_attention
        self.hidden_nf = hidden_nf
        self.edges_in_d = edges_in_d
        self.graphnorm = graphnorm
        self.attention_activation_fn = attention_activation_fn
        attention_activation = _ATT_MODULES[attention_activation_fn] \
            if not softmax_attention else nn.Identity
        self.attention_activation = attention_activation
        self.softmax_attention = softmax_attention
        self.math = math
        self.record_side_channels = True
        self._att = self._natt = self._coords = self._side_csr = None

        # creation order == reference (same RNG draws for a given seed)
        self.edge_mlp = nn.Sequential(
            nn.Linear(input_edge + 1 + edges_in_d, hidden_nf), act_fn,
            nn.Linear(hidden_nf, hidden_nf), act_fn)
        self.node_mlp = nn.Sequential(
            nn.Linear(hidden_nf + input_nf, hidden_nf),
            GraphNorm(hidden_nf) if graphnorm else nn.Identity(), act_fn,
            nn.Linear(hidden_nf, output_nf))
        layer = nn.Linear(hidden_nf, 1, bias=False)
        torch.nn.init.xavier_uniform_(layer.weight, gain=0.001)
        self.coord_mlp = nn.Sequential(
            nn.Linear(hidden_nf, hidden_nf), act_fn, layer,
            nn.Tanh() if tanh else nn.Identity())
        if self.edge_attention:
            self.att_mlp = nn.Sequential(
                nn.Linear(hidden_nf, 1), attention_activation())
        if self.node_attention:
            self.node_att_mlp = nn.Sequential(
                nn.Linear(hidden_nf, 1), attention_activation())
        if self.rezero:
            if self.edge_residual:
                self.edge_gate_parameter = nn.Parameter(torch.zeros(1))
            if self.residual:
                self.node_gate_parameter = nn.Parameter(torch.zeros(1))
        elif self.gated_residual:
            if self.edge_residual:
                self.edge_gate_parameter = nn.Parameter(0.5 * torch.ones(1))
            if self.residual:
                self.node_gate_parameter = nn.Parameter(0.5 * torch.ones(1))

    # -- C-ABI views --------------------------------------------------------
    def c_flags(self):
        f = 0
        for on, bit in ((self.residual, _cabi.F_RESIDUAL),
                        (self.edge_residual, _cabi.F_EDGE_RESIDUAL),
                        (self.edge_attention, _cabi.F_EDGE_ATTENTION),
                        (self.normalize, _cabi.F_NORMALIZE),
                        (self.tanh, _cabi.F_TANH),
                        (self.graphnorm, _cabi.F_GRAPHNORM),
                        (self.use_coords, _cabi.F_UPDATE_COORDS),
                        (self.permutation_invariance, _cabi.F_PERM_INVARIANT),
                        (self.node_attention, _cabi.F_NODE_ATTENTION),
                        (self.gated_residual, _cabi.F_GATED_RESIDUAL),
                        (self.rezero, _cabi.F_REZERO),
                        (self.softmax_attention, _cabi.F_SOFTMAX_ATTENTION)):
            if on:
                f |= bit
        return f

    def c_config(self):
        act = 'none' if self.softmax_attention else self.attention_activation_fn
        return _cabi.LayerConfig(self.hidden_nf, self.edges_in_d,
                                 self.c_flags(), _cabi.ACT[act],
                                 _cabi.MATH[self.math], 0, None, None, None)

    def c_params(self, params):
        """struct pvs_layer_params of `params` (PARAM_FIELDS order), cached on
        the parameters' storage addresses: twenty pointer fields per call are a
        measurable part of a training step's host time."""
        key = tuple(0 if p is None else p.data_ptr() for p in params)
        cached = self.__dict__.get('_c_params')
        if cached is not None and cached[0] == key:
            return cached[1]
        if any(p is not None and not p.is_contiguous() for p in params):
            keep = [None if p is None else p.detach().contiguous() for p in params]
            st = _cabi.LayerParams(*[ptr(p) for p in keep])
            st._keep = keep
            return st
        st = _cabi.LayerParams(*[C.c_void_p(a) if a else None for a in key])
        self.__dict__['_c_params'] = (key, st)
        return st

    def param_list(self):
        """Parameters in _cabi.PARAM_FIELDS order (None where absent)."""
        gn = self.node_mlp[1] if self.graphnorm else None
        att = self.att_mlp[0] if self.edge_attention else None
        natt = self.node_att_mlp[0] if self.node_attention else None
        return [
            self.edge_mlp[0].weight, self.edge_mlp[0].bias,
            self.edge_mlp[2].weight, self.edge_mlp[2].bias,
            self.coord_mlp[0].weight, self.coord_mlp[0].bias,
            self.coord_mlp[2].weight,
            None if att is None else att.weight,
            None if att is None else att.bias,
            self.node_mlp[0].weight, self.node_mlp[0].bias,
            None if gn is None else gn.weight,
            None if gn is None else gn.bias,
            None if gn is None else gn.mean_scale,
            self.node_mlp[3].weight, self.node_mlp[3].bias,
            None if natt is None else natt.weight,
            None if natt is None else natt.bias,
            getattr(self, 'edge_gate_parameter', None),
            getattr(self, 'node_gate_parameter', None),
        ]

    # -- side channels (numpy in the reference; lazy here) --------------------
    @property
    def att_val(self):
        if self._att is None:
            return None
        return self._side_csr.to_caller_order(self._att).unsqueeze(1).cpu().numpy()

    @att_val.setter
    def att_val(self, value):
        self._att = value

    @property
    def node_att_val(self):
        return None if self._natt is None else \
            self._natt.unsqueeze(1).cpu().numpy()

    @node_att_val.setter
    def node_att_val(self, value):
        self._natt = value

    @property
    def intermediate_coords(self):
        return None if self._coords is None else self._coords.cpu().numpy()

    @intermediate_coords.setter
    def intermediate_coords(self, value):
        self._coords = value

    # -- execution -------------------------------------------------------------
    def apply_csr(self, csr, h, x, m_prev=None, want_m=True):
        """Run the layer on a prebuilt CSR.  m_prev / returned m are in CSR
        order.  Returns (h', x', m or None)."""
        _cabi.require_cuda(h, x)
        if h.shape[1] != self.hidden_nf:
            raise ValueError(f'h has {h.shape[1]} channels, layer expects '
                             f'{self.hidden_nf}')
        if self.edges_in_d > 8:
            raise ValueError('edges_in_d > 8 unsupported')
        if self.edges_in_d and csr.n_edges and csr.n_classes > self.edges_in_d:
            raise ValueError(
                f'edge_attr has {csr.n_classes} classes, layer was built '
                f'with edges_in_d={self.edges_in_d}')
        side = self.record_side_channels
        if not (self.edge_residual and m_prev is not None):
            m_prev = None
        h_out, x_out, m, att, natt = _EGNNLayerFn.apply(
            self, csr, want_m, side, h.float(), x.float(), m_prev,
            *self.param_list())
        if side:
            self._side_csr = csr
            self._att, self._natt = att, natt
            self._coords = x_out.detach() if self.use_coords else None
        return h_out, x_out, m

    def forward(self, h, edge_index, coord, edge_attr=None, edge_messages=None):
        """Reference signature (egnn_satorras.py:189).  `coord` is updated IN
        PLACE, as the reference does (`coord += agg`, :174)."""
        csr = _csr_for(edge_index, edge_attr if self.edges_in_d else None,
                       h.shape[0])
        m_prev = None
        if self.edge_residual and edge_messages is not None:
            m_prev = csr.from_caller_order(edge_messages)
        h_out, x_out, m = self.apply_csr(csr, h, coord, m_prev, want_m=True)
        if self.use_coords:
            if coord.requires_grad or x_out.requires_grad:
                coord = x_out
            else:
                coord.copy_(x_out)
        return h_out, coord, edge_attr, csr.to_caller_order(m)


class PygLinearPass(nn.Module):
    """Mirror of PygLinearPass (pnn_geometric_base.py:61-94): the embedding
    `Linear(dim_input -> k)` with the layer calling convention."""

    def __init__(self, module, feats_appended_to_coords=False,
                 return_coords_and_edges=False):
        super().__init__()
        self.m = module
        self.feats_appended_to_coords = feats_appended_to_coords
        self.return_coords_and_edges = return_coords_and_edges
        self._coords = None

    @property
    def intermediate_coords(self):
        return None if self._coords is None else self._coords.cpu().numpy()

    def embed(self, feats):
        from .dense import linear
        return linear(feats, self.m.weight, self.m.bias, 'none')

    def forward(self, h, **kwargs):
        if self.feats_appended_to_coords:
            self._coords = h[:, :3].detach()
            res = torch.hstack([h[:, :3], self.embed(h[:, 3:])])
        else:
            self._coords = kwargs['coord'].detach().clone()
            res = self.embed(h)
        if self.return_coords_and_edges:
            return res, kwargs['coord'], kwargs['edge_attr'], kwargs.get(
                'edge_messages', None)
        return res


class PNNGeometricBase(PointNeuralNetworkBase):
    """Mirror of PNNGeometricBase (pnn_geometric_base.py:17-58)."""

    def get_embeddings(self, feats, edges, coords, edge_attributes, batch):
        raise NotImplementedError

    def _pool_and_head(self, feats, batch, graph, head):
        from .dense import mean_pool, run_head
        n_graphs = getattr(graph, 'num_graphs', None)
        graph_ptr = getattr(graph, 'graph_ptr', None)
        if graph_ptr is not None:
            n_graphs = graph_ptr.numel() - 1
        elif n_graphs is None:
            # the reference syncs here too (pnn_geometric_base.py:27)
            n_graphs = int(batch.max().item()) + 1
        pooled = mean_pool(feats, batch, n_graphs, graph_ptr)
        out = run_head(head, pooled)
        if n_graphs == 1:   # reference returns [dim_output] for one graph (:31)
            out = out.reshape(-1)
        return out

    def _unpack_for_forward(self, graph):
        """unpack_graph, except that a batch carrying a prebuilt CSR
        (PackedBatch) never materialises edge_index / one-hot edge_attr."""
        csr = getattr(graph, 'pvs_csr', None)
        if csr is None:
            return (*self.unpack_graph(graph), None)
        dev = self.device_for_inputs()
        batch = None if getattr(graph, 'graph_ptr', None) is not None \
            else graph.batch.to(dev)
        return (graph.x.float().to(dev), None, graph.pos.float().to(dev), None,
                batch, csr)

    # -- one-call scoring path ---------------------------------------------------
    def _apply(self, fn, *args, **kwargs):
        self.__dict__.pop('_c_cache', None)      # parameter storage may move
        return super()._apply(fn, *args, **kwargs)

    def _fast_path_ok(self):
        if torch.is_grad_enabled() and any(
                p.requires_grad for p in self.parameters()):
            return False
        if self.training and getattr(self, 'dropout_p', 0) > 0:
            return False        # edge dropout rebuilds the graph per call
        if STAGE_TIMER is not None and getattr(STAGE_TIMER, 'split_stages', True):
            return False
        egnn = [l for l in self.layers if isinstance(l, EGNNLayer)]
        if any(l.record_side_channels for l in egnn):
            return False
        if getattr(self, 'record_embed_coords', True):
            return False
        return not self.layers[0].feats_appended_to_coords

    def _c_model(self, head):
        """ctypes descriptor of the whole model (cached; it holds raw pointers
        into the live parameter storage, so in-place optimiser updates and
        load_state_dict are seen without rebuilding)."""
        cache = self.__dict__.setdefault('_c_cache', {})
        egnn = [l for l in self.layers if isinstance(l, EGNNLayer)]
        key = (id(head), tuple(l.math for l in egnn))
        if key in cache:
            return cache[key]
        keep = []

        def dptr(t):
            if t is None:
                return None
            t = t.detach()
            if not t.is_contiguous():
                raise _cabi.PvsError('parameters must be contiguous')
            keep.append(t)
            return C.c_void_p(t.data_ptr())

        cfgs = (_cabi.LayerConfig * max(1, len(egnn)))()
        params = (_cabi.LayerParams * max(1, len(egnn)))()
        for i, layer in enumerate(egnn):
            cfgs[i] = layer.c_config()
            params[i] = _cabi.LayerParams(*[dptr(p) for p in layer.param_list()])
        mods = list(head)
        heads = []
        i = 0
        while i < len(mods):
            lin = mods[i]
            if not isinstance(lin, nn.Linear):
                raise NotImplementedError(f'head module {type(lin).__name__}')
            act = 'none'
            if i + 1 < len(mods) and not isinstance(mods[i + 1], nn.Linear):
                act = {nn.SiLU: 'silu', nn.ReLU: 'relu',
                       nn.Softplus: 'softplus'}[type(mods[i + 1])]
                i += 1
            heads.append(_cabi.HeadLayer(dptr(lin.weight), dptr(lin.bias),
                                         lin.in_features, lin.out_features,
                                         _cabi.ACT[act]))
            i += 1
        head_arr = (_cabi.HeadLayer * len(heads))(*heads)
        embed = self.layers[0].m
        desc = _cabi.ModelDesc(len(egnn), egnn[0].hidden_nf if egnn else
                               embed.out_features, embed.in_features,
                               len(heads), dptr(embed.weight), dptr(embed.bias),
                               cfgs, params, head_arr)
        cache[key] = (desc, cfgs, (params, head_arr, keep), heads[-1].ko)
        return cache[key]

    def _forward_fast(self, graph, head):
        """Whole scoring pass in one C call (pvs_egnn_model_fwd)."""
        dev = self.device_for_inputs()
        csr = getattr(graph, 'pvs_csr', None)
        feats = graph.x.float().to(dev).contiguous()
        pos = graph.pos.float().to(dev).contiguous()
        if csr is None:
            csr = _csr_for(graph.edge_index.to(dev), graph.edge_attr.to(dev),
                           feats.shape[0])
        graph_ptr = getattr(graph, 'graph_ptr', None)
        if graph_ptr is None:
            from .dense import batch_to_ptr
            batch = graph.batch.to(dev)
            n_graphs = int(batch.max().item()) + 1   # as the reference (:27)
            graph_ptr = batch_to_ptr(batch, n_graphs)
        n_graphs = int(graph_ptr.numel()) - 1
        desc, cfgs, _keep, dim_out = self._c_model(head)
        timer = STAGE_TIMER
        if timer is not None:
            for i in range(desc.n_layers):
                cfgs[i].ev_edge_begin, cfgs[i].ev_edge_end = \
                    timer.next_edge_events()
        elif cfgs[0].ev_edge_begin:
            for i in range(desc.n_layers):
                cfgs[i].ev_edge_begin = cfgs[i].ev_edge_end = None
        h = lib()
        nbytes = int(h.pvs_egnn_model_workspace_bytes(
            csr.n_nodes, csr.n_edges, n_graphs, C.byref(desc)))
        if nbytes < 0:
            raise _cabi.PvsError(
                'unsupported model for the fused scoring pass: ' + _width_error(
                    desc.k, any(cfgs[i].math == _cabi.MATH['fp32']
                                for i in range(desc.n_layers))))
        ws = _cabi.scratch('model_fwd', nbytes, dev)
        scores = torch.empty((n_graphs, dim_out), dtype=torch.float32,
                             device=dev)
        maths = [l.math for l in self.layers if isinstance(l, EGNNLayer)]
        g = csr.c_struct(node_tiles='fp32' in maths,
                         packed_tiles=any(m != 'fp32' for m in maths))
        with torch.cuda.device(dev):
            check(h.pvs_egnn_model_fwd(
                C.byref(g), C.byref(desc), ptr(feats), feats.shape[1],
                ptr(pos), ptr(graph_ptr), n_graphs, ptr(scores), ptr(pos),
                None, ptr(ws), C.c_int64(ws.numel()), stream()),
                'pvs_egnn_model_fwd')
        if pos.data_ptr() != graph.pos.data_ptr() and \
                graph.pos.dtype == torch.float32 and graph.pos.is_cuda:
            graph.pos.copy_(pos)      # keep the in-place coordinate update
        return scores.reshape(-1) if n_graphs == 1 else scores

    def forward(self, x):
        if self.feats_linear_layers is not None and self._fast_path_ok():
            return self._forward_fast(x, self.feats_linear_layers)
        feats, edges, coords, edge_attributes, batch, csr = \
            self._unpack_for_forward(x)
        feats, _ = self.get_embeddings(
            feats, edges, coords, edge_attributes, batch,
            _csr=csr, _want_messages=False)
        if self.feats_linear_layers is not None:
            feats = self._pool_and_head(feats, batch, x,
                                        self.feats_linear_layers)
        return feats

    def unpack_input_data_and_predict(self, input_data):
        y_true = input_data.y
        try:
            y_true = y_true.float()
        except (AttributeError, TypeError):
            pass
        y_pred = self(input_data).reshape(-1, )
        return y_pred, y_true, input_data.lig_fname, input_data.rec_fname

    def unpack_graph(self, graph):
        dev = self.device_for_inputs()
        return (graph.x.float().to(dev), graph.edge_index.to(dev),
                graph.pos.float().to(dev), graph.edge_attr.to(dev),
                graph.batch.to(dev))

    def device_for_inputs(self):
        return next(self.parameters()).device


class SartorrasEGNN(PNNGeometricBase):
    """Mirror of SartorrasEGNN (egnn_satorras.py:209-329): the `egnn` model."""
    # pylint: disable = R, W0201, W0613

    def build_net(self, dim_input, k, dim_output, act_fn=nn.SiLU(),
                  num_layers=4, residual=True, edge_residual=False,
                  edge_attention=False, normalize=True, tanh=True, dropout=0.0,
                  graphnorm=True, multi_fc=False, update_coords=True,
                  permutation_invariance=False,
                  attention_activation_fn='sigmoid', node_attention=False,
                  gated_residual=False, rezero=False,
                  model_task='classification', include_strain_info=False,
                  final_softplus=False, softmax_attention=False, **kwargs):
        layers = [PygLinearPass(nn.Linear(dim_input, k),
                                return_coords_and_edges=True)]
        self.n_layers = num_layers
        self.dropout_p = dropout
        self.residual, self.edge_residual = residual, edge_residual
        self.gated_residual, self.rezero = gated_residual, rezero
        self.model_task = model_task
        self.include_strain_info = include_strain_info
        self.softmax_attention = softmax_attention
        math = kwargs.get('math', 'fp32')
        assert not (gated_residual and rezero), \
            'gated_residual and rezero are incompatible'
        for _ in range(num_layers):
            layers.append(EGNNLayer(
                k, k, k, edges_in_d=3, act_fn=act_fn, residual=residual,
                edge_attention=edge_attention, normalize=normalize,
                graphnorm=graphnorm, tanh=tanh, update_coords=update_coords,
                permutation_invariance=permutation_invariance,
                attention_activation_fn=attention_activation_fn,
                node_attention=node_attention, edge_residual=edge_residual,
                gated_residual=gated_residual, rezero=rezero,
                softmax_attention=softmax_attention, math=math))
        if include_strain_info:
            k += 1
        if multi_fc:
            fc_layer_dims = ((k, 32), (32, 16), (16, dim_output))
        else:
            fc_layer_dims = ((k, dim_output),)
        feats_linear_layers = []
        for idx, (in_dim, out_dim) in enumerate(fc_layer_dims):
            feats_linear_layers.append(nn.Linear(in_dim, out_dim))
            if idx < len(fc_layer_dims) - 1:
                feats_linear_layers.append(nn.SiLU())
        if final_softplus:
            feats_linear_layers.append(nn.Softplus())
        self.feats_linear_layers = nn.Sequential(*feats_linear_layers)
        return nn.Sequential(*layers)

    def set_math(self, math):
        """'fp32' (FFMA), 'bf16x3' or 'fp16x2' (tcgen05, fp32-class) or 'bf16'
        (tcgen05, fast)."""
        if math not in _cabi.MATH:
            raise ValueError(f'math must be one of {sorted(_cabi.MATH)}')
        for layer in self.layers:
            if isinstance(layer, EGNNLayer):
                layer.math = math
        self.__dict__.pop('_c_cache', None)
        return self

    def set_record_side_channels(self, on):
        for layer in self.layers:
            if isinstance(layer, EGNNLayer):
                layer.record_side_channels = bool(on)
        return self

    def _stack_ok(self, egnn_layers, h, want_messages):
        """Training pass through all layers in one call each way: gradients
        wanted, nobody needs edge messages / side channels / stage timing, one
        arithmetic mode."""
        if not egnn_layers or want_messages or STAGE_TIMER is not None:
            return False
        if not torch.is_grad_enabled() or not (
                h.requires_grad or any(p.requires_grad
                                       for p in egnn_layers[0].parameters())):
            return False
        # PVS_STACK_TRAIN=1 forces the stacked pass, =0 forbids it; by default
        # it is used by models that are being trained through `backprop()`
        # (base.py sets `_lean_training`), in its lean form: the device time of
        # a step is the same either way, the host time is less than half
        # (sixteen autograd Functions with 27 inputs each -> two calls), which
        # decides the step time whenever the host is the slower side.
        env = os.environ.get('PVS_STACK_TRAIN', '')
        if env == '0' or (env in ('', None) and
                          not getattr(self, '_lean_training', False)):
            return False
        return all(not l.edge_residual and not l.record_side_channels and
                   l.math == egnn_layers[0].math and
                   l.hidden_nf == egnn_layers[0].hidden_nf
                   for l in egnn_layers)

    def get_embeddings(self, feats, edges, coords, edge_attributes, batch,
                       _csr=None, _want_messages=True):
        """Reference signature (egnn_satorras.py:319-329) -> (h [N,k],
        m [E,k] in the caller's edge order).  `coords` is updated in place
        when it is an fp32 CUDA tensor, as in the reference."""
        _cabi.require_cuda(feats, coords)
        csr = _csr if isinstance(_csr, CSRGraph) else \
            _csr_for(edges, edge_attributes, feats.shape[0])
        if self.dropout_p > 0 and self.training:
            # the messages returned below are those of the thinned edge list
            csr = dropout_adj(csr, self.dropout_p, force_undirected=True)
        embed = self.layers[0]
        if embed.feats_appended_to_coords:
            raise NotImplementedError('feats_appended_to_coords')
        embed._coords = coords.detach().clone() \
            if getattr(self, 'record_embed_coords', True) else None
        h = embed.embed(feats.float())
        x = coords.float()
        m = None
        egnn_layers = list(self.layers)[1:]
        if self._stack_ok(egnn_layers, h, _want_messages):
            if getattr(self, '_lean_training', False):
                plan = _StackPlan.of(self, egnn_layers)
                h, x = _EGNNStackLeanFn.apply(plan, csr, h.contiguous(),
                                              x.contiguous(), plan.anchor)
            else:
                flat = [p for layer in egnn_layers for p in layer.param_list()]
                h, x = _EGNNStackFn.apply(tuple(egnn_layers), csr,
                                          h.contiguous(), x.contiguous(), *flat)
            egnn_layers = []
        for i, layer in enumerate(egnn_layers):
            last = i == len(egnn_layers) - 1
            want_m = layer_needs = (
                (not last and egnn_layers[i + 1].edge_residual) or
                (last and _want_messages))
            h, x, m_new = layer.apply_csr(csr, h, x, m, want_m=want_m)
            m = m_new if layer_needs else None
        if x is not coords and coords.dtype == torch.float32 and \
                not x.requires_grad:
            coords.copy_(x)     # the reference's in-place `coord += agg`
        if m is not None:
            m = csr.to_caller_order(m)
        return h, m


class MultitaskSatorrasEGNN(SartorrasEGNN):
    """Mirror of MultitaskSatorrasEGNN (egnn_multitask.py:11-166)."""
    # pylint: disable = R, W0201, W0613, W0221

    def build_net(self, dim_input, k, dim_output, act_fn=nn.SiLU(),
                  num_layers=4, residual=True, edge_residual=False,
                  edge_attention=False, normalize=True, tanh=True, dropout=0.0,
                  graphnorm=True, update_coords=True,
                  permutation_invariance=False,
                  attention_activation_fn='sigmoid', node_attention=False,
                  node_attention_final_only=False,
                  edge_attention_final_only=False,
                  node_attention_first_only=False,
                  edge_attention_first_only=False, gated_residual=False,
                  rezero=False, model_task='classification',
                  final_softplus=False, softmax_attention=False, **kwargs):
        embedding_layers = [PygLinearPass(nn.Linear(dim_input, k),
                                          return_coords_and_edges=True)]
        self.n_layers = num_layers
        self.dropout_p = dropout
        self.residual, self.edge_residual = residual, edge_residual
        self.gated_residual, self.rezero = gated_residual, rezero
        self.model_task = model_task
        self.softmax_attention = softmax_attention
        math = kwargs.get('math', 'fp32')
        assert not (gated_residual and rezero), \
            'gated_residual and rezero are incompatible'

        def placed(on, first_only, final_only, i):   # egnn_multitask.py:96-122
            if not on:
                return False
            if not first_only and not final_only:
                return True
            if first_only and i == 0:
                return True
            return bool(final_only and i == num_layers - 1)

        for i in range(num_layers):
            embedding_layers.append(EGNNLayer(
                k, k, k, edges_in_d=3, act_fn=act_fn, residual=residual,
                edge_attention=placed(edge_attention,
                                      edge_attention_first_only,
                                      edge_attention_final_only, i),
                normalize=normalize, graphnorm=graphnorm, tanh=tanh,
                update_coords=update_coords,
                permutation_invariance=permutation_invariance,
                attention_activation_fn=attention_activation_fn,
                node_attention=placed(node_attention,
                                      node_attention_first_only,
                                      node_attention_final_only, i),
                edge_residual=edge_residual, gated_residual=gated_residual,
                rezero=rezero, softmax_attention=softmax_attention, math=math))
        feats_linear_layers_affinity = [nn.Linear(k, dim_output)]
        feats_linear_layers_affinity.append(
            nn.Softplus() if final_softplus else nn.ReLU())
        self.feats_linear_layers_pose = nn.Sequential(nn.Linear(k, 1))
        self.feats_linear_layers_affinity = nn.Sequential(
            *feats_linear_layers_affinity)
        self.feats_linear_layers = None
        return nn.Sequential(*embedding_layers)

    def forward(self, graph):
        head = self.feats_linear_layers_pose \
            if 'classification' in self.model_task \
            else self.feats_linear_layers_affinity
        if self._fast_path_ok():
            return self._forward_fast(graph, head)
        feats, edges, coords, edge_attributes, batch, csr = \
            self._unpack_for_forward(graph)
        feats, _ = self.get_embeddings(
            feats, edges, coords, edge_attributes, batch,
            _csr=csr, _want_messages=False)
        head = self.feats_linear_layers_pose \
            if 'classification' in self.model_task \
            else self.feats_linear_layers_affinity
        return self._pool_and_head(feats, batch, graph, head)
