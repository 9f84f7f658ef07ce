"""Backward passes of the autograd Functions (K3 and the dense helpers).

Training goes through the same C ABI as scoring: these functions only marshal
tensors into pvs_egnn_layer_bwd / pvs_linear_bwd / pvs_mean_pool_bwd.  The
kernels recompute the layer from its saved inputs; PyTorch autograd is used
only to chain the layers together (and for the loss and optimiser, as in the
reference's `backprop`, point_neural_network_base.py:417-429).
"""
import ctypes as C

import torch

from . import _cabi
from ._cabi import check, lib, ptr, stream


# Gradient arena of the model whose `backprop()` is running (parallel.GradArena)
# or None: the backward passes below then allocate their own zero-filled
# gradient tensors.
ARENA = None


class use_arena:
    """Context manager: parameter gradients of the backward passes inside go
    straight into `arena`'s slots."""

    def __init__(self, arena):
        self.arena = arena

    def __enter__(self):
        global ARENA
        self.prev, ARENA = ARENA, self.arena
        return self.arena

    def __exit__(self, *exc):
        global ARENA
        ARENA = self.prev
        return False


def _zeros_like_or_none(p):
    return None if p is None else torch.zeros_like(p, dtype=torch.float32)


def _unused_fields(layer, no_dx, no_m_prev):
    """Parameters that cannot influence the loss get no gradient at all (None),
    as under the reference's autograd: an optimiser with weight decay skips
    them instead of decaying them.  That is the coordinate MLP of a layer
    whose output coordinates nobody consumes (the last layer), or which does
    not update coordinates; and the edge gate of a layer without incoming
    messages."""
    unused = ()
    if no_dx or not layer.use_coords:
        unused += ('coord_w1', 'coord_b1', 'coord_w2')
    if no_m_prev:
        unused += ('edge_gate',)
    return unused


def _bwd_workspace(cfg, n, e, dev):
    """Scratch of pvs_egnn_layer_bwd: never escapes the call and every use is
    ordered on the stream, so one grow-only buffer serves all layers."""
    nbytes = int(lib().pvs_egnn_layer_bwd_workspace_bytes(n, e, C.byref(cfg)))
    return _cabi.scratch('layer_bwd', nbytes, dev)


class _LayerBwdPlan:
    """What egnn_layer_backward needs again on every step while the layer's
    parameters and the gradient arena stay where they are: the pointer block of
    the gradient slots, their keys and span."""

    def __init__(self, arena, pstruct, gstruct, params, in_arena, grads):
        self.arena, self.pstruct, self.gstruct = arena, pstruct, gstruct
        self._keep = grads                      # the views the pointers refer to
        self.keys = frozenset(p.data_ptr() for p in in_arena)
        self.span = arena.span(in_arena)
        self.nones = (None,) * len(params)
        self._by_field = {name: p.data_ptr()
                          for name, p in zip(_cabi.PARAM_FIELDS, params)
                          if p is not None}
        self._granted = {}

    def granted(self, unused):
        keys = self._granted.get(unused)
        if keys is None:
            drop = {self._by_field[name] for name in unused
                    if name in self._by_field}
            keys = frozenset(self.keys - drop)
            self._granted[unused] = keys
        return keys


def egnn_layer_backward(ctx, d_h, d_x, d_m):
    layer, csr = ctx.layer, ctx.csr
    h, x, m_prev, *params = ctx.saved_tensors
    cfg = layer.c_config()
    # differentiate the function the forward evaluated, also when set_math()
    # ran in between
    cfg.math = _cabi.MATH[ctx.fwd_math]
    fwd_ws = getattr(ctx, 'fwd_ws', None)
    if fwd_ws is not None:
        cfg.saved_fwd_workspace = ptr(fwd_ws)
    n, e, k = csr.n_nodes, csr.n_edges, layer.hidden_nf
    dev = h.device
    d_h = torch.zeros_like(h) if d_h is None else d_h.contiguous().float()
    no_dx = d_x is None
    d_x = None if d_x is None else d_x.contiguous().float()
    d_m = None if d_m is None else d_m.contiguous().float()
    csc_ptr, csc_eid = csr.csc()

    pstruct = layer.c_params(params)
    arena = ARENA
    unused = _unused_fields(layer, no_dx, m_prev is None)
    plan = layer.__dict__.get('_bwd_plan')
    if arena is not None and plan is not None and plan.arena is arena \
            and plan.pstruct is pstruct and arena.hand_out_all(plan.keys):
        # steady state of a training run: every gradient of the layer has an
        # arena slot, and the pointer block built on an earlier step is reused
        d_h_in = torch.empty_like(h)
        d_x_in = torch.empty_like(x)
        d_m_prev = torch.zeros_like(m_prev) if m_prev is not None else None
        ws = _bwd_workspace(cfg, n, e, dev)
        g = csr.c_struct()
        with torch.cuda.device(dev):
            check(lib().pvs_egnn_layer_bwd(
                C.byref(g), ptr(csc_ptr), ptr(csc_eid), C.byref(cfg),
                C.byref(pstruct), ptr(h), ptr(x), ptr(m_prev), ptr(d_h), ptr(d_x),
                ptr(d_m), ptr(d_h_in), ptr(d_x_in), ptr(d_m_prev),
                C.byref(plan.gstruct), ptr(ws), C.c_int64(ws.numel()), stream()),
                'pvs_egnn_layer_bwd')
        if arena.reduce_in_backward:
            arena.reduce_async(*plan.span)
        arena.grant_all(plan.granted(unused))
        return (None, None, None, None, d_h_in, d_x_in, d_m_prev, *plan.nones)
    by_name = dict(zip(_cabi.PARAM_FIELDS, params))
    grads, in_arena = {}, []
    if arena is not None:
        # the model's gradient arena: slots are already zero
        for name in _cabi.GRAD_FIELDS:
            grads[name] = arena.grad_view(by_name[name])
            if grads[name] is not None:
                in_arena.append(by_name[name])
    rest = [name for name in _cabi.GRAD_FIELDS
            if by_name[name] is not None and grads.get(name) is None]
    if rest:
        # one zero-filled flat buffer for the remaining gradients of the layer
        sizes = {name: by_name[name].numel() for name in rest}
        flat = torch.zeros(sum(sizes.values()), dtype=torch.float32, device=dev)
        off = 0
        for name in rest:
            grads[name] = flat[off:off + sizes[name]]
            off += sizes[name]
    for name in _cabi.GRAD_FIELDS:
        grads.setdefault(name, None)
    gstruct = _cabi.LayerGrads(*[ptr(grads[name]) for name in _cabi.GRAD_FIELDS])

    d_h_in = torch.empty_like(h)
    d_x_in = torch.empty_like(x)
    d_m_prev = torch.zeros_like(m_prev) if m_prev is not None else None
    ws = _bwd_workspace(cfg, n, e, dev)
    g = csr.c_struct()
    with torch.cuda.device(dev):
        check(lib().pvs_egnn_layer_bwd(
            C.byref(g), ptr(csc_ptr), ptr(csc_eid), C.byref(cfg),
            C.byref(pstruct), ptr(h), ptr(x), ptr(m_prev), ptr(d_h), ptr(d_x),
            ptr(d_m), ptr(d_h_in), ptr(d_x_in), ptr(d_m_prev),
            C.byref(gstruct), ptr(ws), C.c_int64(ws.numel()), stream()),
            'pvs_egnn_layer_bwd')
    if arena is not None and arena.reduce_in_backward and in_arena:
        # data-parallel: this layer's slice of the arena is complete -- average
        # it over the ranks while the next layer's backward runs
        arena.reduce_async(*arena.span(in_arena))
    if arena is not None and not rest \
            and layer.__dict__.get('_c_params', (None, None))[1] is pstruct:
        # every gradient of the layer sits in the arena: remember the pointer
        # block for the following steps
        layer.__dict__['_bwd_plan'] = _LayerBwdPlan(arena, pstruct, gstruct, params,
                                                    in_arena, grads)
    # inputs of _EGNNLayerFn.forward: layer, csr, want_m, want_side, h, x,
    # m_prev, *params
    # Parameters that cannot influence the loss get no gradient at all (None),
    # as under the reference's autograd: an optimiser with weight decay skips
    # them instead of decaying them.  That is the coordinate MLP of a layer
    # whose output coordinates nobody consumes (the last layer), or which does
    # not update coordinates.
    arena_ptrs = {p.data_ptr() for p in in_arena}
    param_grads = []
    for name, p in zip(_cabi.PARAM_FIELDS, params):
        if p is None or name not in grads or grads[name] is None \
                or name in unused:
            param_grads.append(None)
        elif p.data_ptr() in arena_ptrs:
            # the gradient already sits in the parameter's arena slot, which
            # becomes `p.grad` (GradArena.attach_grads): nothing for autograd
            # to accumulate
            arena.grant(p)
            param_grads.append(None)
        else:
            param_grads.append(grads[name].reshape(p.shape))
    return (None, None, None, None, d_h_in, d_x_in, d_m_prev, *param_grads)


def egnn_stack_backward(ctx, d_h, d_x):
    """Backward of _EGNNStackFn: every layer's K3 in one library call."""
    layers, csr = ctx.layers, ctx.csr
    L = len(layers)
    per = len(_cabi.PARAM_FIELDS)
    saved = list(ctx.saved_tensors)
    params = [saved.pop(0) if present else None for present in ctx.param_mask]
    H, X, ws = ctx.H, ctx.X, ctx.ws
    n, e = csr.n_nodes, csr.n_edges
    dev = H.device
    d_h = torch.zeros_like(H[L]) if d_h is None else d_h.contiguous().float()
    no_dx = d_x is None
    d_x = None if no_dx else d_x.contiguous().float()
    csc_ptr, csc_eid = csr.csc()
    arena = ARENA
    cfgs = (_cabi.LayerConfig * L)()
    pstructs = (_cabi.LayerParams * L)()
    gstructs = (_cabi.LayerGrads * L)()
    keep, plans = [], []
    span_params = []
    for i, layer in enumerate(layers):
        cfgs[i] = layer.c_config()
        cfgs[i].math = _cabi.MATH[ctx.math]     # the forward's, as in the layer
        ps = params[i * per:(i + 1) * per]
        det = [None if p is None else p.detach().contiguous() for p in ps]
        keep.append(det)
        pstructs[i] = _cabi.LayerParams(*[ptr(p) for p in det])
        by_name = dict(zip(_cabi.PARAM_FIELDS, ps))
        grads, in_arena = {}, set()
        for name in _cabi.GRAD_FIELDS:
            p = by_name[name]
            view = arena.grad_view(p) if (arena is not None and p is not None) \
                else None
            if view is not None:
                in_arena.add(name)
                span_params.append(p)
            elif p is not None:
                view = torch.zeros_like(p, dtype=torch.float32)
            grads[name] = view
        keep.append(grads)
        gstructs[i] = _cabi.LayerGrads(*[ptr(grads[name])
                                         for name in _cabi.GRAD_FIELDS])
        plans.append((by_name, grads, in_arena))
    d_h_in = torch.empty_like(H[0])
    d_x_in = torch.empty_like(X[0])
    nbytes = int(lib().pvs_egnn_stack_bwd_workspace_bytes(n, e, L, cfgs))
    bws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    g = csr.c_struct()
    with torch.cuda.device(dev):
        check(lib().pvs_egnn_stack_bwd(
            C.byref(g), ptr(csc_ptr), ptr(csc_eid), L, cfgs, pstructs, gstructs,
            ptr(H), ptr(X), ptr(ws),
            C.c_int64(ctx.stride), ptr(d_h), ptr(d_x), ptr(d_h_in), ptr(d_x_in),
            ptr(bws), C.c_int64(bws.numel()), stream()), 'pvs_egnn_stack_bwd')
    if arena is not None and arena.reduce_in_backward and span_params:
        arena.reduce_async(*arena.span(span_params))
    # same rules as egnn_layer_backward for parameters that cannot influence the
    # loss: the coordinate MLP of a layer whose output coordinates nobody
    # consumes (the last layer when d_x is None) or which does not update
    # coordinates, and the edge gate (no incoming messages in a stack)
    out = []
    for i, layer in enumerate(layers):
        by_name, grads, in_arena = plans[i]
        unused = {'edge_gate'}
        if not layer.use_coords or (no_dx and i == L - 1):
            unused.update(('coord_w1', 'coord_b1', 'coord_w2'))
        for name in _cabi.PARAM_FIELDS:
            p = by_name[name]
            if p is None or grads[name] is None or name in unused:
                out.append(None)
            elif name in in_arena:
                arena.grant(p)
                out.append(None)
            else:
                out.append(grads[name].reshape(p.shape))
    return (None, None, d_h_in, d_x_in, *out)


class _StackGradPlan:
    """Gradient pointer block of a stacked backward for one gradient arena."""

    def __init__(self, plan, arena):
        layers, params = plan.layers, plan.params
        L, per = len(layers), len(_cabi.PARAM_FIELDS)
        self.ok = all(p is None or not p.requires_grad or
                      p.data_ptr() in arena.slots for p in params)
        if not self.ok:
            return
        live = [p for p in params if p is not None and p.requires_grad]
        self.keys = frozenset(p.data_ptr() for p in live)
        self.ok = len(self.keys) == len(live)      # a parameter shared by layers
        if not self.ok:
            return
        self.gstructs = (_cabi.LayerGrads * L)()
        for i in range(L):
            ps = params[i * per:(i + 1) * per]
            self.gstructs[i] = _cabi.LayerGrads(*[
                ptr(arena.views[p.data_ptr()])
                if (p is not None and p.requires_grad) else None for p in ps])
        self.span = arena.span(live)
        self._granted = {}
        self._plan = plan

    def granted(self, no_dx):
        keys = self._granted.get(no_dx)
        if keys is None:
            keys = frozenset(self.keys - _stack_unused_keys(self._plan, no_dx))
            self._granted[no_dx] = keys
        return keys


def _stack_unused_keys(plan, no_dx):
    """data_ptrs of the parameters that cannot influence the loss in a stacked
    pass (same rules as egnn_layer_backward): every edge gate (no incoming
    messages), the coordinate MLP of a layer that does not update coordinates
    or -- the last layer -- whose coordinates nobody consumes."""
    per = len(_cabi.PARAM_FIELDS)
    L = len(plan.layers)
    drop = set()
    for i, layer in enumerate(plan.layers):
        unused = ['edge_gate']
        if not layer.use_coords or (no_dx and i == L - 1):
            unused += ['coord_w1', 'coord_b1', 'coord_w2']
        for name in unused:
            p = plan.params[i * per + _cabi.PARAM_FIELDS.index(name)]
            if p is not None:
                drop.add(p.data_ptr())
    return drop


def egnn_stack_backward_lean(ctx, d_h, d_x):
    """Backward of _EGNNStackLeanFn.  Parameter gradients go into the gradient
    arena (steady state of `backprop()`: cached pointer block, no per-parameter
    Python work), or are accumulated into `p.grad` here when there is no arena
    or it does not hold every parameter."""
    plan, csr = ctx.plan, ctx.csr
    layers = plan.layers
    L, per = len(layers), len(_cabi.PARAM_FIELDS)
    H, X, ws = ctx.H, ctx.X, ctx.ws
    n, e = csr.n_nodes, csr.n_edges
    dev = H.device
    d_h = torch.zeros_like(H[L]) if d_h is None else d_h.contiguous().float()
    no_dx = d_x is None
    d_x = None if no_dx else d_x.contiguous().float()
    csc_ptr, csc_eid = csr.csc()
    arena = ARENA
    gp = None
    if arena is not None:
        gp = plan.grad_plans.get(id(arena))
        if gp is None or gp.arena_ref() is not arena:
            gp = _StackGradPlan(plan, arena)
            gp.arena_ref = _weak(arena)
            plan.grad_plans = {id(arena): gp}
        if not gp.ok or not arena.hand_out_all(gp.keys):
            gp = None
    flat, manual = None, []
    if gp is not None:
        gstructs = gp.gstructs
    else:
        # no arena (or not every parameter in it): zero-filled gradients of our
        # own, handed to `p.grad` below
        live = [(i, p) for i, p in enumerate(plan.params)
                if p is not None and p.requires_grad]
        flat = torch.zeros(sum(p.numel() for _, p in live) or 1,
                           dtype=torch.float32, device=dev)
        views, off = {}, 0
        for i, p in live:
            views[i] = flat[off:off + p.numel()]
            off += p.numel()
            manual.append((i, p))
        gstructs = (_cabi.LayerGrads * L)()
        for li in range(L):
            gstructs[li] = _cabi.LayerGrads(*[
                ptr(views.get(li * per + j)) for j in range(per)])
    d_h_in = torch.empty_like(H[0])
    d_x_in = torch.empty_like(X[0])
    nbytes = int(lib().pvs_egnn_stack_bwd_workspace_bytes(n, e, L, plan.cfgs))
    bws = _cabi.scratch('stack_bwd', nbytes, dev)
    g = csr.c_struct()
    with torch.cuda.device(dev):
        check(lib().pvs_egnn_stack_bwd(
            C.byref(g), ptr(csc_ptr), ptr(csc_eid), L, plan.cfgs, plan.pstructs,
            gstructs, ptr(H), ptr(X), ptr(ws), C.c_int64(ctx.stride), ptr(d_h),
            ptr(d_x), ptr(d_h_in), ptr(d_x_in), ptr(bws), C.c_int64(bws.numel()),
            stream()), 'pvs_egnn_stack_bwd')
    if gp is not None:
        if arena.reduce_in_backward:
            arena.reduce_async(*gp.span)
        arena.grant_all(gp.granted(no_dx))
    else:
        drop = _stack_unused_keys(plan, no_dx)
        with torch.no_grad():
            for i, p in manual:
                if p.data_ptr() in drop:
                    continue
                gview = views[i].view(p.shape)
                p.grad = gview if p.grad is None else p.grad + gview
    return (None, None, d_h_in, d_x_in, None)


def _weak(obj):
    import weakref
    return weakref.ref(obj)


def linear_backward(ctx, d_out):
    inp, w, out = ctx.saved_tensors
    bias = ctx.bias_ref
    d_out = d_out.contiguous().float()
    rows, ki = inp.shape
    ko = w.shape[0]
    if ko > 64:
        raise NotImplementedError('linear backward supports at most 64 '
                                  'output features')
    need_in = ctx.needs_input_grad[0]
    d_in = torch.empty_like(inp) if need_in else None
    arena = ARENA
    d_w = arena.grad_view(w) if arena is not None else None
    w_in_arena = d_w is not None
    if d_w is None:
        d_w = torch.zeros_like(w)
    d_b, b_in_arena = None, False
    if ctx.has_bias:
        d_b = arena.grad_view(bias) if arena is not None else None
        b_in_arena = d_b is not None
        if d_b is None:
            d_b = torch.zeros(ko, dtype=torch.float32, device=inp.device)
    nbytes = int(lib().pvs_linear_bwd_workspace_bytes(rows, ki, ko))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=inp.device)
    with torch.cuda.device(inp.device):
        check(lib().pvs_linear_bwd(
            ptr(inp), ki, rows, ki, ptr(w), ki, ptr(bias), ko,
            _cabi.ACT[ctx.act], ptr(d_out), ko, ptr(d_in), ki, ptr(d_w), ki,
            ptr(d_b), ptr(ws), C.c_int64(ws.numel()), stream()),
            'pvs_linear_bwd')
    if w_in_arena:
        arena.grant(w)
        d_w = None
    if b_in_arena:
        arena.grant(bias)
        d_b = None
    return d_in, d_w, d_b, None


def mean_pool_backward(ctx, d_pooled):
    (graph_ptr,) = ctx.saved_tensors
    d_pooled = d_pooled.contiguous().float()
    d_h = torch.zeros((ctx.n_nodes, ctx.k), dtype=torch.float32,
                      device=d_pooled.device)
    with torch.cuda.device(d_pooled.device):
        check(lib().pvs_mean_pool_bwd(ptr(d_pooled), ptr(graph_ptr),
                                      ctx.n_graphs, ctx.k, ptr(d_h), stream()),
              'pvs_mean_pool_bwd')
    return d_h, None, None
