"""Seeded sweep of the training backward against float64 autograd.

A. Every generated model and batch is trained for one step in each math mode:
   the gradients of a weighted sum of the scores (every parameter, the input
   coordinates and the input features) are compared with torch autograd of
   the CPU oracle in float64, on the edge list the device built.  The
   per-layer, stacked and lean passes, the capacity-bounded graph and a rerun
   must give bit-identical gradients.
B. pvs_egnn_layer_bwd through the C ABI against the float64 vector-Jacobian
   product of one layer, checking the header's contract: outputs overwritten
   (NaN-filled before the call, workspace too), parameter gradients
   accumulated, NULL members skipped without changing the others.
C. relu attention away from its kink, and a backward that runs after
   set_math() still differentiates the function the forward evaluated.

Bounds, per math mode and part, on every gradient tensor and on every row and
column of each weight matrix, of the coordinate and of the feature gradient:

    tensor:  max|g - r| <= rtol * max|r_tensor| + ATOL
    slice:   max|g - r| <= srtol * max(max|r_slice|, SLICE_FLOOR * max|r_tensor|) + ATOL

A zeroed or mis-scaled row or column fails this even when its values are
small next to the tensor's largest.  Single-pass bf16 rounds every GEMM
operand to bf16; its rtol per tensor is the larger of BF16_FLOOR and a
multiple of the change that rounding the operands makes in the float64
gradient (as the forward sweep does for the scores), and it has no slice
bound.  The contract checks of part B hold in every mode.

`test_grad_sweep_reaches_every_switch` (no GPU) checks that the generator
still reaches the shapes that select different code paths.
"""
import ctypes as C
import functools
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from tests import gpu_helpers as gh
from tests import helpers
from tests.test_gpu_layer_paths import OPTIONS as LAYER_PATH_OPTIONS
from tests.test_gpu_sweep import DIM_INPUTS, HEADS, KINDS, SMALLK_ROWS, _batch

MATHS = ('fp32', 'bf16x3', 'fp16x2', 'bf16')
WIDTHS = (1, 4, 31, 32, 33, 63, 64)
N_CASES = 40
# relu attention: att_mlp (and node_att_mlp) bias shifted by +-3 and weight
# scaled by 0.1, so that every pre-activation sits far from the kink: all on,
# all off
RELU_SHIFTS = {N_CASES: 3.0, N_CASES + 1: -3.0}
# rtol per tensor (A: model sweep, B: one layer through the C ABI).  Measured
# worst against float64, A / B: fp32 2.0e-4 (a k = 1 GraphNorm weight) /
# 3.8e-4 (k = 1), bf16x3 1.3e-3 / 2.8e-3 (a coordinate MLP at gain 1000),
# fp16x2 4.7e-3 / 3.6e-2.  B's fp16x2 worst is edge_mlp.2 of a k = 1
# permutation-invariant layer: a 1 x 1 gradient whose float64 terms sum to
# 1/247 of their absolute sum, so 1.5e-4 of rounding per term.
RTOL = {'fp32': 4e-4, 'bf16x3': 3e-3, 'fp16x2': 1e-2}
LAYER_RTOL = {'fp32': 8e-4, 'bf16x3': 5e-3, 'fp16x2': 5e-2}
# bf16: max(BF16_FLOOR, factor x the bf16 probe).  A's probe rounds the
# parameters and input features (measured worst 6.6e-2 where the floor holds);
# B's rounds every GEMM operand too, and the error reached 2.1 x that probe
# (softmax attention weight at a hub).
BF16_FLOOR = 1e-1
BF16_PROBE_FACTOR = 2.0
LAYER_BF16_PROBE_FACTOR = 3.0
SLICE_FLOOR = 1e-2
# rtol of a row or column against max(its own largest, SLICE_FLOOR x the
# tensor's): a row sums terms that cancel more than the tensor's do.  Each
# still fails a zeroed or doubled row.  Measured worst, A / B: fp32 1.2e-3 /
# 1.6e-3, bf16x3 3.8e-2 (one element of a k = 1 head) / 1.9e-2, fp16x2
# 9.5e-2 / 2.0e-1 (softmax attention at a hub).  bf16 has none: a row's error
# reaches 0.85 of its largest value there (GraphNorm layer at a hub), so only
# the per-tensor bound applies.
SLICE_RTOL = {'fp32': 3e-3, 'bf16x3': 1e-1, 'fp16x2': 2e-1, 'bf16': None}
LAYER_SLICE_RTOL = {'fp32': 3e-3, 'bf16x3': 5e-2, 'fp16x2': 3e-1, 'bf16': None}
ATOL = 1e-12
ATT_ACTS = ('sigmoid', 'tanh', 'silu')


# ---------------------------------------------------------------------------
# A. case generator (numpy only: the coverage test runs without a GPU)
# ---------------------------------------------------------------------------
def _case(seed):
    rng = np.random.default_rng(9000 + seed)
    relu = seed in RELU_SHIFTS
    if relu:
        kind, k, head = 'ragged', 32, 'fc'
    else:
        kind = KINDS[seed % len(KINDS)]
        k = WIDTHS[seed % len(WIDTHS)]
        head = HEADS[(seed // len(HEADS) + seed) % len(HEADS)]
    if kind.startswith('n40'):      # the streaming embedding needs ki <= 32
        dim_input = int(rng.choice([d for d in DIM_INPUTS if d <= 32]))
    else:
        dim_input = int(DIM_INPUTS[(seed // len(DIM_INPUTS) + seed) % len(DIM_INPUTS)])
    multitask = head.startswith('mt_')
    att = bool(rng.integers(0, 2))
    kw = dict(dim_input=dim_input, k=k,
              dim_output=int(rng.choice([1, 3])),
              num_layers=int(rng.integers(1, 5)),
              residual=bool(rng.integers(0, 2)),
              edge_residual=bool(rng.integers(0, 2)),
              edge_attention=att,
              softmax_attention=att and bool(rng.integers(0, 2)),
              node_attention=bool(rng.integers(0, 2)),
              normalize=bool(rng.integers(0, 2)), tanh=bool(rng.integers(0, 2)),
              graphnorm=bool(rng.integers(0, 2)),
              update_coords=bool(rng.integers(0, 4) > 0),
              permutation_invariance=bool(rng.integers(0, 4) == 0),
              attention_activation_fn=str(rng.choice(ATT_ACTS)),
              final_softplus=head.endswith('softplus'))
    mode = int(rng.integers(0, 3))
    kw['gated_residual'] = mode == 1
    kw['rezero'] = mode == 2
    if multitask:
        kw['edge_attention_first_only'] = bool(rng.integers(0, 2))
        kw['node_attention_final_only'] = bool(rng.integers(0, 2))
    else:
        kw['multi_fc'] = head.startswith('multi_fc')
    shift = RELU_SHIFTS.get(seed, 0.0)
    if relu:
        kw.update(edge_attention=True, softmax_attention=False,
                  node_attention=shift > 0, attention_activation_fn='relu',
                  num_layers=2, residual=True)
    task = 'classification' if head == 'mt_pose' else 'regression'
    parts, inter, intra = _batch(kind, rng, seed)
    coords = np.concatenate([p[0] for p in parts])
    bp = np.concatenate([p[1] for p in parts])
    sizes = [len(p[0]) for p in parts]
    feats = rng.normal(size=(len(coords), dim_input)).astype(np.float32)
    n_out = len(sizes) * (1 if head == 'mt_pose' else kw['dim_output'])
    return SimpleNamespace(
        seed=seed, kind=kind, head=head, kw=kw, multitask=multitask, task=task,
        coords=coords, bp=bp, feats=feats, sizes=sizes,
        cptr=np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32),
        inter=inter, intra=intra,
        capacity='auto' if seed % 3 == 0 else None,
        gate=float(rng.uniform(0.2, 0.6)), att_shift=shift,
        # loss weights: distinct per complex and output, so that gradients
        # swapped between complexes fail
        weights=np.linspace(0.5, 1.5, n_out) * np.where(np.arange(n_out) % 2, -1.0, 1.0),
        # a parameter whose reference gradient must be nonzero: the first
        # EGNN layer's, unless no message can reach the scores
        live='layers.0.m.weight' if (kind == 'no_edges' or shift < 0)
        else 'layers.1.edge_mlp.0.weight')


def _seeds():
    return list(range(N_CASES)) + sorted(RELU_SHIFTS)


def _params():
    out = []
    for seed in _seeds():
        c = _case(seed)
        for math in MATHS:
            out.append(pytest.param(
                seed, math, id=f"{seed}-{math}-{c.kind}-k{c.kw['k']}-{c.head}"))
    return out


# ---------------------------------------------------------------------------
# bounds
# ---------------------------------------------------------------------------
def _compare(name, got, ref, rtol, srtol, what, floor=0.0):
    """Assert the per-tensor bound (rtol) and the per-row/column bound
    (srtol, at least rtol); returns (error
    relative to the tensor's scale, worst slice error relative to its slice
    scale).  floor: least scale of the tensor, SLICE_FLOOR times the largest
    gradient of its layer (a gradient that is zero in exact arithmetic, such
    as a softmax logit's bias, is held to the rounding of its neighbours)."""
    assert got is not None, (name, what)
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, (name, got.shape, ref.shape, what)
    assert np.isfinite(got).all(), (name, 'non-finite gradient', what)
    if ref.size == 0:
        return 0.0, 0.0
    diff = np.abs(got - ref)
    scale = max(float(np.abs(ref).max()), floor)
    err = float(diff.max())
    assert err <= rtol * scale + ATOL, \
        f'{name}: err {err:.3e} > {rtol:.1e} * {scale:.3e} ({what})'
    worst = 0.0
    if ref.ndim == 2 and srtol is not None:
        srtol = max(rtol, srtol)
        for axis, label in ((1, 'row'), (0, 'column')):
            d = diff.max(axis=axis)
            den = np.maximum(np.abs(ref).max(axis=axis), SLICE_FLOOR * scale)
            bad = np.flatnonzero(d > srtol * den + ATOL)
            assert bad.size == 0, \
                (f'{name}: {label} {int(bad[0])} err {d[bad[0]]:.3e} > '
                 f'{srtol:.1e} * {den[bad[0]]:.3e} ({what})')
            worst = max(worst, float((d / np.maximum(den, 1e-300)).max()))
    return err / max(scale, 1e-300), worst


def _floors(ref):
    """SLICE_FLOOR x the largest gradient of each tensor's layer (prefix up
    to the module index, e.g. 'layers.2.'); inputs are their own layer."""
    top = {}

    def layer(name):
        parts = name.split('.')
        return '.'.join(parts[:2]) if parts[0] == 'layers' else parts[0]
    for name, r in ref.items():
        if r is not None and r.size:
            top[layer(name)] = max(top.get(layer(name), 0.0), float(np.abs(r).max()))
    return {name: SLICE_FLOOR * top.get(layer(name), 0.0) for name in ref}


def _rtols(math, ref, ref_bf16, table=RTOL, factor=BF16_PROBE_FACTOR):
    """rtol per gradient name.  bf16: max(BF16_FLOOR, factor x the change
    that rounding the operands to bf16 makes in the float64 gradient)."""
    if math != 'bf16':
        return {name: table[math] for name in ref}
    out = {}
    for name, r in ref.items():
        if r is None or r.size == 0 or not np.abs(r).max():
            out[name] = BF16_FLOOR
            continue
        probe = float(np.abs(ref_bf16[name] - r).max() / np.abs(r).max())
        out[name] = max(BF16_FLOOR, factor * probe)
    return out


# ---------------------------------------------------------------------------
# A. float64 reference (CPU)
# ---------------------------------------------------------------------------
def reference_grads(c, state_dict, feats, pos, edge_index, edge_attr, batch,
                    bf16_operands=False):
    """float64 torch autograd of oracle.model_forward for the loss
    sum_b w_b out_b.  -> {parameter name: grad or None, 'pos': ..,
    'feats': ..} as float64 numpy arrays."""
    from oracle import egnn_oracle

    def leaf(t):
        t = t.detach().cpu()
        if bf16_operands:
            t = t.to(torch.bfloat16)
        return t.double().requires_grad_(True)
    sd = {k: leaf(v) if v.is_floating_point() else v.detach().cpu()
          for k, v in state_dict.items()}
    x = leaf(feats)
    p = pos.detach().cpu().double().requires_grad_(True)
    out, _ = egnn_oracle.model_forward(
        sd, x, edge_index.cpu(), p, edge_attr.cpu(), batch.cpu(),
        num_layers=c.kw['num_layers'], multitask=c.multitask,
        model_task=c.task, final_softplus=c.kw['final_softplus'],
        **helpers.oracle_kwargs(c.kw))
    (out.reshape(-1) * torch.from_numpy(c.weights)).sum().backward()
    grads = {k: (None if v.grad is None else v.grad.numpy())
             for k, v in sd.items() if isinstance(v, torch.Tensor) and v.requires_grad}
    grads['pos'] = None if p.grad is None else p.grad.numpy()
    grads['feats'] = None if x.grad is None else x.grad.numpy()
    return grads, out.detach()


def _model(c):
    model = gh.build_model(c.kw, multitask=c.multitask, seed=c.seed,
                           coord_gain=1.0)
    if c.multitask:
        model.set_task(c.task)
    g = torch.Generator().manual_seed(c.seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if 'gate_parameter' in name:
                p.fill_(c.gate)
            if 'node_mlp.1.' in name and c.kw['graphnorm']:
                p.add_(0.2 * torch.randn(p.shape, generator=g).to(p.device))
            if c.att_shift and 'att_mlp.0.' in name:
                if name.endswith('weight'):
                    p.mul_(0.1)
                else:
                    p.add_(c.att_shift)
    return model


def _graph(c, capacity=None):
    import pointvs_b200 as pv
    return pv.PackedBatch.from_arrays(c.coords, c.bp, c.feats, c.cptr, c.inter,
                                      c.intra, edge_capacity=capacity)


@functools.lru_cache(maxsize=None)
def _reference(seed, bf16_operands=False):
    c = _case(seed)
    graph = _graph(c)
    model = _model(c)
    grads, _ = reference_grads(c, model.state_dict(), graph.x, graph.pos,
                               graph.edge_index, graph.edge_attr, graph.batch,
                               bf16_operands)
    return grads, graph.pvs_csr.n_edges


# ---------------------------------------------------------------------------
# A. GPU side
# ---------------------------------------------------------------------------
PATHS = ('per_layer', 'stacked', 'lean')


def _select(monkeypatch, model, path):
    monkeypatch.setenv('PVS_STACK_TRAIN', {'per_layer': '0', 'stacked': '1',
                                           'lean': ''}[path])
    model._lean_training = path == 'lean'


def _train_step(c, model, graph, pos0, feats0):
    """One forward and backward of sum_b w_b out_b -> gradients by name."""
    model.zero_grad(set_to_none=True)
    graph.pos = pos0.clone().requires_grad_(True)
    graph.x = feats0.clone().requires_grad_(True)
    out = model(graph).reshape(-1)
    w = torch.from_numpy(c.weights).float().to(out.device)
    (out * w).sum().backward()
    grads = {n: (None if p.grad is None else p.grad.detach().cpu().numpy())
             for n, p in model.named_parameters()}
    grads['pos'] = None if graph.pos.grad is None else graph.pos.grad.cpu().numpy()
    grads['feats'] = None if graph.x.grad is None else graph.x.grad.cpu().numpy()
    return grads


def _bits(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _assert_same_bits(base, other, tag, what):
    assert base.keys() == other.keys()
    for name, g in base.items():
        assert (g is None) == (other[name] is None), (tag, name, what)
        if g is not None:
            assert np.array_equal(_bits(g), _bits(other[name])), (tag, name, what)


@pytest.mark.gpu
@pytest.mark.parametrize('seed,math', _params())
def test_grad_sweep_vs_float64_autograd(seed, math, monkeypatch):
    c = _case(seed)
    ref, n_edges = _reference(seed)
    ref_bf16 = _reference(seed, True)[0] if math == 'bf16' else None
    what = (f'seed {seed} {math} {c.kind} sizes={c.sizes} E={n_edges} '
            f'{c.head} {c.kw}')
    assert np.abs(ref[c.live]).max() > 0, ('vacuous case', c.live, what)
    if c.att_shift:     # relu attention: every edge on (+3) or off (-3)
        assert _relu_attention_state(seed) == (c.att_shift > 0), what

    model = _model(c).set_math(math).train()
    model.set_record_side_channels(False)
    layers = list(model.layers)[1:]
    graphs = [_graph(c)]
    if c.capacity is not None:
        graphs.append(_graph(c, c.capacity))
    pos0, feats0 = graphs[0].pos.clone(), graphs[0].x.clone()

    _select(monkeypatch, model, 'per_layer')
    got = _train_step(c, model, graphs[0], pos0, feats0)
    runs = [('rerun', graphs[0])]
    if len(graphs) > 1:
        runs.append(('capacity-bounded graph', graphs[1]))
    for tag, g in runs:
        _assert_same_bits(got, _train_step(c, model, g, pos0, feats0), tag, what)
    for path in ('stacked', 'lean'):
        _select(monkeypatch, model, path)
        with torch.enable_grad():
            ok = model._stack_ok(layers, feats0.clone().requires_grad_(True),
                                 False)
        assert ok == (not c.kw['edge_residual']), (path, what)
        if ok:
            _assert_same_bits(got, _train_step(c, model, graphs[0], pos0, feats0),
                              path, what)

    # against float64
    rtols = _rtols(math, ref, ref_bf16)
    floors = _floors(ref)
    errs = {'param': (0.0, ''), 'pos': (0.0, ''), 'feats': (0.0, '')}
    worst_slice = 0.0
    for name, r in ref.items():
        if r is None:
            assert got[name] is None, (name, 'has a gradient the reference lacks', what)
            continue
        e, s = _compare(name, got[name], r, rtols[name], SLICE_RTOL[math], what,
                        floors[name])
        key = name if name in ('pos', 'feats') else 'param'
        if e >= errs[key][0]:
            errs[key] = (e, name)
        worst_slice = max(worst_slice, s)
    assert set(got) == set(ref), (set(got) ^ set(ref), what)
    print(f"GRADSWEEP seed={seed} math={math} k={c.kw['k']} kind={c.kind} "
          f"param_err={errs['param'][0]:.3e} ({errs['param'][1]}) "
          f"pos_err={errs['pos'][0]:.3e} feat_err={errs['feats'][0]:.3e} "
          f"slice_err={worst_slice:.3e} "
          f"rtol={min(rtols.values()):.1e}..{max(rtols.values()):.1e} "
          f"slice_floor={SLICE_FLOOR:.0e}")


@functools.lru_cache(maxsize=None)
def _relu_attention_state(seed):
    """True if every relu attention value of the float64 oracle is positive,
    False if every one is zero (None: mixed)."""
    c = _case(seed)
    graph = _graph(c)
    model = _model(c)
    trace = []
    gh.oracle_forward(model, c.kw, graph, multitask=c.multitask, task=c.task,
                      dtype=torch.float64, trace=trace)
    att = torch.cat([t[name].reshape(-1) for t in trace
                     for name in ('att_val', 'node_att_val') if name in t])
    if bool((att > 1e-3).all()):
        return True
    if bool((att == 0).all()):
        return False
    return None


# ---------------------------------------------------------------------------
# C. set_math() between the forward and the backward
# ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('graphnorm', (False, True))
@pytest.mark.parametrize('path', PATHS)
def test_backward_after_set_math_differentiates_the_forward(path, graphnorm,
                                                            monkeypatch):
    """Forward in bf16, set_math('fp32'), backward: the gradients are those
    of the bf16 forward, bit for bit (GraphNorm: the backward recomputes the
    layer instead of reading the forward's workspace)."""
    kw = dict(dim_input=13, dim_output=1, k=32, num_layers=3,
              edge_attention=True, node_attention=True, residual=True,
              normalize=True, tanh=True, graphnorm=graphnorm)
    results = []
    for switch in (False, True):
        model = gh.build_model(kw, seed=11, coord_gain=1.0).train()
        model.set_math('bf16').set_record_side_channels(False)
        _select(monkeypatch, model, path)
        graph = gh.synthetic_graph(910, 3, 200, 15, ragged=True)
        graph.pos = graph.pos.clone().requires_grad_(True)
        out = model(graph)
        if switch:
            model.set_math('fp32')
        (out.reshape(-1) * torch.tensor([1.0, -0.5, 2.0], device='cuda')).sum().backward()
        grads = {n: p.grad.clone() for n, p in model.named_parameters()
                 if p.grad is not None}
        grads['pos'] = graph.pos.grad.clone()
        results.append(grads)
    plain, switched = results
    assert plain.keys() == switched.keys()
    for name in plain:
        assert torch.equal(plain[name], switched[name]), name


# ---------------------------------------------------------------------------
# B. pvs_egnn_layer_bwd through the C ABI
# ---------------------------------------------------------------------------
LAYER_WIDTHS = (1, 4, 31, 33, 63, 64)
# layer options -> (EGNNLayer flags, d_m_out given)
LAYER_OPTIONS = dict(LAYER_PATH_OPTIONS)
LAYER_OPTIONS.update({
    'gated': (dict(edge_residual=True, gated_residual=True, edge_attention=True,
                   attention_activation_fn='tanh'), True),
    'rezero': (dict(edge_residual=True, rezero=True, node_attention=True,
                    attention_activation_fn='silu', normalize=True), True),
    'perm_invariant': (dict(permutation_invariance=True, tanh=True), False),
})


def _graph_spec(name):
    """-> n, row, col, attr (int64 numpy, any order), coordinates."""
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == 'ragged':
        from oracle import radius_graph as rg
        from pointvs_b200.synthetic import synthetic_batch
        coords, bp, _, cptr = synthetic_batch(720, 3, 110, 12, ragged=True)
        rows, cols, attrs = [], [], []
        for lo, hi in zip(cptr[:-1], cptr[1:]):
            _, r, cc, a = rg.radius_graph(coords[lo:hi], bp[lo:hi], 4.0, 4.0)
            rows.append(r + lo), cols.append(cc + lo), attrs.append(a)
        return (len(coords), np.concatenate(rows), np.concatenate(cols),
                np.concatenate(attrs), coords)
    if name == 'hub':       # node 0 hears 150 others, which all hear it
        n = 160
        others = np.arange(1, 151)
        extra = rng.integers(1, n, 40)
        row = np.concatenate([np.zeros(150, np.int64), others, extra])
        col = np.concatenate([others, np.zeros(150, np.int64),
                              1 + (extra + rng.integers(0, n - 2, 40)) % (n - 1)])
    elif name in ('e256', 'e257'):      # a whole number of 128-edge tiles, +1
        n = 90
        e = int(name[1:])
        row = rng.integers(0, n, e)
        col = (row + rng.integers(1, n, e)) % n
    elif name == 'n1':
        n, row, col = 1, np.zeros(0, np.int64), np.zeros(0, np.int64)
    else:                               # 'e0': seven nodes, no edges
        n, row, col = 7, np.zeros(0, np.int64), np.zeros(0, np.int64)
    coords = rng.normal(size=(n, 3)) * 2.0
    return n, row.astype(np.int64), col.astype(np.int64), \
        rng.integers(0, 3, len(row)), coords


LAYER_GRAPHS = ('ragged', 'hub', 'e256', 'e257', 'n1', 'e0')


@functools.lru_cache(maxsize=None)
def _layer_graph(name):
    """Device CSR of the graph and its edges in CSR order (numpy)."""
    from pointvs_b200.graph import csr_from_edge_index
    n, row, col, attr, coords = _graph_spec(name)
    ei = torch.from_numpy(np.stack([row, col])).cuda()
    onehot = torch.nn.functional.one_hot(torch.from_numpy(attr).long(), 3).cuda()
    csr = csr_from_edge_index(ei, onehot, n)
    e = csr.n_edges
    order = csr.perm.long().cpu().numpy() if e else np.zeros(0, np.int64)
    return SimpleNamespace(csr=csr, n=n, e=e, row=row[order], col=col[order],
                           attr=attr[order], ei=ei, onehot=onehot,
                           x=coords.astype(np.float32))


def _layer_setup(k, option, spec_n, spec_e, seed):
    """CPU layer (parameters off their init) and float32 inputs."""
    from pointvs_b200 import EGNNLayer
    flags, give_dm = LAYER_OPTIONS[option]
    torch.manual_seed(seed)
    layer = EGNNLayer(k, k, k, edges_in_d=3, **flags)
    with torch.no_grad():
        for p in layer.parameters():
            p.add_(0.05 * torch.randn_like(p))
        layer.coord_mlp[2].weight.mul_(1000.0)
        for name, p in layer.named_parameters():
            if 'gate_parameter' in name:
                p.fill_(0.35)
    gen = torch.Generator().manual_seed(seed + 1)
    t = dict(h=torch.randn(spec_n, k, generator=gen),
             d_h=torch.randn(spec_n, k, generator=gen),
             d_x=torch.randn(spec_n, 3, generator=gen))
    if layer.edge_residual:
        t['m_prev'] = torch.randn(spec_e, k, generator=gen)
    if give_dm:
        t['d_m'] = torch.randn(spec_e, k, generator=gen)
    return layer, t


def layer_vjp(layer, t, row, col, attr, x, bf16_operands=False):
    """float64 VJPs of oracle.layer_forward for the losses <d_h, h_out> +
    <d_x, x_out> + <d_m, m_out> (key True) and the same without the x_out
    term (key False: d_x_out NULL).  -> {key: {name: grad}}; parameter names
    as in _cabi.GRAD_FIELDS, inputs 'd_h_in', 'd_x_in', 'd_m_prev'.

    bf16_operands: the probe of the single-pass bf16 mode.  Besides the
    parameters and inputs, every Linear's input and weight is rounded to bf16,
    as that mode rounds every GEMM operand: inside one layer, the coordinate
    MLP (at gain 1000) turns the rounding of the messages it reads into most
    of its gradient's error."""
    if not bf16_operands:
        return _layer_vjp(layer, t, row, col, attr, x, False)
    import torch.nn.functional as F
    linear = F.linear

    def bf16_linear(inp, w, b=None):
        r = lambda v: v.to(torch.bfloat16).double()
        return linear(r(inp), r(w), b)
    F.linear = bf16_linear
    try:
        return _layer_vjp(layer, t, row, col, attr, x, True)
    finally:
        F.linear = linear


def _layer_vjp(layer, t, row, col, attr, x, bf16_operands):
    from oracle import egnn_oracle
    from pointvs_b200 import _cabi

    def leaf(v):
        v = v.detach().cpu()
        if bf16_operands:
            v = v.to(torch.bfloat16)
        return v.double().requires_grad_(True)
    sd = {name: leaf(v) for name, v in layer.state_dict().items()}
    h = leaf(t['h'])
    xx = torch.from_numpy(x).double().requires_grad_(True)
    m_prev = leaf(t['m_prev']) if 'm_prev' in t else None
    cfg = egnn_oracle.LayerConfig(
        residual=layer.residual, edge_residual=layer.edge_residual,
        edge_attention=layer.edge_attention, normalize=layer.normalize,
        tanh=layer.tanh, graphnorm=layer.graphnorm,
        update_coords=layer.use_coords,
        permutation_invariance=layer.permutation_invariance,
        node_attention=layer.node_attention,
        attention_activation_fn=layer.attention_activation_fn,
        gated_residual=layer.gated_residual, rezero=layer.rezero,
        softmax_attention=layer.softmax_attention)
    ea = torch.nn.functional.one_hot(torch.from_numpy(attr).long(), 3)
    h_out, x_out, m_out, _ = egnn_oracle.layer_forward(
        sd, '', cfg, h, torch.from_numpy(row), torch.from_numpy(col), xx, ea,
        m_prev)
    loss = (h_out * t['d_h'].double()).sum()
    if 'd_m' in t:
        loss = loss + (m_out * t['d_m'].double()).sum()
    names = [n for n in _param_names(layer)]
    inputs = [sd[n] for n in names if n is not None] + [h, xx] + \
        ([m_prev] if m_prev is not None else [])
    shapes = [v.shape for v in inputs]
    out = {}
    for with_dx in (False, True):
        if with_dx:
            loss = loss + (x_out * t['d_x'].double()).sum()
        got = torch.autograd.grad(loss, inputs, allow_unused=True,
                                  retain_graph=not with_dx)
        got = [np.zeros(s) if v is None else v.numpy()
               for v, s in zip(got, shapes)]
        res, i = {}, 0
        for field, n in zip(_cabi.GRAD_FIELDS, names):
            if n is not None:
                res[field] = got[i]
                i += 1
        res['d_h_in'], res['d_x_in'] = got[i], got[i + 1]
        if m_prev is not None:
            res['d_m_prev'] = got[i + 2]
        out[with_dx] = res
    return out


def _param_names(layer):
    """state_dict name of each pvs_layer_params member (None if absent)."""
    ids = {id(p): n for n, p in layer.named_parameters()}
    return [None if p is None else ids[id(p)] for p in layer.param_list()]


@functools.lru_cache(maxsize=None)
def _layer_reference(k, option, gname, bf16_operands):
    g = _layer_graph(gname)
    layer, t = _layer_setup(k, option, g.n, g.e, seed=31 * k + len(option))
    return layer_vjp(layer, t, g.row, g.col, g.attr, g.x, bf16_operands)


def _nan(shape, dev='cuda'):
    return torch.full(shape, float('nan'), dtype=torch.float32, device=dev)


def _layer_call(layer, g, t, grads0, d_x_on, math, drop=None):
    """pvs_egnn_layer_bwd with NaN-filled outputs and workspace and gradient
    members pre-filled with grads0 (member `drop` NULL) -> outputs (numpy)."""
    from pointvs_b200 import _cabi
    from pointvs_b200._cabi import check, ptr, stream
    lib = _cabi.lib()
    n, e, k = g.n, g.e, layer.hidden_nf
    cfg = layer.c_config()
    cfg.math = _cabi.MATH[math]
    params = [None if p is None else p.detach().cuda().contiguous()
              for p in layer.param_list()]
    pstruct = _cabi.LayerParams(*[ptr(p) for p in params])
    grads = {f: (None if (g0 is None or f == drop) else torch.from_numpy(g0).cuda())
             for f, g0 in grads0.items()}
    gstruct = _cabi.LayerGrads(*[ptr(grads[f]) for f in _cabi.GRAD_FIELDS])
    dev = {name: v.cuda().contiguous() for name, v in t.items()}
    x = torch.from_numpy(g.x).cuda()
    d_h_in, d_x_in = _nan((n, k)), _nan((n, 3))
    d_m_prev = _nan((e, k)) if 'm_prev' in dev else None
    csc_ptr, csc_eid = g.csr.csc()
    gs = g.csr.c_struct()
    nbytes = int(lib.pvs_egnn_layer_bwd_workspace_bytes(n, e, C.byref(cfg)))
    ws = torch.full((max(1, nbytes),), 0xFF, dtype=torch.uint8, device='cuda')
    check(lib.pvs_egnn_layer_bwd(
        C.byref(gs), ptr(csc_ptr), ptr(csc_eid), C.byref(cfg), C.byref(pstruct),
        ptr(dev['h']), ptr(x), ptr(dev.get('m_prev')), ptr(dev['d_h']),
        ptr(dev['d_x']) if d_x_on else None, ptr(dev.get('d_m')),
        ptr(d_h_in), ptr(d_x_in), ptr(d_m_prev), C.byref(gstruct), ptr(ws),
        C.c_int64(nbytes), stream()), 'pvs_egnn_layer_bwd')
    torch.cuda.synchronize()
    out = {f: (None if v is None else v.cpu().numpy()) for f, v in grads.items()}
    out['d_h_in'] = d_h_in.cpu().numpy()
    out['d_x_in'] = d_x_in.cpu().numpy()
    if d_m_prev is not None:
        out['d_m_prev'] = d_m_prev.cpu().numpy()
    for name, v in out.items():     # nothing left unwritten, nothing read stale
        assert v is None or np.isfinite(v).all(), (name, 'not finite', math, k)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('k', LAYER_WIDTHS)
@pytest.mark.parametrize('math', MATHS)
def test_layer_bwd_contract_vs_float64(math, k):
    """Every option on every graph: a hub with more than 128 incoming edges,
    edge counts of 2 x 128 and one more, n = 1, E = 0 and a ragged batch.
    Every output is finite (they start as NaN, the workspace too); parameter
    gradients land on their starting values G0 as G0 + (what a zero start
    gives), and match float64 after subtracting G0; a NULL member changes no
    other output."""
    from pointvs_b200 import _cabi
    worst = worst_slice = 0.0
    for gname in LAYER_GRAPHS:
        g = _layer_graph(gname)
        for i, option in enumerate(LAYER_OPTIONS):
            layer, t = _layer_setup(k, option, g.n, g.e, seed=31 * k + len(option))
            refs = _layer_reference(k, option, gname, False)
            refs_bf16 = _layer_reference(k, option, gname, True) \
                if math == 'bf16' else {True: None, False: None}
            rng = np.random.default_rng(i)
            grads0 = {f: (None if p is None else
                          rng.normal(size=tuple(p.shape)).astype(np.float32))
                      for f, p in zip(_cabi.GRAD_FIELDS, layer.param_list())}
            what = f'{math} k={k} {option} graph={gname} n={g.n} E={g.e}'
            full = None
            for d_x_on in (True, False):
                got = _layer_call(layer, g, t, grads0, d_x_on, math)
                ref = refs[d_x_on]
                rtols = _rtols(math, ref, refs_bf16[d_x_on], LAYER_RTOL,
                                LAYER_BF16_PROBE_FACTOR)
                top = SLICE_FLOOR * max(float(np.abs(r).max()) for f, r in ref.items()
                                        if f in grads0 and r.size)
                for name, r in ref.items():
                    v = got[name]
                    if name in grads0:      # accumulated: subtract G0
                        v = v.astype(np.float64) - grads0[name]
                    e, sl = _compare(name, v, r, rtols[name], LAYER_SLICE_RTOL[math],
                                     f'{what} d_x_out={"set" if d_x_on else "NULL"}',
                                     top if name in grads0 else 0.0)
                    worst = max(worst, e)
                    worst_slice = max(worst_slice, sl)
                if d_x_on:
                    full = got
            # accumulated: from a zero start the same call gives S, from G0 it
            # gives G0 + S up to the rounding of that addition
            zero = _layer_call(layer, g, t, {f: (None if g0 is None else np.zeros_like(g0))
                                             for f, g0 in grads0.items()}, True, math)
            for f, g0 in grads0.items():
                if g0 is not None:
                    s_ = zero[f].astype(np.float64)
                    dev_ = np.abs(full[f] - (g0 + s_))
                    assert (dev_ <= 1e-6 * (np.abs(g0) + np.abs(s_)) + ATOL).all(), \
                        (f, 'not accumulated onto its starting value', what)
            # one member NULL: the others are unchanged, bit for bit
            present = [f for f, g0 in grads0.items() if g0 is not None]
            drop = present[(i + LAYER_GRAPHS.index(gname)) % len(present)]
            part = _layer_call(layer, g, t, grads0, True, math, drop=drop)
            assert part[drop] is None
            for name, v in full.items():
                if name != drop and v is not None:
                    assert np.array_equal(_bits(v), _bits(part[name])), \
                        (name, 'changed with', drop, 'NULL', what)
    print(f'LAYERBWD math={math} k={k} worst_err={worst:.3e} '
          f'slice_err={worst_slice:.3e}')


# ---------------------------------------------------------------------------
# coverage of the generator (no GPU)
# ---------------------------------------------------------------------------
def test_grad_sweep_reaches_every_switch():
    """The generator reaches every width in every math mode, every batch kind,
    head, input width and layer option.  Runs without a GPU, so narrowing the
    generator fails here."""
    from oracle import radius_graph as rg
    cases = [_case(s) for s in range(N_CASES)]
    assert len(_params()) == len(_seeds()) * len(MATHS)
    # every width, one short of and at the 32- and 64-wide tiles, in every mode
    assert {c.kw['k'] for c in cases} == set(WIDTHS)
    assert {c.kind for c in cases} == set(KINDS)
    for n in (SMALLK_ROWS - 1, SMALLK_ROWS, SMALLK_ROWS + 1):
        assert any(sum(c.sizes) == n and c.kw['dim_input'] <= 32 for c in cases), n
    for s in (1, 2, 3):
        assert any(s in c.sizes for c in cases), s
    assert {c.kw['dim_input'] for c in cases} == set(DIM_INPUTS)
    assert {c.kw['num_layers'] for c in cases} == {1, 2, 3, 4}
    assert {c.head for c in cases} == set(HEADS)
    assert {c.kw['dim_output'] for c in cases
            if c.head in ('fc', 'multi_fc', 'mt_affinity')} == {1, 3}
    assert {c.capacity for c in cases} == {'auto', None}
    for opt in ('residual', 'edge_residual', 'edge_attention',
                'softmax_attention', 'node_attention', 'normalize', 'tanh',
                'graphnorm', 'update_coords', 'permutation_invariance',
                'gated_residual', 'rezero'):
        assert {bool(c.kw[opt]) for c in cases} == {False, True}, opt
    for opt in ('edge_attention_first_only', 'node_attention_final_only'):
        placed = {c.kw[opt] for c in cases if c.multitask and c.kw['num_layers'] > 1
                  and c.kw[opt.split('_attention')[0] + '_attention']}
        assert placed == {False, True}, opt
    # stacked and lean passes (no edge residual) on a 1-layer stack and on
    # deeper ones, with GraphNorm, softmax attention and permutation invariance
    stackable = [c for c in cases if not c.kw['edge_residual']]
    assert {c.kw['num_layers'] for c in stackable} >= {1, 2}
    for opt in ('graphnorm', 'softmax_attention', 'permutation_invariance'):
        assert any(c.kw[opt] for c in stackable), opt
    assert {c.kw['attention_activation_fn'] for c in cases
            if c.kw['edge_attention'] and not c.kw['softmax_attention']} == set(ATT_ACTS)
    relu = [_case(s) for s in RELU_SHIFTS]
    assert {c.att_shift > 0 for c in relu} == {False, True}
    assert all(c.kw['attention_activation_fn'] == 'relu' for c in relu)

    def in_degrees(c):
        deg = np.zeros(len(c.coords), dtype=np.int64)
        for lo, hi in zip(c.cptr[:-1], c.cptr[1:]):
            _, row, _, _ = rg.radius_graph(c.coords[lo:hi], c.bp[lo:hi],
                                           c.inter, c.intra)
            deg[lo:hi] = np.bincount(row, minlength=hi - lo)
        return deg

    # an empty edge list, edgeless complexes beside others, and a destination
    # with more than 300 incoming edges in a layer without softmax attention
    assert any(in_degrees(c).sum() == 0 for c in cases if c.kind == 'no_edges')
    for c in (c for c in cases if c.kind == 'edgeless'):
        deg = in_degrees(c)
        per = [deg[lo:hi].sum() for lo, hi in zip(c.cptr[:-1], c.cptr[1:])]
        assert 0 in per and deg.sum() > 0
    assert any(in_degrees(c).max() > 300 and not c.kw['softmax_attention']
               for c in cases if c.kind == 'dense')
    # part B: every option on graphs with a > 128-edge hub, 2 x 128 and 2 x 128
    # + 1 edges, one node, no edges
    specs = {name: _graph_spec(name) for name in LAYER_GRAPHS}
    assert np.bincount(specs['hub'][1]).max() > 128
    assert len(specs['e256'][1]) == 256 and len(specs['e257'][1]) == 257
    assert specs['n1'][0] == 1 and len(specs['e0'][1]) == 0
    assert {'gated', 'rezero', 'perm_invariant'} <= set(LAYER_OPTIONS)
    assert set(LAYER_PATH_OPTIONS) <= set(LAYER_OPTIONS)
