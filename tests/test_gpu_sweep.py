"""Seeded sweep of the scoring path and of the dense helpers against float64
references.

A. Every generated model and batch is scored through the per-layer path (side
   channels on) and through the one-call pass (`pvs_egnn_model_fwd`).  The two
   must agree bit for bit, scores and final coordinates, and the one-call
   result must hold DESIGN §2's per-mode bound against the CPU oracle in
   float64.  Widths 4..64 run in every math mode, 65..128 in the three
   tensor-core modes.  Capacity-bounded graphs must score bit for bit like
   the exactly sized graph.
B. The dense helpers of the C ABI (linear forward and backward, mean pool,
   batch -> graph offsets, exclusive scan, edge-packed tiles) against numpy
   float64 at the shapes that select their different code paths.

`test_sweep_reaches_every_switch` (no GPU) checks that the generator still
reaches the shapes that select those paths.
"""
import ctypes as C
import functools
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from tests import helpers
from tests import gpu_helpers as gh

TOL = {'fp32': 1e-4, 'bf16x3': 1e-4, 'fp16x2': 5e-4, 'bf16': 3e-2}
MATHS = ('fp32', 'bf16x3', 'fp16x2', 'bf16')
NARROW = (4, 31, 32, 33, 63, 64)        # every math mode
WIDE = (65, 72, 97, 127, 128)           # tensor-core modes only
KINDS = ('tiny', 'edgeless', 'n4095', 'ragged', 'n4096', 'dense', 'no_edges',
         'n4097')
HEADS = ('fc', 'fc_softplus', 'multi_fc', 'multi_fc_softplus', 'mt_pose',
         'mt_affinity', 'mt_affinity_softplus')
DIM_INPUTS = (1, 12, 13, 32, 33, 40)
N_CASES = 48
# the embedding takes the streaming kernel (linear_smallk_kernel) from this
# many rows on, when dim_input <= 32 and k <= 64 (egnn_fwd.cu:launch_linear)
SMALLK_ROWS = 4096


# ---------------------------------------------------------------------------
# A. case generator (numpy only: the coverage test runs without a GPU)
# ---------------------------------------------------------------------------
def _split(rng, total, parts, most=1400):
    while True:
        cuts = np.sort(rng.choice(np.arange(1, total), parts - 1, replace=False))
        sizes = np.diff(np.concatenate([[0], cuts, [total]]))
        if sizes.max() <= most:
            return [int(s) for s in sizes]


def _line(n, origin, spacing=8.0):
    """n atoms `spacing` A apart on a line: no edge at any cut-off used here."""
    c = np.zeros((n, 3))
    c[:, 0] = spacing * np.arange(n)
    c += origin
    bp = np.ones(n, dtype=np.int32)
    bp[0] = 0
    return c.astype(np.float32).astype(np.float64), bp


def _batch(kind, rng, seed):
    """-> parts [(coords, bp)], inter, intra."""
    from pointvs_b200.synthetic import synthetic_complex
    inter = float(rng.choice([2.5, 4.0, 5.5]))
    intra = float(rng.choice([1.5, 2.0, inter]))
    if kind == 'tiny':
        sizes = [int(s) for s in rng.permutation([1, 2, 3, 60])]
    elif kind == 'edgeless':
        sizes = [130, 'line5', 61]
    elif kind == 'no_edges':
        sizes = [1, 'line4', 1, 'line3']
    elif kind.startswith('n40'):
        sizes = _split(rng, int(kind[1:]), int(rng.integers(3, 6)))
    elif kind == 'ragged':
        sizes = [int(s) for s in rng.choice([61, 127, 130, 193, 257, 300],
                                            int(rng.integers(3, 6)))]
    elif kind == 'dense':
        # a 350-atom ball at a 12 A cut-off: central atoms see nearly every
        # other atom (> 300 incoming edges), beside a small complex
        sizes = [350, 17]
        inter = intra = 12.0
    parts = []
    for i, s in enumerate(sizes):
        if isinstance(s, str):
            parts.append(_line(int(s[4:]), origin=(0.0, 40.0 * i, 0.0)))
        else:
            c, bp, _ = synthetic_complex(1000 * seed + i, s, max(1, s // 10))
            parts.append((c, bp))
    return parts, inter, intra


def _case(seed):
    rng = np.random.default_rng(7000 + seed)
    kind = KINDS[seed % len(KINDS)]
    head = HEADS[seed % len(HEADS)]
    big = kind.startswith('n40')
    if big:     # both sides of the streaming-embedding switch: k <= 64, ki <= 32
        k = NARROW[(seed // len(KINDS) + seed % len(KINDS)) % len(NARROW)]
        dim_input = int(rng.choice([d for d in DIM_INPUTS if d <= 32]))
    else:
        # cycle through the widths over the other kinds, the wide ones twice
        # per cycle (they run in three modes only)
        others = [i for i, kd in enumerate(KINDS) if not kd.startswith('n40')]
        j = seed // len(KINDS) * len(others) + others.index(seed % len(KINDS))
        widths = NARROW + WIDE + WIDE
        k = widths[j % len(widths)]
        dim_input = int(rng.choice(DIM_INPUTS))
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
              attention_activation_fn=str(rng.choice(
                  ['sigmoid', 'tanh', 'silu', 'relu'])),
              final_softplus=head.endswith('softplus'))
    mode = int(rng.integers(0, 3))
    kw['gated_residual'] = mode == 1
    kw['rezero'] = mode == 2
    if multitask:
        kw['edge_attention_first_only'] = bool(rng.integers(0, 2))
        kw['node_attention_final_only'] = bool(rng.integers(0, 2))
    else:
        kw['multi_fc'] = head.startswith('multi_fc')
    task = 'classification' if head == 'mt_pose' else 'regression'
    parts, inter, intra = _batch(kind, rng, seed)
    coords = np.concatenate([p[0] for p in parts])
    bp = np.concatenate([p[1] for p in parts])
    sizes = [len(p[0]) for p in parts]
    feats = rng.normal(size=(len(coords), dim_input)).astype(np.float32)
    return SimpleNamespace(
        seed=seed, kind=kind, head=head, kw=kw, multitask=multitask, task=task,
        coords=coords, bp=bp, feats=feats, sizes=sizes,
        cptr=np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32),
        inter=inter, intra=intra,
        capacity='auto' if seed % 3 == 0 else None,
        gate=float(rng.uniform(0.2, 0.6)))


def _modes(k):
    return MATHS if k <= 64 else MATHS[1:]


def _params():
    out = []
    for seed in range(N_CASES):
        c = _case(seed)
        for math in _modes(c.kw['k']):
            out.append(pytest.param(
                seed, math, id=f"{seed}-{math}-{c.kind}-k{c.kw['k']}-{c.head}"))
    return out


# ---------------------------------------------------------------------------
# A. GPU side
# ---------------------------------------------------------------------------
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
    return model


def _graph(c, capacity=None):
    import pointvs_b200 as pv
    return pv.PackedBatch.from_arrays(c.coords, c.bp, c.feats, c.cptr, c.inter,
                                      c.intra, edge_capacity=capacity)


@functools.lru_cache(maxsize=None)
def _oracle(seed, bf16_operands=False):
    """float64 oracle scores and final coordinates of case `seed`, on the edge
    list the device built (the graph builder is checked bit-exact elsewhere).

    bf16_operands: the parameters and input features rounded to bf16 first.
    How far that moves the result measures how strongly the case amplifies
    the operand rounding of the single-pass bf16 mode."""
    c = _case(seed)
    graph = _graph(c)
    model = _model(c)
    x = graph.x
    if bf16_operands:
        with torch.no_grad():
            for p in model.parameters():
                p.copy_(p.to(torch.bfloat16).float())
        x = x.to(torch.bfloat16).float()
    cpu = SimpleNamespace(x=x, pos=graph.pos.clone(),
                          edge_index=graph.edge_index,
                          edge_attr=graph.edge_attr, batch=graph.batch)
    want, x_want = gh.oracle_forward(model, c.kw, cpu, multitask=c.multitask,
                                     task=c.task, dtype=torch.float64)
    return want.numpy().reshape(-1), x_want.numpy(), graph.pvs_csr.n_edges


def _tolerances(seed, math, want, x_want):
    """Bounds on the score error (relative to max |score|) and on the
    coordinates' scaled_err.  DESIGN §2's per-mode bound, except that in the
    single-pass bf16 mode a badly conditioned case may need more: that mode
    rounds every GEMM operand to bf16, the weights and the activations alike,
    so its error is bounded by twice the perturbation that rounding the
    weights and input features alone causes in the float64 oracle."""
    tol = TOL[math]
    if math != 'bf16':
        return tol, tol
    want_r, x_want_r, _ = _oracle(seed, bf16_operands=True)
    scale = max(1e-3, float(np.abs(want).max()))
    probe = float(np.abs(want_r - want).max()) / scale
    x_probe = helpers.scaled_err(x_want_r, x_want)
    return max(tol, 2.0 * probe), max(tol, 2.0 * x_probe)


def _score(model, graph, pos0, one_call):
    model.set_record_side_channels(not one_call)
    model.record_embed_coords = not one_call
    graph.pos = pos0.clone()
    with torch.no_grad():
        assert model._fast_path_ok() == one_call
        out = model(graph)
    return out.cpu().numpy().reshape(-1), graph.pos.cpu().numpy()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize('seed,math', _params())
def test_sweep_one_call_and_per_layer_vs_float64_oracle(seed, math):
    c = _case(seed)
    want, x_want, n_edges = _oracle(seed)
    model = _model(c).set_math(math)
    graphs = [_graph(c)]
    if c.capacity is not None:
        graphs.append(_graph(c, c.capacity))
    pos0 = graphs[0].pos.clone()
    runs = [(g_i, one_call, _score(model, g, pos0, one_call))
            for g_i, g in enumerate(graphs) for one_call in (False, True)]
    what = f'seed {seed} {math} {c.kind} sizes={c.sizes} E={n_edges} {c.head} {c.kw}'
    base_s, base_x = runs[0][2]
    for g_i, one_call, (s, x) in runs[1:]:
        tag = (f"{'capacity-bounded' if g_i else 'exact'} graph, "
               f"{'one-call' if one_call else 'per-layer'}")
        assert np.array_equal(_bits(s), _bits(base_s)), (tag, what)
        assert np.array_equal(_bits(x), _bits(base_x)), (tag, what)
    got, x_got = runs[1][2]
    tol, x_tol = _tolerances(seed, math, want, x_want)
    scale = max(1e-3, float(np.abs(want).max()))
    err = float(np.abs(got.astype(np.float64) - want).max()) / scale
    x_err = helpers.scaled_err(x_got, x_want)
    print(f"SWEEP seed={seed} math={math} k={c.kw['k']} score_err={err:.3e} "
          f"coord_err={x_err:.3e} bound={tol:.1e}/{x_tol:.1e}")
    assert err <= tol, (err, tol, what)
    assert x_err < x_tol, (x_err, x_tol, what)


@pytest.mark.gpu
def test_sweep_wide_fp32_raises():
    """65..128 has no FFMA forward: both paths refuse fp32."""
    from pointvs_b200._cabi import PvsError
    c = next(_case(s) for s in range(N_CASES) if _case(s).kw['k'] > 64)
    model = _model(c).set_math('fp32')
    graph = _graph(c)
    pos0 = graph.pos.clone()
    for one_call in (False, True):
        with pytest.raises(PvsError, match='tensor-core math mode'):
            _score(model, graph, pos0, one_call)


def test_sweep_reaches_every_switch():
    """The generator reaches every shape that selects a different code path.
    Runs without a GPU, so narrowing the generator fails here."""
    from oracle import radius_graph as rg
    cases = [_case(s) for s in range(N_CASES)]
    pairs = {(c.kw['k'], m) for c in cases for m in _modes(c.kw['k'])}
    # hidden width on both sides of 32 (FFMA KP = 32 / 64), 64 (64- / 128-wide
    # tiles) and 65, in every mode that runs it
    for k in NARROW:
        for m in MATHS:
            assert (k, m) in pairs, (k, m)
    for k in WIDE:
        for m in MATHS[1:]:
            assert (k, m) in pairs, (k, m)
        assert any(c.kw['k'] == k and c.kind != 'no_edges' for c in cases), k
    # GraphNorm where the upper 64-channel half is one channel short of full
    # (kc = 63), feeding further layers, on a batch with edges
    assert any(c.kw['k'] == 127 and c.kw['graphnorm'] and
               c.kw['num_layers'] >= 2 and c.kind != 'no_edges'
               for c in cases)
    # embedding on both sides of the streaming-kernel switch
    for n in (SMALLK_ROWS - 1, SMALLK_ROWS, SMALLK_ROWS + 1):
        assert any(sum(c.sizes) == n and c.kw['dim_input'] <= 32 and
                   c.kw['k'] <= 64 for c in cases), n
    assert any(sum(c.sizes) % 64 and sum(c.sizes) % 128 for c in cases)
    for s in (1, 2, 3):
        assert any(s in c.sizes for c in cases), s
    assert {c.kw['dim_input'] for c in cases} == set(DIM_INPUTS)
    assert {c.kw['num_layers'] for c in cases} == {1, 2, 3, 4}
    assert {c.head for c in cases} == set(HEADS)
    assert {c.kw['dim_output'] for c in cases
            if c.head in ('fc', 'multi_fc', 'mt_affinity')} == {1, 3}
    assert any(c.capacity == 'auto' for c in cases)
    assert any(c.capacity is None for c in cases)
    # every layer option on and off, at widths up to 64 and above it
    for opt in ('residual', 'edge_residual', 'edge_attention',
                'softmax_attention', 'node_attention', 'normalize', 'tanh',
                'graphnorm', 'update_coords', 'permutation_invariance',
                'gated_residual', 'rezero'):
        for side in (NARROW, WIDE):
            vals = {bool(c.kw[opt]) for c in cases if c.kw['k'] in side}
            assert vals == {False, True}, (opt, side)
    for opt in ('edge_attention_first_only', 'node_attention_final_only'):
        assert {c.kw[opt] for c in cases if c.multitask} == {False, True}, opt
    assert {c.kw['attention_activation_fn'] for c in cases} == \
        {'sigmoid', 'tanh', 'silu', 'relu'}

    def in_degrees(c):
        deg = np.zeros(len(c.coords), dtype=np.int64)
        for lo, hi in zip(c.cptr[:-1], c.cptr[1:]):
            _, row, _, _ = rg.radius_graph(c.coords[lo:hi], c.bp[lo:hi],
                                           c.inter, c.intra)
            deg[lo:hi] = np.bincount(row, minlength=hi - lo)
        return deg

    # an empty edge list, an edgeless complex beside others, and a
    # destination with more edges than one 128-edge tile (more than 300)
    assert any(in_degrees(c).sum() == 0 for c in cases if c.kind == 'no_edges')
    edgeless = [c for c in cases if c.kind == 'edgeless']
    assert edgeless
    for c in edgeless:
        deg = in_degrees(c)
        per = [deg[lo:hi].sum() for lo, hi in zip(c.cptr[:-1], c.cptr[1:])]
        assert 0 in per and deg.sum() > 0
    dense = [c for c in cases if c.kind == 'dense']
    assert dense and all(in_degrees(c).max() > 300 for c in dense)


# ---------------------------------------------------------------------------
# B. dense helpers through the C ABI, against numpy float64
# ---------------------------------------------------------------------------
ACTS = ('none', 'sigmoid', 'tanh', 'relu', 'silu', 'softplus')


def _lib():
    from pointvs_b200 import _cabi
    return _cabi.lib()


def _call(fn, *args):
    from pointvs_b200._cabi import check, stream
    check(fn(*args, stream()), fn.__name__)
    torch.cuda.synchronize()


def _addr(t, offset_floats=0):
    return C.c_void_p(t.data_ptr() + 4 * offset_floats)


@np.errstate(over='ignore')
def _act64(v, act):
    if act == 'sigmoid':
        return 1.0 / (1.0 + np.exp(-v))
    if act == 'tanh':
        return np.tanh(v)
    if act == 'relu':
        return np.maximum(v, 0.0)
    if act == 'silu':
        return v / (1.0 + np.exp(-v))
    if act == 'softplus':        # torch.nn.Softplus(beta=1, threshold=20)
        return np.where(v > 20.0, v, np.log1p(np.exp(np.minimum(v, 20.0))))
    return v


@np.errstate(over='ignore')
def _act_grad64(v, act):
    s = 1.0 / (1.0 + np.exp(-v))
    return {'none': np.ones_like(v), 'sigmoid': s * (1.0 - s),
            'tanh': 1.0 - np.tanh(v) ** 2, 'relu': (v > 0).astype(np.float64),
            'silu': s * (1.0 + v * (1.0 - s)),
            'softplus': np.where(v > 20.0, 1.0, s)}[act]


def _linear_inputs(rng, rows, ki, ko, ld_in):
    """Inputs whose rows span three scales, so pre-activations reach past the
    softplus threshold (20) and far below zero."""
    x = rng.normal(size=(rows, ld_in)).astype(np.float32)
    x *= rng.choice(np.float32([0.1, 1.0, 40.0]), size=(rows, 1))
    w = rng.uniform(-1, 1, size=(ko, ki)).astype(np.float32)
    b = rng.uniform(-1, 1, size=ko).astype(np.float32)
    return x, w, b


def _linear_ref(x, w, b, ki, act):
    x64 = x[:, :ki].astype(np.float64)
    w64 = w.astype(np.float64)
    v = x64 @ w64.T + (0.0 if b is None else b.astype(np.float64))
    terms = np.abs(x64) @ np.abs(w64).T + (0.0 if b is None else np.abs(b))
    return v, terms


# (layout, ld_in pad, ld_out pad, out offset in floats, bias)
LAYOUTS = (('packed', 0, 0, 0, True), ('strided', 3, 5, 0, True),
           ('unaligned_out', 0, 0, 1, True), ('no_bias', 2, 1, 0, False))


def _run_linear(rng, rows, ki, ko, act, layout):
    _, pad_in, pad_out, off, has_b = layout
    ld_in, ld_out = ki + pad_in, ko + pad_out
    x, w, b = _linear_inputs(rng, rows, ki, ko, ld_in)
    b = b if has_b else None
    dx = torch.from_numpy(x).cuda()
    dw = torch.from_numpy(w).cuda()
    db = None if b is None else torch.from_numpy(b).cuda()
    out = torch.full((rows * ld_out + off + 1,), float('nan'), device='cuda')
    _call(_lib().pvs_linear_fwd, _addr(dx), ld_in, rows, ki, _addr(dw), ki,
          None if db is None else _addr(db), ko, _ACT_ID[act],
          _addr(out, off), ld_out)
    flat = out.cpu().numpy()
    got = flat[off:off + rows * ld_out].reshape(rows, ld_out)
    # nothing outside the [rows][ko] block is written
    assert np.isnan(flat[:off]).all() and np.isnan(flat[off + rows * ld_out:]).all()
    assert np.isnan(got[:, ko:]).all(), 'wrote into the row padding'
    v, terms = _linear_ref(x, w, b, ki, act)
    want = _act64(v, act)
    # fp32 accumulation: 1e-6 of the sum of |terms| (SiLU's slope reaches 1.1);
    # the activation itself: a few ulps of the result
    bound = 1.1e-6 * terms + 2e-6 * np.abs(want) + 1e-30
    err = np.abs(got[:, :ko].astype(np.float64) - want)
    assert (err <= bound).all(), (rows, ki, ko, act, layout[0],
                                  float((err / bound).max()))


_ACT_ID = {a: i for i, a in enumerate(ACTS)}
LIN_ROWS = (0, 1, 63, 64, 65, 4095, 4096, 4097, 70_001)
LIN_KI = (1, 3, 13, 16, 17, 31, 32, 33, 64, 100, 128)
LIN_KO = (1, 3, 4, 63, 64, 65, 128)


@pytest.mark.gpu
@pytest.mark.parametrize('rows', LIN_ROWS)
def test_linear_fwd_vs_float64(rows):
    """Every (ki, ko) pair at this row count; activation and layout rotate
    over the pairs.  From 4096 rows with ki <= 32 and ko <= 64 this is the
    streaming kernel, whose float4 store needs ko % 4 == 0, ld_out % 4 == 0
    and an aligned `out`."""
    rng = np.random.default_rng(rows)
    i = 0
    for ki in LIN_KI:
        for ko in LIN_KO:
            _run_linear(rng, rows, ki, ko, ACTS[i % len(ACTS)],
                        LAYOUTS[(i // len(ACTS) + i) % len(LAYOUTS)])
            i += 1


@pytest.mark.gpu
@pytest.mark.parametrize('ko', (4, 63, 64))
@pytest.mark.parametrize('ki', (1, 13, 32))
def test_linear_smallk_store_paths(ki, ko):
    """Streaming kernel, every layout and activation: float4 stores, scalar
    tail, strided and unaligned outputs, no bias."""
    rng = np.random.default_rng(100 * ki + ko)
    for layout in LAYOUTS:
        for act in ACTS:
            _run_linear(rng, 4097, ki, ko, act, layout)


# max |act''| over the real line: the largest change of act' per unit of
# error in the pre-activation
ACT_CURVATURE = {'sigmoid': 0.0962, 'tanh': 0.7699, 'silu': 0.5,
                 'softplus': 0.25}


def _linear_bwd_case(rows, ki, ko, act, ld_in, ld_dout):
    """Inputs and float64 reference of pvs_linear_bwd: g = d_out * act'(v).

    Rows are drawn at unit scale (|v| of order 1), so that a bound per row
    stays small beside what a row adds to d_w and d_b; eight rows are scaled
    up so that v crosses the softplus threshold (20) and falls far below zero.
    Returns x, w, b, d_out, g and g_err, a bound on |g_kernel - g| per entry:
    none: act' = 1, exact.  relu: act' is exactly 0 or 1 away from the kink
    (d_out is zeroed where v lies within rounding of it).  Smooth activations:
    v carries 1.1e-6 of its |terms| (as in the forward), which moves act' by
    at most max|act''| times that; act' itself is evaluated to 1e-6 (1 + |v|)
    (the fp32 argument of the exponential loses |v| ulps); the product with
    d_out rounds once."""
    rng = np.random.default_rng(rows + ki + ko)
    x = (rng.normal(size=(rows, ld_in)) / np.sqrt(ki)).astype(np.float32)
    big = rng.choice(rows, min(8, rows // 8), replace=False)
    x[big] *= 60.0
    w = rng.uniform(-1, 1, size=(ko, ki)).astype(np.float32)
    b = rng.uniform(-1, 1, size=ko).astype(np.float32)
    v, vterms = _linear_ref(x, w, b, ki, act)
    d_out = rng.normal(size=(rows, ld_dout)).astype(np.float32)
    if act == 'relu':
        d_out[:, :ko][np.abs(v) < 1e-4 * vterms] = 0.0
    dout64 = np.abs(d_out[:, :ko].astype(np.float64))
    g = d_out[:, :ko].astype(np.float64) * _act_grad64(v, act)
    if act in ('none', 'relu'):
        g_err = np.zeros_like(g)
    else:
        g_err = dout64 * (ACT_CURVATURE[act] * 1.1e-6 * vterms +
                          1e-6 * (1.0 + np.abs(v))) + 1e-7 * np.abs(g)
    return x, w, b, d_out, g, g_err, rng


@pytest.mark.gpu
@pytest.mark.parametrize('act', ACTS)
@pytest.mark.parametrize('rows,ki,ko', [(1, 1, 1), (65, 13, 64),
                                         (4097, 33, 63), (5000, 128, 17)])
def test_linear_bwd_vs_float64(rows, ki, ko, act):
    """d_in = g . W, d_w += g^T . in, d_b += colsum(g), g = d_out * act'(v);
    each output present or NULL, accumulating into non-zero values.  The
    accumulation itself is held to 1e-6 of the sum of |terms|."""
    lib = _lib()
    ld_in, ld_dout, ld_din, ld_dw = ki + 1, ko + 2, ki + 3, ki + 1
    x, w, b, d_out, g, g_err, rng = _linear_bwd_case(rows, ki, ko, act, ld_in,
                                                      ld_dout)
    g_abs = np.abs(g)
    x64 = x[:, :ki].astype(np.float64)
    w64 = w.astype(np.float64)
    want_din = g @ w64
    bound_din = g_err @ np.abs(w64) + 1e-6 * (g_abs @ np.abs(w64)) + 1e-30
    dw0 = rng.normal(size=(ko, ld_dw)).astype(np.float32)
    db0 = rng.normal(size=ko).astype(np.float32)
    want_dw = dw0[:, :ki] + g.T @ x64
    bound_dw = g_err.T @ np.abs(x64) + \
        1e-6 * (np.abs(dw0[:, :ki]) + g_abs.T @ np.abs(x64))
    want_db = db0 + g.sum(0)
    bound_db = g_err.sum(0) + 1e-6 * (np.abs(db0) + g_abs.sum(0))
    dev = {n: torch.from_numpy(a).cuda() for n, a in
           (('x', x), ('w', w), ('b', b), ('d_out', d_out))}
    ws = torch.empty(int(lib.pvs_linear_bwd_workspace_bytes(rows, ki, ko)),
                     dtype=torch.uint8, device='cuda')
    for mask in range(8):
        d_in = torch.full((rows, ld_din), float('nan'), device='cuda') \
            if mask & 1 else None
        d_w = torch.from_numpy(dw0.copy()).cuda() if mask & 2 else None
        d_b = torch.from_numpy(db0.copy()).cuda() if mask & 4 else None
        _call(lib.pvs_linear_bwd, _addr(dev['x']), ld_in, rows, ki,
              _addr(dev['w']), ki, _addr(dev['b']), ko, _ACT_ID[act],
              _addr(dev['d_out']), ld_dout,
              None if d_in is None else _addr(d_in), ld_din,
              None if d_w is None else _addr(d_w), ld_dw,
              None if d_b is None else _addr(d_b), _addr(ws),
              C.c_int64(ws.numel()))
        if d_in is not None:
            got = d_in.cpu().numpy()
            assert np.isnan(got[:, ki:]).all()
            err = np.abs(got[:, :ki] - want_din)
            assert (err <= bound_din).all(), ('d_in', mask, float((err / bound_din).max()))
        if d_w is not None:
            got = d_w.cpu().numpy()
            assert np.array_equal(got[:, ki:], dw0[:, ki:])
            err = np.abs(got[:, :ki] - want_dw)
            assert (err <= bound_dw).all(), ('d_w', mask, float((err / bound_dw).max()))
        if d_b is not None:
            err = np.abs(d_b.cpu().numpy() - want_db)
            assert (err <= bound_db).all(), ('d_b', mask, float((err / bound_db).max()))


def _pool_ptr(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)


# graph sizes: empty graphs first, in the middle and last, a one-node graph
# and one of 100 000 rows
POOL_SIZES = (0, 0, 5, 1, 0, 64, 129, 100_000, 3, 0, 0)


@pytest.mark.gpu
@pytest.mark.parametrize('offset', (0, 1))
@pytest.mark.parametrize('k', (1, 63, 64, 65, 127, 128))
def test_mean_pool_fwd_bwd_vs_float64(k, offset):
    """offset = 1 shifts h by one float, so k = 64 leaves the float4 path."""
    rng = np.random.default_rng(k + 1000 * offset)
    ptr = _pool_ptr(POOL_SIZES)
    n, b = int(ptr[-1]), len(POOL_SIZES)
    h = rng.normal(size=(n, k)).astype(np.float32)
    buf = torch.full((n * k + offset,), float('nan'), device='cuda')
    buf[offset:] = torch.from_numpy(h.reshape(-1)).cuda()
    dptr = torch.from_numpy(ptr).cuda()
    pooled = torch.full((b, k), float('nan'), device='cuda')
    lib = _lib()
    _call(lib.pvs_mean_pool_fwd, _addr(buf, offset), _addr(dptr), b, k,
          _addr(pooled))
    got = pooled.cpu().numpy()
    h64 = h.astype(np.float64)
    for g in range(b):
        lo, hi = ptr[g], ptr[g + 1]
        if hi == lo:
            assert (got[g] == 0).all(), g      # the header promises 0
            continue
        want = h64[lo:hi].mean(0)
        bound = 1e-6 * np.abs(h64[lo:hi]).sum(0) / (hi - lo) + 1e-30
        assert (np.abs(got[g] - want) <= bound).all(), (g, hi - lo)
    d_pooled = rng.normal(size=(b, k)).astype(np.float32)
    d_h = torch.full((n * k + offset,), float('nan'), device='cuda')
    _call(lib.pvs_mean_pool_bwd, _addr(torch.from_numpy(d_pooled).cuda()),
          _addr(dptr), b, k, _addr(d_h, offset))
    got = d_h.cpu().numpy()
    assert np.isnan(got[:offset]).all()
    got = got[offset:].reshape(n, k)
    cnt = np.diff(ptr)
    want = np.repeat(d_pooled.astype(np.float64) / np.maximum(cnt, 1)[:, None],
                     cnt, axis=0)
    assert (np.abs(got - want) <= 2e-7 * np.abs(want)).all()


@pytest.mark.gpu
def test_batch_to_ptr_gaps_and_empty_ends():
    lib = _lib()
    cases = [
        (np.array([2, 2, 2, 4, 4, 7, 7, 7, 7]), 10),    # empty 0, 1, 3, 5, 6, 8, 9
        (np.repeat(np.arange(300), 7)[3:-2], 300),       # contiguous
        (np.zeros(5), 1), (np.full(4, 3), 4),
        (np.zeros(0), 3),                                 # n_nodes = 0
        (np.sort(np.random.default_rng(0).integers(0, 5000, 70_001)), 5003),
    ]
    for batch, n_graphs in cases:
        batch = batch.astype(np.int64)
        want = np.searchsorted(batch, np.arange(n_graphs + 1), 'left')
        db = torch.from_numpy(batch).cuda() if len(batch) else None
        out = torch.full((n_graphs + 1,), -7, dtype=torch.int32, device='cuda')
        _call(lib.pvs_batch_to_ptr, None if db is None else _addr(db),
              len(batch), n_graphs, _addr(out))
        np.testing.assert_array_equal(out.cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize('n', (0, 1, 4095, 4096, 4097, 4_194_305, 8_392_705))
def test_exclusive_scan(n):
    """Above 4 194 304 entries there are more than 1 024 block sums, which the
    block-sum scan walks in a loop (twice, three times)."""
    lib = _lib()
    deg = np.random.default_rng(n).integers(0, 8, n).astype(np.int32)
    want = np.concatenate([[0], np.cumsum(deg, dtype=np.int64)])
    d = torch.from_numpy(deg).cuda() if n else None
    out = torch.full((n + 1,), -7, dtype=torch.int32, device='cuda')
    scratch = torch.empty(int(lib.pvs_scan_scratch_bytes(n)), dtype=torch.uint8,
                          device='cuda')
    _call(lib.pvs_exclusive_scan, None if d is None else _addr(d), n,
          _addr(out), _addr(scratch))
    np.testing.assert_array_equal(out.cpu().numpy(), want)


def _degree_patterns():
    rng = np.random.default_rng(5)
    runs = np.zeros(40, dtype=np.int32)
    runs[[0, 5, 6, 12]] = [128, 100, 28, 256]   # empty nodes on both sides of
    return {                                    # every 128-edge boundary
        'no_edges': np.zeros(17, dtype=np.int32),
        'one_node_no_edges': np.zeros(1, dtype=np.int32),
        'exact_multiple': np.full(24, 16, dtype=np.int32),      # E = 384
        'empty_runs': runs,
        'hub': np.array([0, 0, 700, 0, 1, 0, 0, 127], dtype=np.int32),
        'random_sparse': (rng.integers(0, 40, 3000) *
                          (rng.random(3000) < 0.3)).astype(np.int32),
    }


@pytest.mark.gpu
@pytest.mark.parametrize('slack', (0, 1000))
@pytest.mark.parametrize('pattern', sorted(_degree_patterns()))
def test_build_packed_tiles(pattern, slack):
    """Tile t owns edges [128 t, 128 t + 128); ptile_last[t] is the node of
    its last edge.  slack > 0 passes an edge capacity above the true count
    (the count is read from row_ptr[n])."""
    lib = _lib()
    deg = _degree_patterns()[pattern]
    row_ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    n, e = len(deg), int(row_ptr[-1])
    cap = int(lib.pvs_packed_tiles_capacity(e + slack))
    last = torch.full((cap,), -7, dtype=torch.int32, device='cuda')
    n_tiles = torch.full((1,), -7, dtype=torch.int32, device='cuda')
    _call(lib.pvs_build_packed_tiles, _addr(torch.from_numpy(row_ptr).cuda()),
          n, e + slack, _addr(last), _addr(n_tiles))
    t = max(1, -(-e // 128))
    assert int(n_tiles.item()) == t
    got = last.cpu().numpy()[:t]
    if e == 0:
        assert (got == n - 1).all()
        return
    ends = np.minimum(128 * (np.arange(t) + 1), e) - 1
    np.testing.assert_array_equal(got, np.searchsorted(row_ptr, ends, 'right') - 1)
