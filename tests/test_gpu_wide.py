"""Hidden widths 65..128 on the GPU: the 128-wide tensor-core forward against
the CPU oracle in float64, per layer, per option and end to end.

Tolerances are DESIGN §2's per mode: bf16x3 1e-4 relative on scores, fp16x2
5e-4, bf16 3e-2; per-node tensors by scaled_err with the same bounds."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from tests import helpers
from tests import gpu_helpers as gh

pytestmark = pytest.mark.gpu

TOL = {'bf16x3': 1e-4, 'fp16x2': 5e-4, 'bf16': 3e-2}
BASE = dict(dim_input=13, dim_output=1, k=128, num_layers=3, residual=True,
            normalize=True, tanh=True, graphnorm=False)
CFG3 = dict(dim_input=13, dim_output=1, k=128, num_layers=8,
            edge_attention=True, node_attention=True, residual=True,
            normalize=True, tanh=True, graphnorm=False)


def _cpu(graph, pos=None):
    return SimpleNamespace(x=graph.x, pos=graph.pos if pos is None else pos,
                           edge_index=graph.edge_index,
                           edge_attr=graph.edge_attr, batch=graph.batch)


def _layer_vs_oracle(k, math, edge_index, edge_attr, pos, seed=0, **flags):
    """One EGNNLayer on the GPU and in the oracle (float64): h, x, attention
    values and messages."""
    from oracle import egnn_oracle
    from pointvs_b200 import EGNNLayer
    torch.manual_seed(seed)
    layer = EGNNLayer(k, k, k, edges_in_d=3, math=math, **flags).cuda()
    with torch.no_grad():
        layer.coord_mlp[2].weight.mul_(1000.0)
    n = pos.shape[0]
    h = torch.randn(n, k, generator=torch.Generator().manual_seed(1)).cuda()
    coord = pos.clone()
    with torch.no_grad():
        h2, x2, _, m2 = layer(h, edge_index, coord, edge_attr, None)
    sd = {key: v.detach().cpu().double() for key, v in layer.state_dict().items()}
    cfg = egnn_oracle.LayerConfig(
        residual=flags.get('residual', True),
        edge_attention=flags.get('edge_attention', False),
        normalize=flags.get('normalize', False), tanh=flags.get('tanh', False),
        node_attention=flags.get('node_attention', False))
    ei = edge_index.cpu()
    want = egnn_oracle.layer_forward(
        sd, '', cfg, h.cpu().double(), ei[0], ei[1], pos.cpu().double(),
        edge_attr.cpu())
    got = (h2, x2, m2)
    for name, a, b in zip('hxm', got, want[:3]):
        err = helpers.scaled_err(a.cpu().numpy(), b.numpy())
        assert err < TOL[math], (name, err)
    if flags.get('edge_attention'):
        att = layer.att_val
        att = att.cpu().numpy() if torch.is_tensor(att) else np.asarray(att)
        err = helpers.scaled_err(att.reshape(-1),
                                 want[3]['att_val'].numpy().reshape(-1))
        assert err < TOL[math], ('att', err)
    return h2, x2, m2


@pytest.mark.parametrize('math', ['bf16x3', 'fp16x2', 'bf16'])
@pytest.mark.parametrize('k', [65, 96, 128])
def test_wide_layer_matches_oracle(k, math):
    graph = gh.synthetic_graph(500, 3, 700, 25, ragged=True)
    _layer_vs_oracle(k, math, graph.edge_index, graph.edge_attr, graph.pos,
                     edge_attention=True, node_attention=True, normalize=True,
                     tanh=True)


OPTIONS = {
    'attention': dict(edge_attention=True, node_attention=True),
    'softmax': dict(edge_attention=True, node_attention=True,
                    softmax_attention=True),
    'graphnorm': dict(graphnorm=True, edge_attention=True),
    'gated': dict(gated_residual=True, node_attention=True),
    'rezero': dict(rezero=True, edge_attention=True),
    'edge_residual': dict(edge_residual=True, edge_attention=True),
    'perm_invariant': dict(permutation_invariance=True),
    'static_coords': dict(update_coords=False, edge_attention=True),
}


def _model_vs_oracle(kw, math, graph, multitask=False, seed=3):
    model = gh.build_model(kw, multitask=multitask, seed=seed, coord_gain=1.0)
    model.set_math(math)
    pos0 = graph.pos.clone()
    with torch.no_grad():
        out = model(graph)
    want, _ = gh.oracle_forward(model, kw, _cpu(graph, pos0),
                                multitask=multitask, dtype=torch.float64)
    err = helpers.rel_err(out.cpu().numpy().reshape(-1),
                          want.numpy().reshape(-1))
    assert err < TOL[math], err
    return model, out


@pytest.mark.parametrize('option', sorted(OPTIONS))
def test_wide_model_options_match_oracle(option):
    kw = dict(BASE, **OPTIONS[option])
    ragged = option == 'graphnorm'
    graph = gh.synthetic_graph(40, 4, 600, 25, ragged=ragged)
    _model_vs_oracle(kw, 'bf16x3', graph)


def test_wide_permutation_invariance():
    kw = dict(BASE, permutation_invariance=True, edge_attention=True)
    model = gh.build_model(kw, seed=5, coord_gain=1.0)
    model.set_math('bf16x3')
    g1 = gh.synthetic_graph(41, 2, 400, 20)
    with torch.no_grad():
        a = model(_cpu(g1, g1.pos.clone()))
        perm = torch.randperm(g1.x.shape[0], generator=torch.Generator().manual_seed(0)).cuda()
        # nodes relabelled (within each complex the batch ids stay sorted)
        order = torch.argsort(g1.batch[perm] * perm.numel() + torch.arange(perm.numel(), device=perm.device))
        p = perm[order]
        newid = torch.empty_like(p)
        newid[p] = torch.arange(p.numel(), device=p.device)
        g2 = SimpleNamespace(x=g1.x[p], pos=g1.pos[p].clone(),
                             edge_index=newid[g1.edge_index],
                             edge_attr=g1.edge_attr, batch=g1.batch[p])
        b = model(g2)
    assert helpers.rel_err(b.cpu().numpy(), a.cpu().numpy()) < 1e-4


@pytest.mark.parametrize('math', ['bf16x3', 'fp16x2', 'bf16'])
def test_wide_multitask_first_final_attention_multi_fc(math):
    kw = dict(BASE, edge_attention=True, node_attention=True,
              edge_attention_first_only=True, node_attention_final_only=True,
              multi_fc=True)
    graph = gh.synthetic_graph(42, 4, 600, 25)
    _model_vs_oracle(kw, math, graph, multitask=True)


@pytest.mark.parametrize('math', ['bf16x3', 'fp16x2', 'bf16'])
def test_wide_fused_scoring_pass_equals_per_layer_path(math):
    kw = dict(BASE, edge_attention=True, node_attention=True)
    model = gh.build_model(kw, seed=4, coord_gain=1.0)
    model.set_math(math)
    model.set_record_side_channels(False)
    model.record_embed_coords = False
    with torch.no_grad():
        assert model._fast_path_ok()
        a = model(gh.synthetic_graph(43, 3, 500, 20))
        model.set_record_side_channels(True)
        assert not model._fast_path_ok()
        b = model(gh.synthetic_graph(43, 3, 500, 20))
    assert torch.equal(a, b)


def _hub_graph():
    """Node 0 is a hub with 300 neighbours in both directions; nodes 400..599
    have no edges at all; the rest have random neighbourhoods of 0..40, so
    node boundaries fall anywhere inside the 128-edge tiles."""
    rng = np.random.default_rng(7)
    n = 800
    rows, cols = [], []
    for j in range(1, 301):
        rows += [0, j]
        cols += [j, 0]
    for i in list(range(1, 400)) + list(range(600, n)):
        nb = rng.choice([v for v in range(1, n) if not 400 <= v < 600 and v != i],
                        size=int(rng.integers(0, 40)), replace=False)
        rows += [i] * len(nb)
        cols += list(nb)
    ei = torch.tensor([rows, cols], dtype=torch.long).cuda()
    attr = torch.nn.functional.one_hot(
        torch.from_numpy(rng.integers(0, 3, ei.shape[1])), 3).cuda()
    pos = torch.from_numpy(rng.normal(size=(n, 3)).astype(np.float32) * 3).cuda()
    return ei, attr, pos


@pytest.mark.parametrize('math', ['bf16x3', 'bf16'])
def test_wide_packed_tile_edge_cases(math):
    ei, attr, pos = _hub_graph()
    assert int((ei[0] == 0).sum()) > 128
    _layer_vs_oracle(128, math, ei, attr, pos, edge_attention=True,
                     node_attention=True, normalize=True, tanh=True)


def test_wide_runs_are_bitwise_reproducible():
    kw = dict(BASE, edge_attention=True, node_attention=True)
    model = gh.build_model(kw, seed=6, coord_gain=1.0)
    model.set_math('bf16x3')
    with torch.no_grad():
        a = model(gh.synthetic_graph(44, 8, 800, 25))
        b = model(gh.synthetic_graph(44, 8, 800, 25))
    assert torch.equal(a, b)
    ei, attr, pos = _hub_graph()
    h1 = _layer_vs_oracle(128, 'bf16x3', ei, attr, pos, edge_attention=True)
    h2 = _layer_vs_oracle(128, 'bf16x3', ei, attr, pos, edge_attention=True)
    for a, b in zip(h1, h2):
        assert torch.equal(a, b)


def test_wide_fullsize_invariance_batch_independence_and_oracle_sample():
    """BASELINE-sized batch (128 x 1000 atoms) through 8 layers at k = 128."""
    model = gh.build_model(CFG3, seed=0, coord_gain=1.0)
    model.set_math('bf16x3')
    graph = gh.synthetic_graph(1000, 128, 1000, 30)
    pos0 = graph.pos.clone()
    with torch.no_grad():
        full = model(_cpu(graph, pos0.clone())).reshape(-1)
        # E(3): rotation + reflection + translation of every coordinate
        q, _ = torch.linalg.qr(torch.randn(3, 3, generator=torch.Generator().manual_seed(3)))
        q[:, 0] = -q[:, 0]
        moved = pos0 @ q.cuda().T + torch.tensor([5.0, -3.0, 2.0], device='cuda')
        rot = model(_cpu(graph, moved)).reshape(-1)
        # the first two complexes scored on their own
        n2 = int((graph.batch < 2).sum())
        e_mask = graph.edge_index[0] < n2
        small = SimpleNamespace(x=graph.x[:n2], pos=pos0[:n2].clone(),
                                edge_index=graph.edge_index[:, e_mask],
                                edge_attr=graph.edge_attr[e_mask],
                                batch=graph.batch[:n2])
        alone = model(small).reshape(-1)
    assert full.shape == (128,)
    assert helpers.rel_err(rot.cpu().numpy(), full.cpu().numpy()) < 1e-4
    assert helpers.rel_err(alone.cpu().numpy(), full[:2].cpu().numpy()) < 1e-4
    want, _ = gh.oracle_forward(model, CFG3, _cpu(small, pos0[:n2]),
                                dtype=torch.float64)
    assert helpers.rel_err(alone.cpu().numpy(), want.numpy().reshape(-1)) < 1e-4


def test_wide_checkpoint_inference_attribution_and_stream(tmp_path):
    """A seeded k = 128 multitask model saved in the reference's format is
    loaded and scored by the inference CLI, and serves atom_masking and
    ScoreStream."""
    import yaml
    import pointvs_b200 as pv
    from oracle import egnn_oracle
    from pointvs_b200 import attribution, inference
    from pointvs_b200.pipeline import ScoreStream
    from tests.golden.loader_configs import CONFIGS, ROOT
    from tests.test_gpu_data import _reference_batch
    gold = helpers.load_npz('loader.npz')
    cfg = 'atomic_h_r6_e3'
    c = CONFIGS[cfg]
    dim = int(gold[f'{cfg}/feature_dim'])
    kw = dict(dim_input=dim, dim_output=1, k=128, num_layers=3, graphnorm=True,
              edge_attention=True, node_attention=True, residual=True,
              normalize=True, tanh=True)
    run = tmp_path / 'run'
    run.mkdir()
    torch.manual_seed(11)
    model = pv.MultitaskSatorrasEGNN(run, 1e-3, 1e-4, None, None, silent=True,
                                     **kw)
    model.save()
    with open(run / 'model_kwargs.yaml', 'w') as f:
        yaml.dump(kw, f)
    with open(run / 'cmd_args.yaml', 'w') as f:
        yaml.dump({'model': 'multitask', 'learning_rate': 1e-3,
                   'weight_decay': 1e-4, 'save_path': str(run),
                   'compact': c['compact'], 'radius': c['radius'],
                   'use_atomic_numbers': c['use_atomic_numbers'],
                   'hydrogens': c['polar_hydrogens'], 'batch_size': 3,
                   'edge_radius': c['edge_radius'],
                   'estimate_bonds': c.get('estimate_bonds', False),
                   'input_suffix': 'parquet', 'egnn_attention': True,
                   'model_task': 'classification', 'channels': 128}, f)
    assert list((run / 'checkpoints').glob('*.pt'))
    out = inference.main([str(run), str(ROOT / 'pose.types'), str(ROOT),
                          '--math', 'bf16x3'])
    pose = out.parent / ('pose_' + out.name)
    lines = pose.read_text().splitlines()
    n = int(gold[f'{cfg}/n'])
    assert len(lines) == n
    sd = {key: v.detach().cpu().double() for key, v in model.state_dict().items()}
    for start in range(0, n, 3):      # GraphNorm statistics are per batch
        items = list(range(start, min(n, start + 3)))
        x, pos, row, col, attr, batch = _reference_batch(gold, cfg, items)
        want, _ = egnn_oracle.model_forward(
            sd, torch.from_numpy(x).double(),
            torch.from_numpy(np.stack([row, col])),
            torch.from_numpy(pos).double(),
            torch.nn.functional.one_hot(
                torch.from_numpy(attr.astype(np.int64)), 3),
            torch.from_numpy(batch), num_layers=3, multitask=True,
            model_task='classification', **helpers.oracle_kwargs(kw))
        want = torch.sigmoid(want).reshape(-1).numpy()
        for j, i in enumerate(items):
            y_pred = float(lines[i].split(' | ')[1].split(' ')[0])
            assert abs(y_pred - want[j]) <= 6e-4 + 1e-4 * abs(want[j])
    # attribution and streaming on the same wide model
    model = model.cuda().eval().set_math('bf16x3')
    x, pos, row, col, attr, batch = _reference_batch(gold, cfg, [0])
    scores = attribution.atom_masking(
        model, p=torch.from_numpy(pos).unsqueeze(0).cuda(),
        v=torch.from_numpy(x).unsqueeze(0).cuda(),
        edge_indices=torch.from_numpy(np.stack([row, col])).cuda(),
        edge_attrs=torch.nn.functional.one_hot(
            torch.from_numpy(attr.astype(np.int64)), 3).cuda(), bs=16)
    assert scores.shape[0] == x.shape[0] and np.all(np.isfinite(scores))
    model.set_record_side_channels(False)
    model.record_embed_coords = False
    g = gh.synthetic_graph(45, 3, 300, 15)
    from pointvs_b200.synthetic import synthetic_batch
    coords, bp, feats, cptr = synthetic_batch(45, 3, n_atoms=300, n_lig=15)
    kw13 = dict(kw, dim_input=13)
    m13 = gh.build_model(kw13, seed=2, coord_gain=1.0)
    m13.set_math('bf16x3')
    m13.set_record_side_channels(False)
    m13.record_embed_coords = False
    with torch.no_grad():
        want = m13(g).reshape(len(cptr) - 1, -1).cpu().numpy()
    stream = ScoreStream(m13, 4.0, 4.0, depth=2)
    stream.submit(coords, bp, feats, cptr, tag=0)
    got = stream.results() + stream.drain()
    assert [t for t, _ in got] == [0]
    np.testing.assert_array_equal(got[0][1], want)


def test_wide_backward_raises():
    from pointvs_b200 import EGNNLayer
    from pointvs_b200._cabi import PvsError
    graph = gh.synthetic_graph(46, 2, 300, 15)
    layer = EGNNLayer(96, 96, 96, edges_in_d=3, math='bf16x3').cuda()
    h = torch.randn(graph.x.shape[0], 96, device='cuda', requires_grad=True)
    h2, x2, _, _ = layer(h, graph.edge_index, graph.pos.clone(),
                         graph.edge_attr, None)
    with pytest.raises(PvsError):
        h2.sum().backward()
