"""K1p on the GPU: the pocket graph of K0-assembled complexes is K1's, byte for
byte, and `score_poses` scores what the crop_batch -> radius_graph_batch ->
model chain scores, bit for bit."""
import numpy as np
import pytest
import torch

from tests import gpu_helpers as gh
from tests.golden.loader_configs import CONFIGS, ROOT
from oracle import radius_graph as rg

pytestmark = pytest.mark.gpu

N_LIG, N_POCKET, N_TYPES = 30, 800, 12


def _synthetic(n_poses, n_pocket=N_POCKET, first=0):
    """The configs[4] pocket (resident triple) and `n_poses` ligand poses."""
    from pointvs_b200 import data
    from pointvs_b200.synthetic import synthetic_pocket_poses
    coords, _, feats, _ = synthetic_pocket_poses(first, n_poses, n_pocket,
                                                 N_LIG)
    types = feats[:, :N_TYPES].argmax(1)
    per = N_LIG + n_pocket
    rec = (torch.from_numpy(coords[N_LIG:per].copy()).cuda(),
           torch.ones(n_pocket, dtype=torch.uint8, device='cuda'),
           torch.from_numpy((types[N_LIG:per] + N_TYPES).astype(np.int16)
                            ).cuda())
    ligs = [data.Ligand(coords[p * per:p * per + N_LIG].copy(),
                        np.ones(N_LIG, dtype=np.uint8),
                        types[p * per:p * per + N_LIG].astype(np.int16))
            for p in range(n_poses)]
    torch.cuda.synchronize()
    return rec, ligs


def _graphs(pocket, ligs, rec_of_pose, radius, n_features=N_TYPES,
            compact=True, capacity=None):
    """K0 once, then K1 and K1p on its output."""
    from pointvs_b200.graph import radius_graph_batch
    crop = pocket.crop(ligs, rec_of_pose, radius, n_features, compact)
    want = radius_graph_batch(crop.coords, crop.bp, crop.complex_ptr_host,
                              pocket.inter_radius, pocket.intra_radius,
                              device='cuda', edge_capacity=capacity)
    lig_count = [int(np.count_nonzero(l.emit)) for l in ligs]
    got = pocket.radius_graph(crop, lig_count, edge_capacity=capacity)
    return crop, want, got


def _assert_same_graph(want, got):
    n = want.n_nodes
    assert got.n_nodes == n
    np.testing.assert_array_equal(got.row_ptr.cpu().numpy(),
                                  want.row_ptr.cpu().numpy())
    e = int(want.row_ptr[-1].item())
    assert e == int(got.row_ptr[-1].item())
    np.testing.assert_array_equal(got.col[:e].cpu().numpy(),
                                  want.col[:e].cpu().numpy())
    np.testing.assert_array_equal(got.attr[:e].cpu().numpy(),
                                  want.attr[:e].cpu().numpy())
    np.testing.assert_array_equal(got.n_inter[:n].cpu().numpy(),
                                  want.n_inter[:n].cpu().numpy())
    return e


def _oracle_check(crop, graph, inter, intra, poses):
    """A few complexes against the C restatement of generate_edges."""
    cptr = crop.complex_ptr_host
    coords = crop.coords.cpu().numpy()
    bp = crop.bp.cpu().numpy()
    row_ptr = graph.row_ptr.cpu().numpy()
    col = graph.col.cpu().numpy()
    attr = graph.attr.cpu().numpy()
    for b in poses:
        lo, hi = int(cptr[b]), int(cptr[b + 1])
        r, c, a = rg.radius_graph_c(coords[lo:hi], bp[lo:hi], inter, intra)
        e0, e1 = row_ptr[lo], row_ptr[hi]
        rows = np.repeat(np.arange(hi - lo), np.diff(row_ptr[lo:hi + 1]))
        want = rg.canonical(r, c, a)
        got = rg.canonical(rows, col[e0:e1] - lo, attr[e0:e1])
        for w, g in zip(want, got):
            np.testing.assert_array_equal(w, g)


@pytest.mark.parametrize('radii', [(4.0, 4.0), (4.0, 2.0)])
@pytest.mark.parametrize('crop_radius', [None, 10.0, 6.0])
def test_synthetic_pocket_graph_is_k1s(radii, crop_radius):
    from pointvs_b200.screening import Pocket
    rec, ligs = _synthetic(48)
    pocket = Pocket(rec, *radii)
    radius = np.inf if crop_radius is None else crop_radius
    crop, want, got = _graphs(pocket, ligs, np.zeros(48, np.int32), radius)
    assert _assert_same_graph(want, got) > 0
    _oracle_check(crop, got, *radii, poses=(0, 17, 47))


@pytest.mark.parametrize('cfg', ['smina_r10_e4', 'atomic_h_r6_e3',
                                 'smina_wide_r7_bonds'])
def test_real_receptors_mixed_in_one_batch(cfg):
    """Receptors 10378 and 18061 with their actives and decoys, interleaved
    through rec_of_pose; the smina configs drop the hydrogens (non-emitted
    ligand and receptor atoms), estimate_bonds gives radii (5, 2)."""
    from pointvs_b200 import data
    from pointvs_b200.screening import Pocket
    ds = data.ComplexDataset(ROOT, types_fname=ROOT / 'pose.types', rot=False,
                             device='cuda', device_crop=True, **CONFIGS[cfg])
    names = ['receptors/10378.parquet', 'receptors/18061.parquet']
    pocket = Pocket.from_dataset(ds, names)
    items = [i for i in range(len(ds)) if ds.receptor_fnames[i] in names]
    assert len(items) == 6
    items = items + items[::-1]
    ligs = [ds.load_ligand(i) for i in items]
    rop = np.array([names.index(ds.receptor_fnames[i]) for i in items],
                   np.int32)
    assert len(set(rop)) == 2
    crop, want, got = _graphs(pocket, ligs, rop, ds.radius, ds.n_features,
                              ds.compact)
    _assert_same_graph(want, got)
    _oracle_check(crop, got, ds.inter_radius, ds.intra_radius,
                  poses=range(len(items)))
    # and the complexes are the host loader's
    host = [ds.load(i) for i in items]
    np.testing.assert_array_equal(crop.coords.cpu().numpy(),
                                  np.concatenate([c.coords for c in host]))


def _special_ligands(pocket_xyz):
    """Ligands that sit on the edge cases of the pair test."""
    from pointvs_b200 import data
    rng = np.random.default_rng(7)
    p = pocket_xyz

    def lig(xyz, emit=None):
        xyz = np.ascontiguousarray(xyz, dtype=np.float64)
        emit = np.ones(len(xyz), np.uint8) if emit is None else emit
        return data.Ligand(xyz, emit, rng.integers(0, N_TYPES, len(xyz)
                                                   ).astype(np.int16))
    ligs = []
    # an atom coincident with a receptor atom, and a ligand atom duplicated
    ligs.append(lig(np.stack([p[5], p[5] + [0.5, 0, 0], p[5] + [0.5, 0, 0],
                              p[9] + [1.0, 1.0, 0.0]])))
    # pairs at the cut-offs 4 and 2, exactly and one ulp either side, also on
    # a diagonal (sqrt evaluated in the +-1e-15 band)
    at = []
    for r in (4.0, 2.0):
        for d in (r, np.nextafter(r, 0.0), np.nextafter(r, 10.0)):
            at.append(p[11] + [d, 0.0, 0.0])
        q = r / np.sqrt(3.0)
        for d in (q, np.nextafter(q, 0.0), np.nextafter(q, 10.0)):
            at.append(p[13] + [d, d, d])
    ligs.append(lig(np.stack(at)))
    # ligand-ligand pairs at the cut-off
    base = p[20] + [0.3, 0.2, 0.1]
    ligs.append(lig(np.stack([base, base + [4.0, 0, 0], base + [2.0, 0, 0],
                              base + [0, np.nextafter(2.0, 0.0), 0]])))
    # no receptor atom in reach; a one-atom ligand; hydrogens not emitted
    ligs.append(lig(np.full((5, 3), 1000.0) + rng.random((5, 3))))
    ligs.append(lig(p[30:31] + 0.7))
    xyz = p[40:52] + rng.normal(scale=0.8, size=(12, 3))
    emit = np.ones(12, np.uint8)
    emit[::3] = 0
    ligs.append(lig(xyz, emit))
    # the ligand-size bound itself: 256 emitted atoms (and 20 hydrogens)
    xyz = p[rng.integers(0, len(p), 276)] + rng.normal(scale=1.5,
                                                       size=(276, 3))
    emit = np.ones(276, np.uint8)
    emit[:20] = 0
    ligs.append(lig(xyz, emit))
    return ligs


@pytest.mark.parametrize('radii', [(4.0, 4.0), (4.0, 2.0)])
def test_edge_cases_and_ligand_bound(radii):
    from pointvs_b200 import _cabi
    from pointvs_b200.screening import Pocket
    rec, ligs = _synthetic(4)
    pocket = Pocket(rec, *radii)
    special = _special_ligands(rec[0].cpu().numpy())
    assert int(np.count_nonzero(special[-1].emit)) == \
        _cabi.POCKET_MAX_LIG_ATOMS
    for radius in (np.inf, 6.0):
        batch = special + ligs
        crop, want, got = _graphs(pocket, batch, np.zeros(len(batch), np.int32),
                                  radius)
        _assert_same_graph(want, got)
        _oracle_check(crop, got, *radii, poses=range(len(special)))
        # a batch of one pose
        for one in (special[1], special[4]):
            crop, want, got = _graphs(pocket, [one], np.zeros(1, np.int32),
                                      radius)
            _assert_same_graph(want, got)
    # one emitted atom above the bound
    over = special[-1]
    emit = over.emit.copy()
    emit[0] = 1
    from pointvs_b200 import data
    too_big = data.Ligand(over.coords, emit, over.code)
    with pytest.raises(_cabi.PvsError, match='too large'):
        pocket.batch([too_big], radius=None, n_features=N_TYPES)


def test_capacity_auto_and_overflow_as_k1():
    from pointvs_b200.graph import auto_edge_capacity
    from pointvs_b200.screening import Pocket
    rec, ligs = _synthetic(16)
    pocket = Pocket(rec, 4.0, 4.0)
    zeros = np.zeros(16, np.int32)
    crop, want, got = _graphs(pocket, ligs, zeros, np.inf, capacity='auto')
    assert not got.exact_edge_count
    assert got.n_edges == auto_edge_capacity(crop.coords.shape[0], 4.0, 4.0)
    _assert_same_graph(want, got)
    assert int(got._overflow.item()) == 0
    got.check_overflow()
    # a capacity that cuts the graph: overflow set, row_ptr cut exactly as K1
    cap = 5000
    crop, want, got = _graphs(pocket, ligs, zeros, np.inf, capacity=cap)
    assert int(want._overflow.item()) == 1 and int(got._overflow.item()) == 1
    np.testing.assert_array_equal(got.row_ptr.cpu().numpy(),
                                  want.row_ptr.cpu().numpy())
    assert int(got.row_ptr[-1].item()) == cap
    np.testing.assert_array_equal(got.col.cpu().numpy(),
                                  want.col.cpu().numpy())
    np.testing.assert_array_equal(got.attr.cpu().numpy(),
                                  want.attr.cpu().numpy())
    with pytest.raises(Exception, match='edge capacity'):
        got.check_overflow()


def test_receptor_search_is_not_relaunched_per_batch():
    """Per batch: K0 (count, scan, fill) and K1p (2 count kernels, scan, 2
    fill kernels, capacity cut) -- no receptor-receptor search."""
    from pointvs_b200 import _cabi
    from pointvs_b200.screening import Pocket
    rec, ligs = _synthetic(96)
    lib = _cabi.lib()
    n0 = lib.pvs_launch_count()
    pocket = Pocket(rec, 4.0, 4.0)
    build = lib.pvs_launch_count() - n0
    assert build == 5   # cell list, rr count, 2-kernel scan, rr fill
    deltas = []
    for s in range(0, 96, 32):
        crop = pocket.crop(ligs[s:s + 32], np.zeros(32, np.int32), np.inf,
                           N_TYPES)
        n = int(crop.complex_ptr_host[-1])
        before = lib.pvs_launch_count()
        pocket.radius_graph(crop, [N_LIG] * 32, edge_capacity='auto')
        deltas.append(lib.pvs_launch_count() - before)
        scan = 3 if n > 4096 else 2
        assert deltas[-1] == 2 + scan + 2 + 1
    assert len(set(deltas)) == 1


def _long_receptor():
    """A 126 A slab along x: 126 / 4.000004 = 31.5 cell edges at r_max = 4,
    so the receptor grid hits its 32-cell cap on that axis.  Pairs 3.96 A
    apart straddle the boundaries a 126 / 32 A grid would have, each pair's
    atoms two such cells apart."""
    rng = np.random.default_rng(11)
    n = 320
    xyz = np.column_stack([rng.random(n) * 126.0, rng.random(n) * 6.0,
                           rng.random(n) * 6.0])
    xyz[0] = [0.0, 3.0, 3.0]
    xyz[1] = [126.0, 3.0, 3.0]
    edge = 126.0 / 32 * (1 + 1e-6)
    pairs = []
    for k in range(2, 31, 2):
        x1 = k * edge - 0.01
        pairs += [[x1, 1.0, 5.5], [x1 + 3.96, 1.0, 5.5]]
    xyz = np.concatenate([xyz, np.array(pairs)]).astype(np.float32).astype(np.float64)
    types = rng.integers(0, N_TYPES, len(xyz))
    return xyz, types, np.array(pairs[::2])


@pytest.mark.parametrize('radii', [(4.0, 4.0), (4.0, 2.0)])
def test_receptor_at_the_cell_cap_keeps_every_pair(radii):
    from pointvs_b200 import data
    from pointvs_b200.screening import Pocket
    xyz, types, left = _long_receptor()
    rec = (torch.from_numpy(xyz).cuda(),
           torch.ones(len(xyz), dtype=torch.uint8, device='cuda'),
           torch.from_numpy((types + N_TYPES).astype(np.int16)).cuda())
    torch.cuda.synchronize()
    pocket = Pocket(rec, *radii)
    # receptor-receptor rows against the oracle on the whole receptor
    r, c, _ = rg.radius_graph_c(xyz, np.ones(len(xyz), np.int32), *radii)
    rr_ptr = pocket.rr_ptr.cpu().numpy()
    rr_col = pocket.rr_col.cpu().numpy()
    rows = np.repeat(np.arange(len(xyz)), np.diff(rr_ptr))
    want = rg.canonical(r, c, np.zeros_like(r))
    got = rg.canonical(rows, rr_col[:len(rows)], np.zeros_like(rows))
    for w, g in zip(want, got):
        np.testing.assert_array_equal(w, g)
    # ligands next to the straddling pairs: ligand-receptor pairs straddle too
    rng = np.random.default_rng(12)
    ligs = []
    for p in left[::2]:
        lx = np.stack([p + [0.0, 0.3, 0.0], p + [0.0, 0.3, -1.2],
                       p + [2.0, 2.0, -2.0]]).astype(np.float32).astype(np.float64)
        ligs.append(data.Ligand(lx, np.ones(3, np.uint8),
                                rng.integers(0, N_TYPES, 3).astype(np.int16)))
    for radius in (np.inf, 6.0):
        crop, want_g, got_g = _graphs(pocket, ligs, np.zeros(len(ligs), np.int32),
                                      radius)
        _assert_same_graph(want_g, got_g)
        _oracle_check(crop, got_g, *radii, poses=range(len(ligs)))


def test_pose_over_the_ligand_bound_raises_the_overflow_flag():
    """Through the C ABI: a lig_count above max_ligand_atoms empties the
    pose's rows and the fill reports it as *overflow = 2."""
    import ctypes as C
    from pointvs_b200 import _cabi
    from pointvs_b200.screening import Pocket
    rec, ligs = _synthetic(4)
    pocket = Pocket(rec, 4.0, 4.0)
    crop = pocket.crop(ligs, np.zeros(4, np.int32), np.inf, N_TYPES)
    n = int(crop.complex_ptr_host[-1])
    lib = _cabi.lib()
    # pose 0 claims one emitted ligand atom more than the bound passed below
    lc = torch.tensor([N_LIG + 1, N_LIG, N_LIG, N_LIG], dtype=torch.int32,
                      device='cuda')
    deg = torch.empty(n, dtype=torch.int32, device='cuda')
    n_inter = torch.empty(n, dtype=torch.int32, device='cuda')
    row_ptr = torch.empty(n + 1, dtype=torch.int32, device='cuda')
    scratch = torch.empty(int(lib.pvs_scan_scratch_bytes(n)) + 256,
                          dtype=torch.uint8, device='cuda')
    col = torch.empty(200000, dtype=torch.int32, device='cuda')
    attr = torch.empty(200000, dtype=torch.uint8, device='cuda')
    overflow = torch.zeros(1, dtype=torch.int32, device='cuda')
    args = (C.byref(pocket.desc), _cabi.ptr(crop.coords), _cabi.ptr(crop.complex_ptr),
            4, n, _cabi.ptr(crop.mask), crop.mask_words, _cabi.ptr(lc), N_LIG,
            _cabi.ptr(crop.rec_of_pose), C.c_double(4.0), C.c_double(4.0))
    _cabi.check(lib.pvs_pocket_graph_count(*args, _cabi.ptr(deg), _cabi.ptr(n_inter),
                                           _cabi.ptr(row_ptr), _cabi.ptr(scratch),
                                           _cabi.stream()))
    _cabi.check(lib.pvs_pocket_graph_fill(*args, _cabi.ptr(row_ptr), 200000,
                                          _cabi.ptr(col), _cabi.ptr(attr),
                                          _cabi.ptr(overflow), _cabi.stream()))
    assert int(overflow.item()) == 2
    cptr = crop.complex_ptr_host
    rp = row_ptr.cpu().numpy()
    assert rp[cptr[1]] == 0                   # pose 0: rows empty
    assert rp[cptr[2]] > 0                    # pose 1: its graph is built


def test_auto_capacity_queues_without_a_host_sync():
    """With edge_capacity='auto' the graph call returns while the stream is
    still busy with earlier work: nothing in it waits for the device."""
    from pointvs_b200.screening import Pocket
    rec, ligs = _synthetic(32)
    pocket = Pocket(rec, 4.0, 4.0)
    crop = pocket.crop(ligs, np.zeros(32, np.int32), np.inf, N_TYPES)
    pocket.radius_graph(crop, [N_LIG] * 32, edge_capacity='auto')   # warm
    torch.cuda.synchronize()
    torch.cuda._sleep(1 << 30)                # ~0.5 s of device time
    busy = torch.cuda.Event()
    busy.record()
    g = pocket.radius_graph(crop, [N_LIG] * 32, edge_capacity='auto')
    assert not busy.query()
    torch.cuda.synchronize()
    _, want, _ = _graphs(pocket, ligs, np.zeros(32, np.int32), np.inf)
    _assert_same_graph(want, g)


KW = dict(dim_input=13, dim_output=1, k=64, num_layers=3, graphnorm=False,
          edge_attention=True, node_attention=True, residual=True,
          normalize=True, tanh=True)


def _chain_scores(model, rec, ligs, radius, batch_size, edge_capacity):
    """The existing chain: crop_batch -> radius_graph_batch -> model."""
    import pointvs_b200 as pv
    from pointvs_b200 import data
    from pointvs_b200.graph import radius_graph_batch
    out = []
    for s in range(0, len(ligs), batch_size):
        part = ligs[s:s + batch_size]
        c, b, f, cp = data.crop_batch(part, [rec], np.zeros(len(part), np.int32),
                                      radius, N_TYPES, True, 'cuda')
        csr = radius_graph_batch(c, b, cp, 4.0, 4.0, device='cuda',
                                 edge_capacity=edge_capacity)
        with torch.no_grad():
            sc = model(pv.PackedBatch(f, c.float(), csr, csr.complex_ptr))
        out.append(torch.sigmoid(sc.reshape(len(part), -1)).cpu().numpy())
    return np.concatenate(out)


@pytest.mark.parametrize('multitask,k,math', [
    (False, 64, 'bf16x3'), (False, 64, 'fp32'), (True, 64, 'bf16x3'),
    (True, 64, 'fp32'), (False, 96, 'bf16x3'), (True, 128, 'bf16x3')])
def test_score_poses_is_the_chain_bit_for_bit(multitask, k, math):
    import pointvs_b200 as pv
    rec, ligs = _synthetic(80)
    model = gh.build_model(dict(KW, k=k), multitask=multitask, seed=3)
    model.set_math(math)
    model.set_record_side_channels(False)
    model.record_embed_coords = False
    pocket = pv.Pocket(rec, 4.0, 4.0)
    for radius, cap in ((None, 'auto'), (8.0, None)):
        got = pv.score_poses(model, pocket, ligs, radius=radius, batch_size=32,
                             n_features=N_TYPES, edge_capacity=cap)
        want = _chain_scores(model, rec, ligs,
                             np.inf if radius is None else radius, 32, cap)
        assert got.shape == want.shape == (80, want.shape[1])
        np.testing.assert_array_equal(got, want)


def test_score_poses_matches_parallel_screen():
    import pointvs_b200 as pv
    from pointvs_b200 import parallel
    rec, ligs = _synthetic(24)
    model = gh.build_model(KW, seed=4)
    model.set_record_side_channels(False)
    model.record_embed_coords = False
    pocket = pv.Pocket(rec, 4.0, 4.0)
    got = pv.score_poses(model, pocket, ligs, radius=9.0, batch_size=10,
                         n_features=N_TYPES, group=None, activation=None)
    crop = pocket.crop(ligs, np.zeros(24, np.int32), 9.0, N_TYPES)
    cptr = crop.complex_ptr_host
    coords, bp = crop.coords.cpu().numpy(), crop.bp.cpu().numpy()
    feats = crop.feats.cpu().numpy()
    complexes = [(coords[cptr[b]:cptr[b + 1]], bp[cptr[b]:cptr[b + 1]],
                  feats[cptr[b]:cptr[b + 1]]) for b in range(24)]
    want = parallel.screen(model, complexes, batch_size=7, activation=None)
    np.testing.assert_allclose(got, want, rtol=2e-5, atol=1e-6)
