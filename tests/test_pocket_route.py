"""(CPU) The device-crop loader's choice between K1p and K1:
`ComplexDataset.plan_pockets` (which receptors get a pocket) and
`ComplexDataset.pocket_route` (which builder a batch runs)."""
import numpy as np
import torch

from pointvs_b200 import _cabi, data


def _dataset(tmp_path, recs, cache=8):
    lines = [f'1 -1 -1.0 {r}.parquet lig/{i}.parquet' for i, r in enumerate(recs)]
    (tmp_path / 't.types').write_text('\n'.join(lines) + '\n')
    return data.ComplexDataset(tmp_path, types_fname=tmp_path / 't.types',
                               polar_hydrogens=False, device_crop=True,
                               receptor_cache=cache)


def _batches(n, size):
    return [list(range(s, min(n, s + size))) for s in range(0, n, size)]


def _route(ds, items, lig=30, rec_atoms=3000, complex_atoms=700):
    names = list(dict.fromkeys(ds.receptor_fnames[i] for i in items))
    return ds.pocket_route(items, {n: rec_atoms for n in names},
                           [lig] * len(items), [complex_atoms] * len(items))


def _resident(ds, name):
    dev = str(torch.device(ds.device or 'cuda'))
    ds._pockets[(name, dev)] = ((float(ds.inter_radius),
                                 float(ds.intra_radius)), object())


def test_threshold_counts_the_poses_of_a_residency(tmp_path):
    n = data.POCKET_MIN_POSES
    recs = ['a'] * n + ['b'] * (n - 1)
    ds = _dataset(tmp_path, recs)
    batches = _batches(len(recs), 64)
    ds.plan_pockets(batches)
    for items in batches:
        names = set(ds.receptor_fnames[i] for i in items)
        use, build = _route(ds, items)
        # 'a' reaches the threshold, 'b' falls one pose short
        assert use == (names == {'a.parquet'}), names
        if use:
            assert build == ['a.parquet']


def test_resident_pocket_is_reused_and_not_rebuilt(tmp_path):
    n = data.POCKET_MIN_POSES
    ds = _dataset(tmp_path, ['a'] * n)
    batches = _batches(n, 32)
    ds.plan_pockets(batches)
    assert _route(ds, batches[0]) == (True, ['a.parquet'])
    _resident(ds, 'a.parquet')
    for items in batches[1:]:
        assert _route(ds, items) == (True, [])


def test_eviction_splits_a_receptor_into_residencies(tmp_path):
    """With one resident receptor, a a b b a a ... never keeps 'a' resident
    for POCKET_MIN_POSES poses, although the file has more than that."""
    n = data.POCKET_MIN_POSES
    recs = []
    for _ in range(4):
        recs += ['a'] * (n // 2) + ['b'] * 8
    batches = _batches(len(recs), n // 2)
    ds = _dataset(tmp_path, recs, cache=1)
    ds.plan_pockets(batches)
    assert all(not _route(ds, items)[0] for items in batches)
    # with room for both, 'a' stays resident and gets its pocket
    ds = _dataset(tmp_path, recs, cache=2)
    ds.plan_pockets(batches)
    assert _route(ds, batches[0]) == (True, ['a.parquet'])


def test_eviction_drops_the_pocket(tmp_path):
    ds = _dataset(tmp_path, ['a', 'b'], cache=1)
    dev = torch.device('cuda')
    key_a = ('a.parquet', str(dev))
    ds._rec_dev[key_a] = 'receptor a'
    _resident(ds, 'a.parquet')
    # what receptor_on_device does when the LRU is full
    ds._rec_dev[('b.parquet', str(dev))] = 'receptor b'
    while len(ds._rec_dev) > max(1, ds._cache_size):
        gone, _ = ds._rec_dev.popitem(last=False)
        ds._pockets.pop(gone, None)
    assert key_a not in ds._pockets
    assert _route(ds, [0]) == (False, [])


def test_size_limits_fall_back_to_k1(tmp_path):
    n = data.POCKET_MIN_POSES
    ds = _dataset(tmp_path, ['a'] * n)
    batches = _batches(n, n)
    ds.plan_pockets(batches)
    items = batches[0]
    assert _route(ds, items)[0]
    assert _route(ds, items, lig=_cabi.POCKET_MAX_LIG_ATOMS)[0]
    assert _route(ds, items, lig=_cabi.POCKET_MAX_LIG_ATOMS + 1) == (False, [])
    assert _route(ds, items, rec_atoms=_cabi.POCKET_MAX_REC_ATOMS)[0]
    assert _route(ds, items, rec_atoms=_cabi.POCKET_MAX_REC_ATOMS + 1) == \
        (False, [])
    # one pose over the bound is enough
    lig = [30] * len(items)
    lig[7] = _cabi.POCKET_MAX_LIG_ATOMS + 1
    assert ds.pocket_route(items, {'a.parquet': 100}, lig,
                           [700] * len(items)) == (False, [])


def test_small_complexes_run_k1(tmp_path):
    n = data.POCKET_MIN_POSES
    ds = _dataset(tmp_path, ['a'] * n)
    items = _batches(n, n)[0]
    ds.plan_pockets([items])
    m = data.POCKET_MIN_COMPLEX_ATOMS
    assert _route(ds, items, complex_atoms=m)[0]
    assert _route(ds, items, complex_atoms=m - 1) == (False, [])
    # the batch mean decides
    sizes = [m - 100] * (len(items) // 2) + [m + 100] * (len(items) // 2)
    assert ds.pocket_route(items, {'a.parquet': 3000}, [30] * len(items),
                           sizes)[0]


def test_sampled_order_builds_nothing(tmp_path):
    n = data.POCKET_MIN_POSES
    ds = _dataset(tmp_path, ['a'] * (4 * n))
    ds.plan_pockets(None)
    assert all(_route(ds, items) == (False, [])
               for items in _batches(4 * n, 64))
    # a pocket already resident (an earlier pass in file order) still serves
    _resident(ds, 'a.parquet')
    assert _route(ds, [0, 5, 9]) == (True, [])


def test_sampler_loader_plans_nothing(tmp_path):
    n = data.POCKET_MIN_POSES
    recs = ['a'] * (2 * n)
    ds = _dataset(tmp_path, recs)
    loader = data.PackedLoader(ds, 64, sampler=list(np.arange(2 * n)[::-1]),
                               num_workers=0)
    ds.load_ligand = lambda i: None   # no parquet is read here
    next(iter(loader.prepared()))
    assert ds._pocket_plan is None
    loader = data.PackedLoader(ds, 64, sampler=None, num_workers=0)
    next(iter(loader.prepared()))
    assert ds._pocket_plan and all(v == {'a.parquet'}
                                   for v in ds._pocket_plan.values())


def test_mixed_receptor_batches(tmp_path):
    n = data.POCKET_MIN_POSES
    # the boundary batch mixes a and b; c is short of the threshold
    recs = ['a'] * (n + 16) + ['b'] * (n + 16) + ['c'] * 8
    ds = _dataset(tmp_path, recs)
    batches = _batches(len(recs), 64)
    ds.plan_pockets(batches)
    mixed = [b for b in batches
             if len(set(ds.receptor_fnames[i] for i in b)) > 1]
    assert len(mixed) == 2
    ab, bc = mixed
    assert set(ds.receptor_fnames[i] for i in ab) == {'a.parquet', 'b.parquet'}
    assert _route(ds, ab) == (True, ['a.parquet', 'b.parquet'])
    _resident(ds, 'a.parquet')
    assert _route(ds, ab) == (True, ['b.parquet'])
    _resident(ds, 'b.parquet')
    assert _route(ds, ab) == (True, [])
    # c has no pocket and gets none: the whole batch runs K1
    assert _route(ds, bc) == (False, [])


def test_other_radii_need_their_own_pocket(tmp_path):
    ds = _dataset(tmp_path, ['a'] * 4)
    ds.plan_pockets(None)
    _resident(ds, 'a.parquet')
    assert _route(ds, [0, 1])[0]
    ds.estimate_bonds = True     # intra radius 2: the resident pocket is 4 / 4
    assert _route(ds, [0, 1]) == (False, [])
