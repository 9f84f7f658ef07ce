"""K1p, the radius graph of ligand poses against a resident pocket (CPU side):
the C ABI refuses bad arguments before any launch, and the Python layer keeps
a pocket to its own radii and `crop_batch` to its old return value."""
import ctypes as C
import inspect

import pytest

FAKE = C.c_void_p(256)   # never dereferenced: the calls return before any launch


def _pocket(max_atoms=800, inter=4.0, intra=4.0, n_atoms=None):
    from pointvs_b200 import _cabi
    n_atoms = max_atoms if n_atoms is None else n_atoms
    return _cabi.PocketDesc(1, n_atoms, max_atoms, inter, intra, FAKE, FAKE,
                            FAKE, FAKE, FAKE, FAKE)


def _count(p, **kw):
    from pointvs_b200 import _cabi
    a = dict(coords=FAKE, cptr=FAKE, n_poses=4, n_nodes=3000, mask=FAKE,
             words=25, lig_count=FAKE, max_lig=30, rec_of_pose=None,
             inter=4.0, intra=4.0)
    a.update(kw)
    return _cabi.lib().pvs_pocket_graph_count(
        C.byref(p), a['coords'], a['cptr'], a['n_poses'], a['n_nodes'],
        a['mask'], a['words'], a['lig_count'], a['max_lig'], a['rec_of_pose'],
        C.c_double(a['inter']), C.c_double(a['intra']), FAKE, FAKE, FAKE,
        FAKE, None)


def _fill(p, **kw):
    from pointvs_b200 import _cabi
    a = dict(n_poses=4, n_nodes=3000, words=25, max_lig=30, inter=4.0,
             intra=4.0, capacity=1000, col=FAKE)
    a.update(kw)
    return _cabi.lib().pvs_pocket_graph_fill(
        C.byref(p), FAKE, FAKE, a['n_poses'], a['n_nodes'], FAKE, a['words'],
        FAKE, a['max_lig'], None, C.c_double(a['inter']),
        C.c_double(a['intra']), FAKE, a['capacity'], a['col'], FAKE, FAKE,
        None)


def test_capability_bit_and_limits():
    from pointvs_b200 import _cabi
    lib = _cabi.lib()
    assert lib.pvs_capabilities() & _cabi.CAP_POCKET
    assert _cabi.POCKET_MAX_LIG_ATOMS == 256
    assert _cabi.POCKET_MAX_REC_ATOMS == 65536
    assert lib.pvs_pocket_cells_bytes(2, 5000) > lib.pvs_pocket_cells_bytes(1, 800) > 0
    assert lib.pvs_pocket_cells_bytes(-1, 10) == -1
    assert lib.pvs_pocket_build_scratch_bytes(1, 800) >= 800 * 4
    assert lib.pvs_pocket_build_scratch_bytes(1, -1) == -1


def test_null_or_negative_arguments_fail_before_any_launch():
    from pointvs_b200 import _cabi
    lib = _cabi.lib()
    n0 = lib.pvs_launch_count()
    ok = _pocket()
    assert lib.pvs_pocket_build_count(None, FAKE, None) == 1
    assert lib.pvs_pocket_build_count(C.byref(_pocket(max_atoms=-1)), FAKE, None) == 1
    assert lib.pvs_pocket_build_count(C.byref(ok), None, None) == 1
    bad = _pocket()
    bad.xyz = None
    assert lib.pvs_pocket_build_count(C.byref(bad), FAKE, None) == 1
    bad = _pocket()
    bad.rr_col = None
    assert lib.pvs_pocket_build_fill(C.byref(bad), None) == 1
    assert lib.pvs_pocket_build_count(C.byref(_pocket(inter=-1.0)), FAKE, None) == 1
    for kw in (dict(n_poses=-1), dict(n_nodes=-1), dict(words=-1),
               dict(max_lig=-1), dict(coords=None), dict(cptr=None),
               dict(mask=None), dict(lig_count=None), dict(inter=-4.0, intra=-4.0),
               dict(words=24)):   # 24 words hold 768 < 800 receptor atoms
        assert _count(ok, **kw) == 1, kw
    for kw in (dict(capacity=-1), dict(col=None), dict(n_poses=-1)):
        assert _fill(ok, **kw) == 1, kw
    assert lib.pvs_launch_count() == n0


def test_radius_mismatch_with_the_pocket_is_an_error():
    ok = _pocket(inter=4.0, intra=2.0)
    for inter, intra in ((4.0, 4.0), (2.0, 2.0), (5.0, 2.0)):
        assert _count(ok, inter=inter, intra=intra) == 1
        assert _fill(ok, inter=inter, intra=intra) == 1


def test_over_bound_ligand_and_receptor_return_too_large():
    from pointvs_b200 import _cabi
    lib = _cabi.lib()
    bound = _cabi.POCKET_MAX_LIG_ATOMS
    assert _count(_pocket(), max_lig=bound + 1) == 3
    assert _fill(_pocket(), max_lig=bound + 1) == 3
    big = _pocket(max_atoms=_cabi.POCKET_MAX_REC_ATOMS + 1)
    assert lib.pvs_pocket_build_count(C.byref(big), FAKE, None) == 3
    assert _count(big, words=(_cabi.POCKET_MAX_REC_ATOMS + 32) // 32) == 3
    assert b'too large' in lib.pvs_status_string(3)


def test_pocket_rejects_radii_other_than_its_own():
    from pointvs_b200.screening import Pocket
    pocket = Pocket.__new__(Pocket)      # radii only: no device state needed
    pocket.inter_radius, pocket.intra_radius = 4.0, 2.0
    pocket.check_radii(4, 2)
    with pytest.raises(ValueError, match='radii'):
        pocket.check_radii(4.0, 4.0)
    with pytest.raises(ValueError, match='radii'):
        pocket.radius_graph(None, [], inter_radius=4.0, intra_radius=4.0)
    with pytest.raises(ValueError, match='non-negative'):
        Pocket([], -1.0, 2.0)


def test_crop_batch_keeps_its_signature_and_four_tuple():
    from pointvs_b200 import data
    params = list(inspect.signature(data.crop_batch).parameters)
    assert params == ['ligands', 'receptors', 'rec_of_pose', 'radius',
                      'n_features', 'compact', 'device', 'receptors_pending']
    out = data.crop_batch([], [], [], 4.0, 11, True, 'cpu')
    assert isinstance(out, tuple) and len(out) == 4
    coords, bp, feats, cptr = out
    assert tuple(coords.shape) == (0, 3) and tuple(feats.shape) == (0, 12)
    assert list(cptr) == [0]


def test_package_exports():
    import pointvs_b200 as pv
    assert 'Pocket' in pv.__all__ and 'score_poses' in pv.__all__
    params = list(inspect.signature(pv.score_poses).parameters)
    assert params == ['model', 'pocket', 'ligands', 'rec_of_pose', 'radius',
                      'batch_size', 'n_features', 'compact', 'edge_capacity',
                      'group', 'activation']
