"""Types-file / parquet complex loader feeding the device graph builder (N2).

Host-side mirror of the scoring-relevant part of the reference's
`PygPointCloudDataset` + `get_data_loader`
(/root/reference/point_vs/preprocessing/data_loaders.py:33-520) and the
preprocessing helpers it calls (`concat_structs`, `make_box`,
`make_bit_vector`, preprocessing/preprocessing.py:165-300): parse the types
file, read the receptor/ligand parquets, crop the receptor to the atoms within
`radius` of any ligand atom, drop hydrogens, type the atoms, one-hot them.

Where the reference then calls `generate_edges` per complex on the CPU and lets
PyG collate the graphs, this loader packs the whole mini-batch into flat host
arrays and hands them to K1 once (`PackedBatch.from_arrays`), so the radius
graph of the batch is built on the device in destination-sorted CSR form.

Reference features that only make sense for augmentation-heavy training are
refused loudly rather than approximated (`augmented_active_count`,
`p_remove_entity`, `p_noise`, `bp`, `include_strain_info`, `prune`: with
`prune=True` the reference itself returns node features for the unpruned
structure and edges indexed into the pruned one).  `rot=True` draws a rotation
with the same distribution (Arvo 1992) from this module's own RNG stream; EGNN
scores are invariant to it.
"""
import math
import threading
from collections import OrderedDict, deque
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np
import torch

from .graph import PackedBatch

_COLUMNS = ('x', 'y', 'z', 'atomic_number', 'types', 'bp')

# Device-crop batches run K1p (screening.Pocket) instead of K1 where it pays
# (profiles/README.md, "Pocket route of the device-crop loader"; B200, 1000 W):
# * K1p's graph stage beats K1's from 681 atoms per complex up (1.26x at 681,
#   7.4x at 5469) and loses below 381 (0.93-0.95x for whole proteins at a
#   10 A crop around 18-atom ligands), so a batch whose complexes average
#   fewer atoms than POCKET_MIN_COMPLEX_ATOMS runs K1;
# * a pocket build takes 0.20-0.23 ms (1754-5450 atoms) and the smallest
#   saving measured where K1p is chosen is 0.23 us per pose, so a receptor
#   gets a pocket only when at least POCKET_MIN_POSES poses will use it while
#   it stays resident.
POCKET_MIN_COMPLEX_ATOMS = 512
POCKET_MIN_POSES = 1024


# --------------------------------------------------------------------------
# types files
# --------------------------------------------------------------------------
def parse_classification_types(types_fname):
    """`classifiaction_types_to_lists` (data_loaders.py:560-642) without the
    strain columns: -> (labels, rmsds, receptors, ligands).

    Line format `<label> <...> <rmsd> <receptor> <ligand> <...>`; a two-column
    line is `<receptor> <ligand>` with label None.  The first token that is
    not a number is the receptor (the token before it is the rmsd), the next
    one the ligand; tokens starting with '#' are skipped."""
    labels, rmsds, recs, ligs = [], [], [], []
    with open(Path(types_fname).expanduser(), 'r', encoding='utf-8') as f:
        for line in f:
            chunks = line.strip().split()
            if not chunks:
                continue
            if len(chunks) == 2:
                label, rmsd, rec, lig = None, None, chunks[0], chunks[1]
            else:
                try:
                    label = int(chunks[0])
                except ValueError:
                    label = None
                rmsd = rec = lig = None
                for idx, chunk in enumerate(chunks):
                    if chunk.startswith('#'):
                        continue
                    try:
                        float(chunk)
                    except ValueError:
                        if rec is None:
                            rec = chunk
                            rmsd = float(chunks[idx - 1])
                        else:
                            # the reference keeps overwriting: last one wins
                            lig = chunk
            if rec is not None and lig is not None:
                labels.append(label)
                rmsds.append(rmsd)
                recs.append(rec)
                ligs.append(lig)
    return labels, rmsds, recs, ligs


def parse_regression_types(data_root, types_fname):
    """`regression_types_to_lists` (data_loaders.py:523-557): whitespace
    separated `<pki> <pkd> <ic50> <receptor> <ligand>` (or the two paths
    only); entries whose files are missing under `data_root` are dropped."""
    rows = []
    with open(Path(types_fname).expanduser(), 'r', encoding='utf-8') as f:
        for line in f:
            chunks = line.strip().split()
            if chunks:
                rows.append(chunks)
    if not rows:
        return [], [], [], [], []
    n_cols = len(rows[0])
    pki, pkd, ic50, recs, ligs = [], [], [], [], []
    for chunks in rows:
        if n_cols >= 5:
            a, b, c, rec, lig = chunks[:5]
            a, b, c = float(a), float(b), float(c)
        else:
            a = b = c = None
            rec, lig = chunks[-2], chunks[-1]
        if Path(data_root, rec).is_file() and Path(data_root, lig).is_file():
            pki.append(a)
            pkd.append(b)
            ic50.append(c)
            recs.append(rec)
            ligs.append(lig)
    return pki, pkd, ic50, recs, ligs


# --------------------------------------------------------------------------
# one complex
# --------------------------------------------------------------------------
def read_structure(path):
    """Parquet -> dict of numpy columns (x, y, z f64; atomic_number, types, bp
    i64), as `pd.read_parquet` gives the reference."""
    import pyarrow.parquet as pq   # noqa: PLC0415 (keeps import torch-light)
    # ParquetFile skips the dataset/filesystem discovery of pq.read_table
    table = pq.ParquetFile(str(path)).read(columns=list(_COLUMNS),
                                           use_threads=False)
    out = {}
    for name in _COLUMNS:
        col = table.column(name).to_numpy()
        out[name] = np.ascontiguousarray(
            col, dtype=np.float64 if name in 'xyz' else np.int64)
    return out


def atomic_number_table(polar_hydrogens):
    """`PointCloudDataset.__init__` (data_loaders.py:199-223): index of each
    recognised element, elements sharing valence properties grouped, every
    other element mapped to `n_features` itself.  -> (dict, n_features)."""
    recognised = (6, 7, 8, 9, 15, 16, 17)
    groupings = ((35, 53), (3, 11, 19), (4, 12, 20), (26, 29, 30))
    table = {num: idx for idx, num in enumerate(recognised)}
    for grouping in groupings:
        nxt = max(table.values()) + 1
        table.update({elem: nxt for elem in grouping})
    if polar_hydrogens:
        table[1] = max(table.values()) + 1
    return table, max(table.values()) + 1


def make_box(lig_xyz, rec_xyz, radius):
    """Indices of the receptor atoms closer than `radius` to any ligand atom
    (`make_box(relative_to_ligand=True)`, preprocessing.py:165-195).  Same
    fp64 arithmetic as scipy's euclidean `cdist`: sqrt(dx²+dy²+dz²) < radius."""
    if len(lig_xyz) == 0 or len(rec_xyz) == 0:
        return np.zeros(0, dtype=np.int64)
    # exact prefilter: an atom outside the ligand's bounding box grown by
    # `radius` (plus slack for rounding) cannot pass the distance test
    lo = lig_xyz.min(axis=0) - radius * (1 + 1e-9) - 1e-9
    hi = lig_xyz.max(axis=0) + radius * (1 + 1e-9) + 1e-9
    near = np.nonzero(((rec_xyz >= lo) & (rec_xyz <= hi)).all(axis=1))[0]
    d = lig_xyz[:, None, :] - rec_xyz[None, near, :]
    dist = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]
                   + d[..., 2] * d[..., 2])
    return near[(dist < radius).any(axis=0)]


def make_bit_vector(atom_types, n_atom_types, compact=True):
    """`make_bit_vector` (preprocessing.py:214-239) -> float32 [N, F].
    compact: one-hot of `type % n` over n + 1 columns, the last column then
    overwritten with `type // n` (0 ligand, 1 receptor)."""
    atom_types = np.asarray(atom_types, dtype=np.int64)
    n = len(atom_types)
    if compact:
        out = np.zeros((n, n_atom_types + 1), dtype=np.float32)
        out[np.arange(n), atom_types % n_atom_types] = 1.0
        out[:, -1] = (atom_types // n_atom_types).astype(np.float32)
    else:
        if n and (atom_types.min() < 0 or atom_types.max() >= 2 * n_atom_types):
            raise ValueError('atom type outside the one-hot range')
        out = np.zeros((n, 2 * n_atom_types), dtype=np.float32)
        out[np.arange(n), atom_types] = 1.0
    return out


def uniform_random_rotation(x, rng):
    """Arvo's fast random rotation, as preprocessing.py:30-53, drawing from
    `rng` (a numpy Generator) instead of the global numpy state."""
    x1, x2, x3 = rng.random(), 2 * np.pi * rng.random(), rng.random()
    rot = np.eye(3)
    rot[0, 0] = rot[1, 1] = np.cos(2 * np.pi * x1)
    rot[0, 1] = -np.sin(2 * np.pi * x1)
    rot[1, 0] = np.sin(2 * np.pi * x1)
    v = np.array([np.cos(x2) * np.sqrt(x3), np.sin(x2) * np.sqrt(x3),
                  np.sqrt(1 - x3)])
    m = -((np.eye(3) - 2 * np.outer(v, v)) @ rot)
    mean = x.mean(axis=0)
    return ((x - mean) @ m) + mean @ m


class Ligand:
    """Host-side half of a complex for the device crop: every ligand atom
    (hydrogens included: they take part in the box test), which of them are
    emitted, and the type code of each."""
    __slots__ = ('coords', 'emit', 'code')

    def __init__(self, coords, emit, code):
        self.coords, self.emit, self.code = coords, emit, code

    def __len__(self):
        return len(self.emit)


def atom_codes(cols, n_features, is_receptor, polar_hydrogens,
               use_atomic_numbers, atomic_number_to_index):
    """(emit u8, code i16) per atom of one parquet: what parquets_to_inputs
    (data_loaders.py:285-292) does to `types` after the box."""
    anum = cols['atomic_number']
    emit = np.ones(len(anum), dtype=np.uint8) if polar_hydrogens \
        else (anum > 1).astype(np.uint8)
    if use_atomic_numbers:
        code = np.array([atomic_number_to_index.get(int(a), n_features)
                         for a in anum], dtype=np.int64).reshape(len(anum))
        code = code + (n_features if is_receptor else 0)
    else:
        code = cols['types'] + (n_features if is_receptor else 0)
    return emit, code.astype(np.int16)


class Complex:
    """One preprocessed complex on the host."""
    __slots__ = ('coords', 'bp', 'feats', 'types', 'atomic_number')

    def __init__(self, coords, bp, feats, types, atomic_number):
        self.coords, self.bp, self.feats = coords, bp, feats
        self.types, self.atomic_number = types, atomic_number

    def __len__(self):
        return len(self.bp)


def build_complex(rec, lig, n_features, radius, polar_hydrogens=False,
                  use_atomic_numbers=False, compact=True,
                  atomic_number_to_index=None):
    """`parquets_to_inputs` (data_loaders.py:259-310) on column dicts:
    concat [ligand; receptor] with receptor types shifted by n_features, box,
    hydrogen filter, optional atomic-number typing, one-hot."""
    cols = {}
    for name in _COLUMNS:
        cols[name] = np.concatenate([lig[name], rec[name]])
    cols['types'] = cols['types'].copy()
    cols['types'][len(lig['types']):] += n_features
    xyz = np.stack([cols['x'], cols['y'], cols['z']], axis=1)
    lig_idx = np.nonzero(cols['bp'] == 0)[0]
    rec_idx = np.nonzero(cols['bp'] == 1)[0]
    keep_rec = rec_idx[make_box(xyz[lig_idx], xyz[rec_idx], radius)]
    keep = np.concatenate([lig_idx, keep_rec])
    if not polar_hydrogens:
        keep = keep[cols['atomic_number'][keep] > 1]
    bp = cols['bp'][keep]
    anum = cols['atomic_number'][keep]
    if use_atomic_numbers:
        idx = np.array([atomic_number_to_index.get(int(a), n_features)
                        for a in anum], dtype=np.int64).reshape(len(anum))
        types = idx + bp * n_features
    else:
        types = cols['types'][keep]
    feats = make_bit_vector(types, n_features, compact)
    return Complex(np.ascontiguousarray(xyz[keep]), bp.astype(np.int32), feats,
                   types, anum)


_SIDE_STREAMS = {}


def _side_stream(device):
    """One high-priority stream per device for the K0 counting pass."""
    key = (device.type, device.index if device.index is not None
           else torch.cuda.current_device())
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device, priority=-1)
    return _SIDE_STREAMS[key]


def crop_batch(ligands, receptors, rec_of_pose, radius, n_features, compact,
               device, receptors_pending=False):
    """K0 (pvs_crop_count / pvs_crop_fill) for one batch of poses.

    ligands: list of `Ligand`; receptors: list of (xyz f64 [n,3], emit u8 [n],
    code i16 [n]) tensors already on `device`; rec_of_pose[b] indexes them.
    -> (coords f64 [N,3], bp i32 [N], feats f32 [N,F]) on the device and the
    host complex_ptr [B+1].

    One host read-back (the B+1 offsets) sizes the outputs.  The ligand
    upload, the counting pass and that read-back run on a side stream, so the
    host does not wait for whatever the caller's stream is still doing (the
    previous batch's layers); the fill joins the caller's stream.  The
    receptor tensors must already be complete on the device (synchronise once
    after uploading them), or pass receptors_pending=True to order the side
    stream after the caller's stream."""
    out = crop_batch_masked(ligands, receptors, rec_of_pose, radius, n_features,
                            compact, device, receptors_pending)
    return out.coords, out.bp, out.feats, out.complex_ptr_host


class CropOutput:
    """What K0 leaves on the device for one batch: the assembled complexes,
    their offsets (host and device), and the per-pose receptor keep bits
    (`mask_words` uint32 words per pose) that K1p consumes."""
    __slots__ = ('coords', 'bp', 'feats', 'complex_ptr_host', 'complex_ptr',
                 'mask', 'mask_words', 'rec_of_pose')

    def __init__(self, **kw):
        for k, v in kw.items():
            setattr(self, k, v)


def crop_batch_masked(ligands, receptors, rec_of_pose, radius, n_features,
                      compact, device, receptors_pending=False,
                      concatenated=None):
    """`crop_batch` that also returns K0's keep-bit mask (-> CropOutput).
    concatenated: the receptors already concatenated, (xyz, emit, code), so
    a resident pocket skips the per-batch copy."""
    import ctypes as C   # noqa: PLC0415
    from . import _cabi   # noqa: PLC0415
    from ._cabi import check, lib, ptr, stream   # noqa: PLC0415
    device = torch.device(device)
    n_poses = len(ligands)
    feature_dim = n_features + 1 if compact else 2 * n_features
    if n_poses == 0:
        return CropOutput(
            coords=torch.zeros((0, 3), dtype=torch.float64, device=device),
            bp=torch.zeros(0, dtype=torch.int32, device=device),
            feats=torch.zeros((0, feature_dim), device=device),
            complex_ptr_host=np.zeros(1, dtype=np.int32),
            complex_ptr=torch.zeros(1, dtype=torch.int32, device=device),
            mask=None, mask_words=0, rec_of_pose=None)
    rec_sizes = [int(r[0].shape[0]) for r in receptors]
    rec_ptr = np.zeros(len(receptors) + 1, dtype=np.int32)
    np.cumsum(rec_sizes, out=rec_ptr[1:])
    lig_ptr = np.zeros(n_poses + 1, dtype=np.int32)
    np.cumsum([len(l) for l in ligands], out=lig_ptr[1:])
    lig_code_h = np.concatenate([l.code for l in ligands])
    if not compact and len(lig_code_h) and (
            lig_code_h.min() < 0 or lig_code_h.max() >= 2 * n_features):
        raise ValueError('atom type outside the one-hot range')
    words = max((max(rec_sizes) + 31) // 32 if rec_sizes else 0, 1)
    h = lib()
    main = torch.cuda.current_stream(device)
    side = _side_stream(device)
    if receptors_pending:
        side.wait_stream(main)
    with torch.cuda.device(device), torch.cuda.stream(side):
        if concatenated is not None:
            rec_xyz, rec_emit, rec_code = concatenated
        elif len(receptors) == 1:
            rec_xyz, rec_emit, rec_code = receptors[0]
        else:
            rec_xyz = torch.cat([r[0] for r in receptors])
            rec_emit = torch.cat([r[1] for r in receptors])
            rec_code = torch.cat([r[2] for r in receptors])
        lig_xyz = torch.from_numpy(
            np.concatenate([l.coords for l in ligands])).to(device)
        lig_emit = torch.from_numpy(
            np.concatenate([l.emit for l in ligands])).to(device)
        lig_code = torch.from_numpy(lig_code_h).to(device)
        lig_ptr_d = torch.from_numpy(lig_ptr).to(device)
        rec_ptr_d = torch.from_numpy(rec_ptr).to(device)
        rec_of_pose_d = torch.from_numpy(
            np.ascontiguousarray(rec_of_pose, dtype=np.int32)).to(device)
        mask = torch.empty(n_poses * words, dtype=torch.int32, device=device)
        counts = torch.empty(n_poses, dtype=torch.int32, device=device)
        cptr = torch.empty(n_poses + 1, dtype=torch.int32, device=device)
        scan_ws = torch.empty(int(h.pvs_scan_scratch_bytes(n_poses)) + 256,
                              dtype=torch.uint8, device=device)
        sptr = C.c_void_p(side.cuda_stream)
        check(h.pvs_crop_count(
            ptr(lig_xyz), ptr(lig_emit), ptr(lig_ptr_d), n_poses,
            ptr(rec_xyz), ptr(rec_emit), ptr(rec_ptr_d), ptr(rec_of_pose_d),
            words, C.c_double(float(radius)), ptr(mask), ptr(counts), sptr),
            'pvs_crop_count')
        check(h.pvs_exclusive_scan(ptr(counts), n_poses, ptr(cptr),
                                   ptr(scan_ws), sptr), 'pvs_exclusive_scan')
        cptr_host = cptr.cpu().numpy()          # waits for the side stream only
    n = int(cptr_host[-1])
    with torch.cuda.device(device):
        main.wait_stream(side)
        coords = torch.empty((max(n, 1), 3), dtype=torch.float64,
                             device=device)
        bp = torch.empty(max(n, 1), dtype=torch.int32, device=device)
        feats = torch.empty((max(n, 1), feature_dim), dtype=torch.float32,
                            device=device)
        check(h.pvs_crop_fill(
            ptr(lig_xyz), ptr(lig_emit), ptr(lig_code), ptr(lig_ptr_d),
            n_poses, ptr(rec_xyz), ptr(rec_code), ptr(rec_ptr_d),
            ptr(rec_of_pose_d), ptr(mask), words, ptr(cptr), n_features,
            int(bool(compact)), ptr(coords), ptr(bp), ptr(feats), stream()),
            'pvs_crop_fill')
        # allocated on the side stream, last read on the caller's stream
        for t in (lig_xyz, lig_emit, lig_code, lig_ptr_d, rec_ptr_d,
                  rec_of_pose_d, mask, cptr, rec_xyz, rec_code):
            t.record_stream(main)
    return CropOutput(coords=coords[:n], bp=bp[:n], feats=feats[:n],
                      complex_ptr_host=cptr_host, complex_ptr=cptr, mask=mask,
                      mask_words=words, rec_of_pose=rec_of_pose_d)


# --------------------------------------------------------------------------
# dataset + loader
# --------------------------------------------------------------------------
class ComplexDataset:
    """Mirror of `PygPointCloudDataset` (constructor argument names and
    defaults of data_loaders.py:36-47).  `dataset[i]` is a one-complex
    `PackedBatch`; `dataset.load(i)` the host-side `Complex`."""

    def __init__(self, base_path, radius=12, polar_hydrogens=True,
                 use_atomic_numbers=False, compact=True, rot=False,
                 augmented_active_count=0, augmented_active_min_angle=90,
                 max_active_rms_distance=None, min_inactive_rms_distance=None,
                 max_inactive_rms_distance=None, fname_suffix='parquet',
                 model_task='classification', types_fname=None,
                 edge_radius=None, estimate_bonds=False, prune=False, bp=None,
                 p_remove_entity=0, extended_atom_types=False, p_noise=-1,
                 include_strain_info=False, device=None, seed=None,
                 receptor_cache=8, device_crop=False, **kwargs):
        del augmented_active_min_angle, fname_suffix, kwargs
        if (max_active_rms_distance is None) != (
                min_inactive_rms_distance is None):
            raise AssertionError('max_active_rms_distance and '
                                 'min_inactive_rms_distance go together')
        for name, bad in (('augmented_active_count', augmented_active_count),
                          ('p_remove_entity', p_remove_entity > 0),
                          ('p_noise', p_noise > 0), ('bp', bp is not None),
                          ('include_strain_info', include_strain_info),
                          ('prune', prune)):
            if bad:
                raise NotImplementedError(
                    f'{name} is not supported by the packed-batch loader')
        if types_fname is None:
            raise ValueError('types_fname is required')
        self.base_path = Path(base_path).expanduser()
        if not self.base_path.exists():
            raise FileNotFoundError(
                f'Dataset {self.base_path} does not exist.')
        self.radius, self.edge_radius = radius, edge_radius
        self.estimate_bonds = estimate_bonds
        self.polar_hydrogens = polar_hydrogens
        self.use_atomic_numbers, self.compact = use_atomic_numbers, compact
        self.model_task, self.rot = model_task, rot
        self.device = device
        # device_crop: receptors stay resident in HBM and the box / hydrogen
        # filter / typing / one-hot of every pose run on the GPU (K0)
        self.device_crop = bool(device_crop)
        self._rec_dev = OrderedDict()
        # resident pockets (K1p), keyed as _rec_dev and dropped with it, and
        # the receptors worth one per upcoming batch (plan_pockets)
        self._pockets = {}
        self._pocket_plan = None
        self.use_types = True
        self._rng = np.random.default_rng(seed)
        self._cache = OrderedDict()
        self._cache_size = receptor_cache
        self._cache_lock = threading.Lock()

        self.sampler = None
        if model_task.endswith('regression'):
            (self.pki, self.pkd, self.ic50, self.receptor_fnames,
             self.ligand_fnames) = parse_regression_types(
                 self.base_path, types_fname)
            labels = []
        else:
            labels, rmsds, recs, ligs = parse_classification_types(types_fname)
            label_by_rmsd = (max_active_rms_distance is not None
                             or min_inactive_rms_distance is not None
                             or max_inactive_rms_distance is not None)
            if label_by_rmsd:
                # pose selection: relabel by rmsd from the crystal pose
                # (data_loaders.py:137-154)
                hi_act = np.inf if max_active_rms_distance is None \
                    else max_active_rms_distance
                hi_inact = np.inf if max_inactive_rms_distance is None \
                    else max_inactive_rms_distance
                lo_inact = 0 if min_inactive_rms_distance is None \
                    else min_inactive_rms_distance
                keep_labels, keep_recs, keep_ligs = [], [], []
                for rmsd, rec, lig in zip(rmsds, recs, ligs):
                    if rmsd < 0:
                        continue
                    if rmsd < hi_act:
                        lab = 1
                    elif rmsd >= hi_inact:
                        continue
                    elif rmsd >= lo_inact:
                        lab = 0
                    else:
                        continue
                    keep_labels.append(lab)
                    keep_recs.append(rec)
                    keep_ligs.append(lig)
                labels, recs, ligs = keep_labels, keep_recs, keep_ligs
            self.receptor_fnames, self.ligand_fnames = recs, ligs
            labels = np.array(labels)
            if len(labels) and labels[0] is not None:
                active = np.sum(labels)
                if 0 < active < len(labels):
                    weights = 1.0 / np.array([len(labels) - active, active])
                    self.sample_weights = torch.from_numpy(
                        np.array([weights[i] for i in labels]))
                    self.sampler = torch.utils.data.WeightedRandomSampler(
                        self.sample_weights, len(self.sample_weights))
        self.labels = labels
        self.pre_aug_ds_len = len(self.ligand_fnames)

        if use_atomic_numbers:
            self.atomic_number_to_index, self.n_features = \
                atomic_number_table(polar_hydrogens)
        elif polar_hydrogens:
            raise NotImplementedError('Hydrogens temporarily disabled.')
        else:
            self.atomic_number_to_index = None
            self.n_features = 11 + 8 * bool(extended_atom_types)
        self.feature_dim = self.n_features + 1 if compact \
            else self.n_features * 2

    def __len__(self):
        return len(self.ligand_fnames)

    # worker processes get a copy without locks, caches or device tensors
    def __getstate__(self):
        state = dict(self.__dict__)
        state['_cache_lock'] = None
        state['_cache'] = OrderedDict()
        state['_rec_dev'] = OrderedDict()
        state['_pockets'] = {}
        state['_pocket_plan'] = None
        state['sampler'] = None
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self._cache_lock = threading.Lock()

    # edge radii exactly as PygPointCloudDataset.__getitem__ (:356-357)
    @property
    def inter_radius(self):
        return self.edge_radius if (self.edge_radius or 0) > 0 else 4

    @property
    def intra_radius(self):
        return 2.0 if self.estimate_bonds else self.inter_radius

    def label(self, item):
        """`index_to_parquets` label (:229-237)."""
        if self.model_task == 'classification':
            return self.labels[item]
        trio = (self.pki[item], self.pkd[item], self.ic50[item])
        if self.model_task == 'multi_regression':
            return trio
        return None if trio[0] is None else max(trio)

    def _receptor(self, path):
        with self._cache_lock:
            hit = self._cache.get(path)
            if hit is not None:
                self._cache.move_to_end(path)
                return hit
        cols = read_structure(path)
        with self._cache_lock:
            self._cache[path] = cols
            while len(self._cache) > self._cache_size:
                self._cache.popitem(last=False)
        return cols

    def load(self, item):
        """Host-side preprocessing of complex `item` -> Complex."""
        rec_path = self.base_path / self.receptor_fnames[item]
        lig_path = self.base_path / self.ligand_fnames[item]
        if not lig_path.is_file():
            raise FileNotFoundError(lig_path, 'does not exist.')
        if not rec_path.is_file():
            raise FileNotFoundError(rec_path, 'does not exist')
        return build_complex(
            self._receptor(rec_path), read_structure(lig_path),
            self.n_features, self.radius, self.polar_hydrogens,
            self.use_atomic_numbers, self.compact, self.atomic_number_to_index)

    # -- device crop (K0) -----------------------------------------------------
    def load_ligand(self, item):
        """Host-side half of the device-crop path: the ligand parquet only."""
        lig_path = self.base_path / self.ligand_fnames[item]
        if not lig_path.is_file():
            raise FileNotFoundError(lig_path, 'does not exist.')
        cols = read_structure(lig_path)
        if cols['bp'].any():
            raise ValueError(f'{lig_path}: ligand file with bp != 0 rows; use '
                             'device_crop=False')
        emit, code = atom_codes(cols, self.n_features, False,
                                self.polar_hydrogens, self.use_atomic_numbers,
                                self.atomic_number_to_index)
        xyz = np.stack([cols['x'], cols['y'], cols['z']], axis=1)
        return Ligand(np.ascontiguousarray(xyz), emit, code)

    def receptor_on_device(self, rec_fname, device):
        """(xyz f64 [n,3], emit u8 [n], code i16 [n]) resident on `device`."""
        key = (str(rec_fname), str(device))
        with self._cache_lock:
            hit = self._rec_dev.get(key)
            if hit is not None:
                self._rec_dev.move_to_end(key)
                return hit
        rec_path = self.base_path / rec_fname
        if not rec_path.is_file():
            raise FileNotFoundError(rec_path, 'does not exist')
        cols = self._receptor(rec_path)
        if not cols['bp'].all():
            raise ValueError(f'{rec_path}: receptor file with bp != 1 rows; '
                             'use device_crop=False')
        emit, code = atom_codes(cols, self.n_features, True,
                                self.polar_hydrogens, self.use_atomic_numbers,
                                self.atomic_number_to_index)
        xyz = np.stack([cols['x'], cols['y'], cols['z']], axis=1)
        entry = (torch.from_numpy(np.ascontiguousarray(xyz)).to(device),
                 torch.from_numpy(emit).to(device),
                 torch.from_numpy(code).to(device))
        # complete before any other stream (K0's side stream) reads them
        torch.cuda.current_stream(device).synchronize()
        with self._cache_lock:
            self._rec_dev[key] = entry
            while len(self._rec_dev) > max(1, self._cache_size):
                gone, _ = self._rec_dev.popitem(last=False)
                self._pockets.pop(gone, None)
        return entry

    # -- resident pockets (K1p) -----------------------------------------------
    def plan_pockets(self, batches):
        """Decide, for the batch sequence `batches` (lists of items, in the
        order they will be packed), which receptors get a pocket: those that
        at least POCKET_MIN_POSES poses use while they stay resident.  The
        residency follows the device receptor LRU (`receptor_cache`) from its
        present state.  batches=None (a sampled order) builds none."""
        if batches is None:
            self._pocket_plan = None
            return
        dev = str(torch.device(self.device or 'cuda'))
        cap = max(1, self._cache_size)
        lru = OrderedDict((k[0], None) for k in self._rec_dev if k[1] == dev)
        # residency: [poses, batch keys]; one per receptor upload
        current, residencies = {}, []
        for items in batches:
            names = list(dict.fromkeys(str(self.receptor_fnames[i])
                                       for i in items))
            for name in names:
                if name in lru:
                    lru.move_to_end(name)
                else:
                    lru[name] = None
                    current.pop(name, None)
                    while len(lru) > cap:
                        gone, _ = lru.popitem(last=False)
                        current.pop(gone, None)
                if name not in current:
                    current[name] = [0, []]
                    residencies.append((name, current[name]))
                res = current[name]
                res[0] += sum(1 for i in items
                              if str(self.receptor_fnames[i]) == name)
                res[1].append(tuple(items))
        plan = {}
        for name, (poses, keys) in residencies:
            if poses >= POCKET_MIN_POSES:
                for key in keys:
                    plan.setdefault(key, set()).add(name)
        self._pocket_plan = plan

    def pocket_route(self, items, rec_atoms, lig_atoms, complex_atoms):
        """The graph builder of device-crop batch `items`: -> (use_k1p,
        names of the receptors whose pocket to build first).

        rec_atoms: atoms of each receptor of the batch (name -> int);
        lig_atoms: emitted ligand atoms of each pose; complex_atoms: atoms of
        each complex K0 assembled.  K1p runs when every receptor has a
        resident pocket for the dataset's radii (or the plan builds it now),
        every receptor and pose is within K1p's bounds and the complexes
        average at least POCKET_MIN_COMPLEX_ATOMS atoms; anything else runs
        K1, which builds the same graph."""
        from ._cabi import (POCKET_MAX_LIG_ATOMS,   # noqa: PLC0415
                            POCKET_MAX_REC_ATOMS)
        if not items or max(lig_atoms) > POCKET_MAX_LIG_ATOMS or \
                max(rec_atoms.values()) > POCKET_MAX_REC_ATOMS or \
                np.mean(complex_atoms) < POCKET_MIN_COMPLEX_ATOMS:
            return False, []
        dev = str(torch.device(self.device or 'cuda'))
        radii = (float(self.inter_radius), float(self.intra_radius))
        planned = (self._pocket_plan or {}).get(tuple(items), ())
        build = []
        for name in rec_atoms:
            have = self._pockets.get((name, dev))
            if have is not None and have[0] == radii:
                continue
            if name not in planned:
                return False, []
            build.append(name)
        return True, build

    def _batch_receptors(self, items):
        """Receptor names of a batch in first-use order, and rec_of_pose."""
        rec_names, rec_index = [], {}
        rec_of_pose = np.zeros(len(items), dtype=np.int32)
        for b, i in enumerate(items):
            name = str(self.receptor_fnames[i])
            if name not in rec_index:
                rec_index[name] = len(rec_names)
                rec_names.append(name)
            rec_of_pose[b] = rec_index[name]
        return rec_names, rec_of_pose

    def crop_on_device(self, items, ligands=None):
        """K0 for the complexes `items`: -> (coords f64 [N,3], bp i32 [N],
        feats f32 [N,F]) on the device and the host complex_ptr [B+1]."""
        device = torch.device(self.device or 'cuda')
        if ligands is None:
            ligands = [self.load_ligand(i) for i in items]
        # receptors of this batch, each uploaded once and kept
        rec_names, rec_of_pose = self._batch_receptors(items)
        recs = [self.receptor_on_device(name, device) for name in rec_names]
        return crop_batch(ligands, recs, rec_of_pose, self.radius,
                          self.n_features, self.compact, device)

    def _device_graph(self, items, ligands, edge_capacity):
        """K0, then K1p or K1 as pocket_route picks, for batch `items` ->
        (CropOutput, CSRGraph)."""
        from .graph import radius_graph_batch   # noqa: PLC0415
        from .screening import Pocket   # noqa: PLC0415
        device = torch.device(self.device or 'cuda')
        if ligands is None:
            ligands = [self.load_ligand(i) for i in items]
        rec_names, rec_of_pose = self._batch_receptors(items)
        recs = [self.receptor_on_device(name, device) for name in rec_names]
        crop = crop_batch_masked(ligands, recs, rec_of_pose, self.radius,
                                 self.n_features, self.compact, device)
        cptr_host = crop.complex_ptr_host
        lig_count = [int(np.count_nonzero(l.emit)) for l in ligands]
        use, build = self.pocket_route(
            items, {n: int(r[0].shape[0]) for n, r in zip(rec_names, recs)},
            lig_count, np.diff(cptr_host))
        if not use:
            return crop, radius_graph_batch(
                crop.coords, crop.bp, cptr_host, self.inter_radius,
                self.intra_radius, device=device, edge_capacity=edge_capacity)
        radii = (float(self.inter_radius), float(self.intra_radius))
        parts = []
        for name, rec in zip(rec_names, recs):
            key = (name, str(device))
            if name in build:
                parts.append(Pocket(rec, *radii))
                with self._cache_lock:   # resident with its receptor only
                    if key in self._rec_dev:
                        self._pockets[key] = (radii, parts[-1])
            else:
                parts.append(self._pockets[key][1])
        # composed on the caller's stream, which K1p runs on
        pocket = Pocket.compose(parts)
        return crop, pocket.radius_graph(crop, lig_count,
                                         edge_capacity=edge_capacity)

    def prepare(self, item):
        """What a loader thread does ahead of the device for one complex."""
        return self.load_ligand(item) if self.device_crop else self.load(item)

    def pack(self, items, complexes=None, edge_capacity=None):
        """Complexes `items` -> one PackedBatch with the batch's radius graph
        built on the device."""
        if self.device_crop:
            return self._pack_device(items, complexes, edge_capacity)
        if complexes is None:
            complexes = [self.load(i) for i in items]
        sizes = [len(c) for c in complexes]
        cptr = np.zeros(len(complexes) + 1, dtype=np.int32)
        np.cumsum(sizes, out=cptr[1:])
        if complexes:
            coords = np.concatenate([c.coords for c in complexes])
            bp = np.concatenate([c.bp for c in complexes])
            feats = np.concatenate([c.feats for c in complexes])
        else:
            coords = np.zeros((0, 3))
            bp = np.zeros(0, dtype=np.int32)
            feats = np.zeros((0, self.feature_dim), dtype=np.float32)
        y = self._labels(items)   # PyG concatenates per-complex label vectors
        batch = PackedBatch.from_arrays(
            coords, bp, feats, cptr, inter_radius=self.inter_radius,
            intra_radius=self.intra_radius, y=y, device=self.device,
            lig_fname=[Path(self.ligand_fnames[i]) for i in items],
            rec_fname=[Path(self.receptor_fnames[i]) for i in items],
            edge_capacity=edge_capacity)
        if self.rot:
            # the reference rotates `pos` only; edges come from the unrotated
            # structure (data_loaders.py:303-305 vs :365)
            pos = coords.copy()
            for b in range(len(complexes)):
                s, e = cptr[b], cptr[b + 1]
                if e > s:
                    pos[s:e] = uniform_random_rotation(pos[s:e], self._rng)
            batch.pos = torch.as_tensor(pos, dtype=torch.float32).to(
                batch.x.device)
        return batch

    def _labels(self, items):
        labels = [self.label(i) for i in items]
        if not labels or labels[0] is None or (
                isinstance(labels[0], tuple) and labels[0][0] is None):
            return None
        if self.model_task == 'classification':
            return torch.tensor([int(v) for v in labels], dtype=torch.long)
        return torch.tensor(np.array(labels, dtype=np.float64).reshape(-1),
                            dtype=torch.float32)

    def _pack_device(self, items, ligands, edge_capacity):
        crop, csr = self._device_graph(items, ligands, edge_capacity)
        coords, feats, cptr_host = crop.coords, crop.feats, \
            crop.complex_ptr_host
        pos = coords.float()
        if self.rot:
            pos_h = coords.cpu().numpy().copy()
            for b in range(len(items)):
                s_, e_ = cptr_host[b], cptr_host[b + 1]
                if e_ > s_:
                    pos_h[s_:e_] = uniform_random_rotation(pos_h[s_:e_],
                                                           self._rng)
            pos = torch.as_tensor(pos_h, dtype=torch.float32).to(coords.device)
        return PackedBatch(
            feats, pos, csr, csr.complex_ptr, y=self._labels(items),
            lig_fname=[Path(self.ligand_fnames[i]) for i in items],
            rec_fname=[Path(self.receptor_fnames[i]) for i in items])

    def __getitem__(self, item):
        return self.pack([item])


_WORKER_DS = None


def _worker_init(dataset):
    global _WORKER_DS
    _WORKER_DS = dataset


def _worker_prepare(items):
    """Runs in a loader process: host-side preparation of one mini-batch."""
    return [_WORKER_DS.prepare(i) for i in items]


class PackedLoader:
    """Iterates a ComplexDataset in mini-batches of PackedBatch (the role of
    `GeoDataLoader(ds, batch_size, False, sampler=..., drop_last=False)`,
    data_loaders.py:514-519).  Parquet reading (and the host crop, if that is
    what the dataset uses) runs `prefetch` batches ahead of the device on
    `num_workers` host threads, or -- `processes=True`, the counterpart of the
    reference's DataLoader workers -- in that many spawned processes, which
    do not share the interpreter lock."""

    def __init__(self, dataset, batch_size=32, sampler=None, num_workers=4,
                 prefetch=2, edge_capacity=None, processes=False):
        self.dataset, self.batch_size, self.sampler = dataset, batch_size, sampler
        self.num_workers, self.prefetch = num_workers, max(1, prefetch)
        self.edge_capacity = edge_capacity
        self.processes = bool(processes) and num_workers > 0
        self._pool = None

    def _process_pool(self):
        if self._pool is None:
            import multiprocessing as mp   # noqa: PLC0415
            from concurrent.futures import ProcessPoolExecutor   # noqa: PLC0415
            self._pool = ProcessPoolExecutor(
                self.num_workers, mp_context=mp.get_context('spawn'),
                initializer=_worker_init, initargs=(self.dataset,))
        return self._pool

    def close(self):
        if self._pool is not None:
            self._pool.shutdown(wait=False, cancel_futures=True)
            self._pool = None

    def __del__(self):
        try:
            self.close()
        except Exception:   # noqa: BLE001 - interpreter shutdown
            pass

    def prepared(self):
        """(items, host-side prepared complexes) per mini-batch, in order --
        everything that happens before the device is involved."""
        batches = self._batches()
        ds = self.dataset
        if ds.device_crop:
            ds.plan_pockets(batches if self.sampler is None else None)
        if self.num_workers <= 0:
            for items in batches:
                yield items, [ds.prepare(i) for i in items]
            return
        if self.processes:
            pool = self._process_pool()
            depth = max(self.prefetch, self.num_workers)
            pending, nxt = deque(), 0
            while nxt < len(batches) or pending:
                while nxt < len(batches) and len(pending) < depth:
                    pending.append((batches[nxt],
                                    pool.submit(_worker_prepare, batches[nxt])))
                    nxt += 1
                items, fut = pending.popleft()
                yield items, fut.result()
            return
        with ThreadPoolExecutor(self.num_workers) as pool:
            pending, nxt = deque(), 0
            while nxt < len(batches) or pending:
                while nxt < len(batches) and len(pending) < self.prefetch:
                    items = batches[nxt]
                    pending.append(
                        (items, [pool.submit(ds.prepare, i) for i in items]))
                    nxt += 1
                items, futures = pending.popleft()
                yield items, [f.result() for f in futures]

    def __len__(self):
        return math.ceil(len(self.dataset) / self.batch_size)

    def _batches(self):
        order = list(self.sampler) if self.sampler is not None \
            else list(range(len(self.dataset)))
        return [order[i:i + self.batch_size]
                for i in range(0, len(order), self.batch_size)]

    def __iter__(self):
        for items, prepared in self.prepared():
            yield self.dataset.pack(items, prepared,
                                    edge_capacity=self.edge_capacity)


def get_data_loader(data_root, dataset_class=None, receptors=None,
                    batch_size=32, compact=True, use_atomic_numbers=False,
                    radius=6, rot=True, augmented_actives=0, min_aug_angle=30,
                    polar_hydrogens=True, mode='train',
                    model_task='classification', max_active_rms_distance=None,
                    fname_suffix='parquet', min_inactive_rms_distance=None,
                    types_fname=None, edge_radius=None, prune=False,
                    estimate_bonds=False, bp=None, p_noise=-1, num_workers=4,
                    device=None, device_crop=False, worker_processes=False,
                    edge_capacity=None, **kwargs):
    """Signature of the reference's `get_data_loader` (data_loaders.py:483-520).
    `dataset_class` is accepted for call compatibility and ignored: there is
    one dataset here.  As in the reference, classification training draws
    complexes with the class-balancing weighted sampler and every other mode
    walks the types file in order.  edge_capacity='auto' (or an int) builds
    capacity-bounded edge lists: no host read-back of the edge count per
    batch, so training steps queue without a sync; `train_model` checks the
    overflow flags with the losses, once per log interval."""
    del dataset_class, receptors
    ds = ComplexDataset(
        data_root, compact=compact, augmented_active_count=augmented_actives,
        augmented_active_min_angle=min_aug_angle,
        polar_hydrogens=polar_hydrogens,
        max_active_rms_distance=max_active_rms_distance,
        min_inactive_rms_distance=min_inactive_rms_distance,
        use_atomic_numbers=use_atomic_numbers, fname_suffix=fname_suffix,
        types_fname=types_fname, edge_radius=edge_radius,
        estimate_bonds=estimate_bonds, prune=prune, bp=bp, radius=radius,
        rot=rot, model_task=model_task, p_noise=p_noise, device=device,
        device_crop=device_crop, **kwargs)
    sampler = ds.sampler if (ds.model_task == 'classification'
                             and mode == 'train') else None
    return PackedLoader(ds, batch_size, sampler=sampler,
                        num_workers=num_workers, processes=worker_processes,
                        edge_capacity=edge_capacity)


__all__ = ['ComplexDataset', 'PackedLoader', 'get_data_loader',
           'parse_classification_types', 'parse_regression_types',
           'read_structure', 'build_complex', 'make_box', 'make_bit_vector',
           'atomic_number_table', 'atom_codes', 'crop_batch',
           'crop_batch_masked', 'CropOutput', 'Complex', 'Ligand']
