"""Score ligand poses against a resident pocket.

The heaviest workload of a virtual screen is many ligand poses scored against
one receptor pocket.  `Pocket` keeps the receptors on the device together with
the part of every pose's radius graph that does not depend on the pose: the
receptor-receptor edges, searched once (K1p build, csrc/pocket.cu).
`score_poses` then runs, per batch of poses:

  K0  (crop_batch_masked) : receptor crop + typing, complexes assembled on
                            the device, keep bits per pose;
  K1p (Pocket.radius_graph): ligand-ligand and ligand-receptor pairs searched,
                            the cached receptor-receptor rows copied through
                            the pose's keep bits;
  the model's fused scoring pass.

The graph is K1's (`radius_graph_batch`) byte for byte on the same complexes,
so the scores are those of the crop_batch -> radius_graph_batch -> model
chain bit for bit.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _cabi
from ._cabi import check, lib, ptr, stream
from .data import crop_batch_masked
from .graph import CSRGraph, PackedBatch, auto_edge_capacity
from .parallel import gather_scores, shard_range


def _as_receptor_list(receptors):
    if isinstance(receptors, tuple) and len(receptors) == 3 and \
            torch.is_tensor(receptors[0]):
        return [receptors]
    return list(receptors)


class Pocket:
    """Resident receptors plus their cached receptor-receptor graph.

    receptors: one (xyz f64 [n,3], emit u8 [n], code i16 [n]) triple of
    device tensors, or a list of them -- what
    `ComplexDataset.receptor_on_device` returns, so parquet input goes
    through the existing readers.  The pocket is built for one
    (inter_radius, intra_radius) pair; graphs with other radii are refused.
    Building costs a few launches and one host read (the receptor-receptor
    edge count); the pocket keeps about 128 KB per receptor plus 40 B per
    atom and its receptor-receptor edges."""

    def __init__(self, receptors, inter_radius=4.0, intra_radius=4.0):
        inter_radius, intra_radius = float(inter_radius), float(intra_radius)
        if not (inter_radius >= 0 and intra_radius >= 0):
            raise ValueError('radii must be non-negative')
        receptors = _as_receptor_list(receptors)
        if not receptors:
            raise ValueError('a pocket needs at least one receptor')
        for rec in receptors:
            _cabi.require_cuda(*rec)
        self.inter_radius, self.intra_radius = inter_radius, intra_radius
        self.device = receptors[0][0].device
        self.receptors = receptors
        sizes = [int(r[0].shape[0]) for r in receptors]
        self.rec_ptr_host = np.zeros(len(sizes) + 1, dtype=np.int32)
        np.cumsum(sizes, out=self.rec_ptr_host[1:])
        n_atoms = int(self.rec_ptr_host[-1])
        h = lib()
        dev = self.device
        with torch.cuda.device(dev):
            if len(receptors) == 1:
                self.xyz, self.emit, self.code = receptors[0]
            else:
                self.xyz = torch.cat([r[0] for r in receptors])
                self.emit = torch.cat([r[1] for r in receptors])
                self.code = torch.cat([r[2] for r in receptors])
            self.xyz = self.xyz.to(torch.float64).contiguous()
            self.emit = self.emit.to(torch.uint8).contiguous()
            self.rec_ptr = torch.from_numpy(self.rec_ptr_host.copy()).to(dev)
            self.cells = torch.empty(
                max(256, int(h.pvs_pocket_cells_bytes(len(sizes), n_atoms))),
                dtype=torch.uint8, device=dev)
            self.rr_ptr = torch.empty(n_atoms + 1, dtype=torch.int32,
                                      device=dev)
            scratch = torch.empty(
                int(h.pvs_pocket_build_scratch_bytes(len(sizes), n_atoms)),
                dtype=torch.uint8, device=dev)
            self.desc = _cabi.PocketDesc(
                len(sizes), n_atoms, max(sizes), inter_radius, intra_radius,
                ptr(self.xyz), ptr(self.emit), ptr(self.rec_ptr),
                ptr(self.cells), ptr(self.rr_ptr), None)
            check(h.pvs_pocket_build_count(C.byref(self.desc), ptr(scratch),
                                           stream()), 'pvs_pocket_build_count')
            self.n_rr_edges = int(self.rr_ptr[-1].item())
            self.rr_col = torch.empty(max(1, self.n_rr_edges),
                                      dtype=torch.int32, device=dev)
            self.desc.rr_col = ptr(self.rr_col).value
            check(h.pvs_pocket_build_fill(C.byref(self.desc), stream()),
                  'pvs_pocket_build_fill')
            # complete before K0's side stream reads the receptors
            torch.cuda.current_stream(dev).synchronize()

    @classmethod
    def compose(cls, pockets):
        """One pocket of the receptors of `pockets` (built pockets of the
        same radii and device), in that order, assembled by device copies:
        no receptor is searched again.  Runs on the current stream, which
        must be ordered before any other stream reads the result."""
        pockets = list(pockets)
        if len(pockets) == 1:
            return pockets[0]
        if not pockets:
            raise ValueError('a pocket needs at least one receptor')
        first = pockets[0]
        for p in pockets[1:]:
            first.check_radii(p.inter_radius, p.intra_radius)
        self = cls.__new__(cls)
        self.inter_radius, self.intra_radius = first.inter_radius, \
            first.intra_radius
        self.device = dev = first.device
        self.receptors = [r for p in pockets for r in p.receptors]
        sizes = [int(r[0].shape[0]) for r in self.receptors]
        self.rec_ptr_host = np.zeros(len(sizes) + 1, dtype=np.int32)
        np.cumsum(sizes, out=self.rec_ptr_host[1:])
        n_atoms = int(self.rec_ptr_host[-1])
        self.n_rr_edges = sum(p.n_rr_edges for p in pockets)
        h = lib()
        with torch.cuda.device(dev):
            self.xyz = torch.cat([p.xyz for p in pockets])
            self.emit = torch.cat([p.emit for p in pockets])
            self.code = torch.cat([p.code.to(torch.int16) for p in pockets])
            self.rec_ptr = torch.from_numpy(self.rec_ptr_host.copy()).to(dev)
            self.cells = torch.empty(
                max(256, int(h.pvs_pocket_cells_bytes(len(sizes), n_atoms))),
                dtype=torch.uint8, device=dev)
            self.rr_ptr = torch.empty(n_atoms + 1, dtype=torch.int32,
                                      device=dev)
            self.rr_col = torch.empty(max(1, self.n_rr_edges),
                                      dtype=torch.int32, device=dev)
            self.desc = _cabi.PocketDesc(
                len(sizes), n_atoms, max(sizes), self.inter_radius,
                self.intra_radius, ptr(self.xyz), ptr(self.emit),
                ptr(self.rec_ptr), ptr(self.cells), ptr(self.rr_ptr),
                ptr(self.rr_col))
            parts = (C.POINTER(_cabi.PocketDesc) * len(pockets))(
                *[C.pointer(p.desc) for p in pockets])
            check(h.pvs_pocket_compose(parts, len(pockets),
                                       C.byref(self.desc), stream()),
                  'pvs_pocket_compose')
        return self

    @classmethod
    def from_dataset(cls, dataset, rec_fnames, device=None):
        """Pocket of `dataset`'s receptors `rec_fnames` (one name or a list)
        at the dataset's edge radii."""
        if isinstance(rec_fnames, (str, bytes)) or not hasattr(
                rec_fnames, '__iter__'):
            rec_fnames = [rec_fnames]
        device = torch.device(device or dataset.device or 'cuda')
        recs = [dataset.receptor_on_device(str(r), device) for r in rec_fnames]
        return cls(recs, dataset.inter_radius, dataset.intra_radius)

    @property
    def n_receptors(self):
        return len(self.receptors)

    def check_radii(self, inter_radius, intra_radius):
        """Raise unless (inter_radius, intra_radius) are the pocket's own."""
        if (float(inter_radius), float(intra_radius)) != (
                self.inter_radius, self.intra_radius):
            raise ValueError(
                f'pocket built for radii ({self.inter_radius}, '
                f'{self.intra_radius}), used with ({inter_radius}, '
                f'{intra_radius}): build a Pocket for these radii')

    def crop(self, ligands, rec_of_pose, radius, n_features, compact=True):
        """K0 against this pocket's receptors -> data.CropOutput."""
        return crop_batch_masked(ligands, self.receptors, rec_of_pose, radius,
                                 n_features, compact, self.device,
                                 concatenated=(self.xyz, self.emit, self.code))

    def radius_graph(self, crop, lig_count, inter_radius=None,
                     intra_radius=None, edge_capacity='auto'):
        """K1p: the radius graph of K0's complexes `crop` (data.CropOutput
        against this pocket).  lig_count: emitted ligand atoms per pose (host
        ints).  Same result and edge_capacity semantics as
        `radius_graph_batch` on crop.coords / crop.bp."""
        inter_radius = self.inter_radius if inter_radius is None \
            else inter_radius
        intra_radius = self.intra_radius if intra_radius is None \
            else intra_radius
        self.check_radii(inter_radius, intra_radius)
        h = lib()
        dev = self.device
        cptr_host = crop.complex_ptr_host
        n = int(cptr_host[-1])
        n_poses = len(cptr_host) - 1
        lig_count = np.ascontiguousarray(lig_count, dtype=np.int32)
        if len(lig_count) != n_poses:
            raise ValueError('lig_count needs one entry per pose')
        max_lig = int(lig_count.max()) if n_poses else 0
        with torch.cuda.device(dev):
            lc = torch.from_numpy(lig_count).pin_memory().to(
                dev, non_blocking=True) if n_poses else None
            deg = torch.empty(max(1, n), dtype=torch.int32, device=dev)
            n_inter = torch.empty(max(1, n), dtype=torch.int32, device=dev)
            row_ptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
            scratch = _cabi.scratch(
                'k1p_scan', int(h.pvs_scan_scratch_bytes(n)) + 256, dev)
            args = (C.byref(self.desc), ptr(crop.coords),
                    ptr(crop.complex_ptr), n_poses, n, ptr(crop.mask),
                    crop.mask_words, ptr(lc), max_lig, ptr(crop.rec_of_pose),
                    C.c_double(inter_radius), C.c_double(intra_radius))
            check(h.pvs_pocket_graph_count(*args, ptr(deg), ptr(n_inter),
                                           ptr(row_ptr), ptr(scratch),
                                           stream()), 'pvs_pocket_graph_count')
            if edge_capacity is None:
                n_edges = int(row_ptr[-1].item())   # the one host sync
                capacity = n_edges
            else:
                capacity = auto_edge_capacity(n, inter_radius, intra_radius) \
                    if edge_capacity == 'auto' else int(edge_capacity)
                n_edges = capacity
            col = torch.empty(max(1, capacity), dtype=torch.int32, device=dev)
            attr = torch.empty(max(1, capacity), dtype=torch.uint8,
                               device=dev)
            overflow = torch.zeros(1, dtype=torch.int32, device=dev)
            check(h.pvs_pocket_graph_fill(*args, ptr(row_ptr), capacity,
                                          ptr(col), ptr(attr), ptr(overflow),
                                          stream()), 'pvs_pocket_graph_fill')
            if lc is not None:
                lc.record_stream(torch.cuda.current_stream(dev))
            g = CSRGraph(n, n_edges, row_ptr, col[:n_edges], attr[:n_edges],
                         n_inter=n_inter[:n])
        g.complex_ptr = crop.complex_ptr
        g.complex_ptr_host = cptr_host
        g.n_edges_dev = row_ptr[-1:]
        g.exact_edge_count = edge_capacity is None
        g.symmetric = True
        g._overflow = overflow
        return g

    def batch(self, ligands, rec_of_pose=None, radius=None, n_features=11,
              compact=True, edge_capacity='auto'):
        """K0 + K1p for one batch of poses -> PackedBatch ready for a model.
        radius: crop radius (None keeps every receptor atom)."""
        if rec_of_pose is None:
            rec_of_pose = np.zeros(len(ligands), dtype=np.int32)
        crop = self.crop(ligands, rec_of_pose,
                         math.inf if radius is None else float(radius),
                         n_features, compact)
        lig_count = [int(np.count_nonzero(l.emit)) for l in ligands]
        csr = self.radius_graph(crop, lig_count, edge_capacity=edge_capacity)
        return PackedBatch(crop.feats, crop.coords.float(), csr,
                           crop.complex_ptr)


def score_poses(model, pocket, ligands, rec_of_pose=None, radius=None,
                batch_size=128, n_features=11, compact=True,
                edge_capacity='auto', group=None, activation='sigmoid'):
    """Score `ligands` (a list of data.Ligand) against `pocket`.

    rec_of_pose[i] picks the pocket receptor of ligand i (None: receptor 0);
    radius is K0's crop radius (None: no crop); n_features / compact as the
    dataset's typing (11 sminatypes by default).  Ligands are sharded by rank
    of `group` in contiguous blocks and the scores gathered on every rank, as
    `parallel.screen` does; activation='sigmoid' applies the sigmoid to the
    raw scores (None: raw).  Returns the dense score array [len(ligands),
    out] in ligand order.

    Per batch the host reads K0's complex offsets and, with
    edge_capacity=None, the exact edge count; nothing else.  With a capacity
    ('auto' or an int), an overflow raises once at the end."""
    world = torch.distributed.get_world_size(group) \
        if torch.distributed.is_initialized() else 1
    rank = torch.distributed.get_rank(group) \
        if torch.distributed.is_initialized() else 0
    n_total = len(ligands)
    if rec_of_pose is None:
        rec_of_pose = np.zeros(n_total, dtype=np.int32)
    rec_of_pose = np.ascontiguousarray(rec_of_pose, dtype=np.int32)
    if len(rec_of_pose) != n_total:
        raise ValueError('rec_of_pose needs one entry per ligand')
    if n_total and (rec_of_pose.min() < 0 or
                    rec_of_pose.max() >= pocket.n_receptors):
        raise ValueError('rec_of_pose indexes a receptor the pocket lacks')
    lo, hi = shard_range(n_total, rank, world)
    model.eval()
    outs = []
    overflow = torch.zeros(1, dtype=torch.int32, device=pocket.device)
    for s in range(lo, hi, batch_size):
        e = min(hi, s + batch_size)
        batch = pocket.batch(ligands[s:e], rec_of_pose[s:e], radius,
                             n_features, compact, edge_capacity)
        with torch.no_grad():
            scores = model(batch)
        scores = scores.reshape(batch.num_graphs, -1)
        if activation == 'sigmoid':
            scores = torch.sigmoid(scores)
        outs.append(scores)
        if edge_capacity is not None:
            overflow += batch.pvs_csr._overflow
    local = torch.cat(outs).float().cpu().numpy() if outs else \
        np.zeros((0, 1), dtype=np.float32)
    if int(overflow.item()):
        raise RuntimeError(
            'edge capacity exceeded: pass a larger edge_capacity (or None to '
            'size the edge list exactly)')
    return gather_scores(np.arange(lo, hi), local, n_total, group)


__all__ = ['Pocket', 'score_poses']
