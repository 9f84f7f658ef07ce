"""The device-crop loader's pocket route: K1 against K1p, K0, pocket builds,
and end to end through `inference`.

* graph stage, per 128-pose batch: K0's output of `--graph-steps` batches is
  kept; K1 (`radius_graph_batch`) and K1p (`Pocket.radius_graph`) then run
  over all of them between two CUDA events, alternating, `--rounds` times
  each (best round reported).  Pockets: the synthetic 800- and 3000-atom ones
  of `synthetic_pocket_poses` (30-atom ligands) and the whole proteins 1h1p,
  4fnn and 5k6a shipped in tests/golden/trained/data_affinity, posed with
  their own ligand moved by a random rotation about its centre and a 1 A
  normal shift; crop none and 10 A, edge radii 4 / 4.
* K0 per batch: the same crops between two CUDA events; each call includes
  K0's one host read of complex_ptr.
* pocket build per receptor: `Pocket(receptor)` between two CUDA events
  (launches, the host read of the edge count, the final synchronise).
* end to end: `inference.get_model_and_test_dl` on the shipped pose
  checkpoint (device crop, 128 poses a batch, 4 reader threads) and
  `model.val`, with the route on and forced off (`pocket_route` patched to
  K1), alternating, for two generated types files: many poses per receptor
  sorted by receptor, and one pose per receptor.  The ligand-reading rate of
  the loader alone is reported beside it.

Prints one JSON document (and writes it to --out).
"""
import argparse
import json
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import pointvs_b200 as pv  # noqa: E402
from pointvs_b200 import data  # noqa: E402
from pointvs_b200.graph import radius_graph_batch  # noqa: E402
from pointvs_b200.synthetic import synthetic_pocket_poses  # noqa: E402

GOLD = ROOT / 'tests' / 'golden' / 'trained'
AFF = GOLD / 'data_affinity'
PROTEINS = ('1h1p', '4fnn', '5k6a')


def gpu_info():
    info = {'gpu': torch.cuda.get_device_name(0), 'power_limit_w': None}
    try:
        out = subprocess.run(
            ['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader,nounits',
             '-i', '0'], capture_output=True, text=True, timeout=30)
        info['power_limit_w'] = float(out.stdout.strip().splitlines()[0])
    except Exception:   # noqa: BLE001 - reported as unknown
        pass
    return info


def rotation(rng):
    q = rng.normal(size=4)
    a, b, c, d = q / np.linalg.norm(q)
    return np.array([[a*a+b*b-c*c-d*d, 2*(b*c-a*d), 2*(b*d+a*c)],
                     [2*(b*c+a*d), a*a-b*b+c*c-d*d, 2*(c*d-a*b)],
                     [2*(b*d-a*c), 2*(c*d+a*b), a*a-b*b-c*c+d*d]])


def posed(xyz, rng):
    """The ligand turned about its centre and shifted by N(0, 1 A)."""
    mid = xyz.mean(0)
    return (xyz - mid) @ rotation(rng).T + mid + rng.normal(size=3)


def synthetic_case(n_pocket, pool, dev):
    n_lig, n_types = 30, 12
    coords, _, feats, _ = synthetic_pocket_poses(0, pool, n_pocket, n_lig)
    types = feats[:, :n_types].argmax(1)
    per = n_lig + n_pocket
    rec = (torch.from_numpy(coords[n_lig:per].copy()).to(dev),
           torch.ones(n_pocket, dtype=torch.uint8, device=dev),
           torch.from_numpy((types[n_lig:per] + n_types).astype(np.int16)).to(dev))
    ligs = [data.Ligand(coords[p * per:p * per + n_lig].copy(),
                        np.ones(n_lig, dtype=np.uint8),
                        types[p * per:p * per + n_lig].astype(np.int16))
            for p in range(pool)]
    torch.cuda.synchronize()
    return f'synthetic {n_pocket}', rec, ligs, n_types, True


def affinity_dataset():
    return data.ComplexDataset(AFF, types_fname=GOLD / 'affinity.types', radius=10,
                               polar_hydrogens=False, compact=False, device='cuda',
                               device_crop=True, model_task='regression')


def protein_case(ds, name, pool, dev, rng):
    i = [k for k, r in enumerate(ds.receptor_fnames) if r.startswith(name)][0]
    rec = ds.receptor_on_device(ds.receptor_fnames[i], dev)
    lig = ds.load_ligand(i)
    ligs = [data.Ligand(posed(lig.coords, rng), lig.emit, lig.code) for _ in range(pool)]
    return name, rec, ligs, ds.n_features, ds.compact


def events():
    return [torch.cuda.Event(enable_timing=True) for _ in range(2)]


def graph_case(label, rec, ligs, n_features, compact, radius, args, dev):
    pocket = pv.Pocket(rec, 4.0, 4.0)
    zeros = np.zeros(args.batch, dtype=np.int32)
    pool = len(ligs)

    def batch_ligs(i):
        return [ligs[(i * args.batch + j) % pool] for j in range(args.batch)]
    lig_counts = [[int(np.count_nonzero(l.emit)) for l in batch_ligs(i)]
                  for i in range(args.graph_steps)]

    def crop(i):
        return pocket.crop(batch_ligs(i), zeros, radius, n_features, compact)

    for i in range(3):
        crop(i)
    torch.cuda.synchronize()
    ev = events()
    k0_ms = []
    for _ in range(args.rounds):
        ev[0].record()
        crops = [crop(i) for i in range(args.graph_steps)]
        ev[1].record()
        torch.cuda.synchronize()
        k0_ms.append(ev[0].elapsed_time(ev[1]) / args.graph_steps)

    def k1(i):
        c = crops[i]
        return radius_graph_batch(c.coords, c.bp, c.complex_ptr_host, 4.0, 4.0,
                                  device=dev, edge_capacity='auto')

    def k1p(i):
        return pocket.radius_graph(crops[i], lig_counts[i], edge_capacity='auto')

    for fn in (k1, k1p):
        for i in range(3):
            fn(i)
    torch.cuda.synchronize()
    graph_ms = {'k1': [], 'k1p': []}
    edges = {}
    for _ in range(args.rounds):
        for name, fn in (('k1', k1), ('k1p', k1p)):
            tot = torch.zeros(1, dtype=torch.int64, device=dev)
            ev[0].record()
            for i in range(len(crops)):
                tot += fn(i).n_edges_dev
            ev[1].record()
            torch.cuda.synchronize()
            graph_ms[name].append(ev[0].elapsed_time(ev[1]) / len(crops))
            edges[name] = int(tot.item())
    # K1 misses the rare pair of a complex between 15 and 16 of its cell
    # edges across (DESIGN.md section 8): reported, not asserted
    a, b = k1(0), k1p(0)
    same = all(torch.equal(getattr(a, f)[:int(a.row_ptr[-1])],
                           getattr(b, f)[:int(b.row_ptr[-1])]) for f in ('col', 'attr')) \
        and torch.equal(a.row_ptr, b.row_ptr)
    n_graph = args.graph_steps * args.batch
    atoms = sum(int(c.complex_ptr_host[-1]) for c in crops)
    kept = atoms - sum(sum(x) for x in lig_counts)
    best = {k: min(v) for k, v in graph_ms.items()}
    return {
        'pocket': label, 'receptor_atoms': int(rec[0].shape[0]),
        'receptor_emitted_atoms': int(rec[1].sum().item()),
        'crop_radius': None if not np.isfinite(radius) else radius,
        'atoms_per_complex': round(atoms / n_graph, 1),
        'kept_receptor_atoms_per_pose': round(kept / n_graph, 1),
        'edges_per_pose': round(edges['k1p'] / n_graph, 1),
        'edges_k1_minus_k1p': edges['k1'] - edges['k1p'],
        'k0_ms_per_batch': round(min(k0_ms), 4),
        'graph_ms_per_batch': {k: round(v, 4) for k, v in best.items()},
        'graph_ms_per_batch_rounds': {k: [round(x, 4) for x in v]
                                      for k, v in graph_ms.items()},
        'graph_speedup': round(best['k1'] / best['k1p'], 3),
        'k1p_saving_us_per_pose': round((best['k1'] - best['k1p']) * 1e3 / args.batch, 4),
        'csr_bytes_equal_first_batch': bool(same),
    }


def build_time(rec, reps, dev):
    pv.Pocket(rec, 4.0, 4.0)
    torch.cuda.synchronize()
    ev = events()
    ms = []
    for _ in range(reps):
        ev[0].record()
        pv.Pocket(rec, 4.0, 4.0)
        ev[1].record()
        torch.cuda.synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    return {'receptor_atoms': int(rec[0].shape[0]),
            'build_ms_median': round(float(np.median(ms)), 4),
            'build_ms_min': round(float(min(ms)), 4)}


def write_ligand(path, cols, xyz):
    import pyarrow as pa
    import pyarrow.parquet as pq
    t = {'x': xyz[:, 0], 'y': xyz[:, 1], 'z': xyz[:, 2]}
    for k in ('atomic_number', 'types', 'bp'):
        t[k] = cols[k]
    path.parent.mkdir(parents=True, exist_ok=True)
    pq.write_table(pa.table(t), str(path))


def make_types(root, poses_per_rec, copies, rng, names=None):
    """Receptors of data_affinity (each under `copies` names), each with
    `poses_per_rec` posed copies of its ligand; lines sorted by receptor."""
    lines = []
    for src in sorted(AFF.iterdir()):
        if names and src.name not in names:
            continue
        prot = next(src.glob('*protein*.parquet'))
        ligf = next(f for f in src.glob('*.parquet') if 'protein' not in f.name)
        cols = data.read_structure(ligf)
        xyz = np.stack([cols['x'], cols['y'], cols['z']], 1)
        for c in range(copies):
            rname = f'rec/{src.name}_{c}.parquet'
            (root / 'rec').mkdir(parents=True, exist_ok=True)
            shutil.copy(prot, root / rname)
            for p in range(poses_per_rec):
                lname = f'lig/{src.name}_{c}/{p}.parquet'
                write_ligand(root / lname, cols, posed(xyz, rng))
                lines.append(f'1 -1 -1.0 {rname} {lname}')
    (root / 'screen.types').write_text('\n'.join(lines) + '\n')
    return root / 'screen.types'


def e2e_case(label, types, root, args, crop=None):
    from pointvs_b200 import inference
    from pointvs_b200.screening import Pocket
    run = Path(tempfile.mkdtemp(prefix='pvs_run_')) / 'run'
    shutil.copytree(GOLD / 'run', run)
    ck = run / 'checkpoints' / 'pose_ckpt_epoch_1.pt'
    k1p_batches = [0]
    orig_graph = Pocket.radius_graph

    def counted(self, *a, **k):
        k1p_batches[0] += 1
        return orig_graph(self, *a, **k)
    Pocket.radius_graph = counted
    orig_route = data.ComplexDataset.pocket_route
    off = lambda self, *a: (False, [])   # noqa: E731
    if crop is not None:   # a model trained with another crop radius
        cfg = run / 'cmd_args.yaml'
        cfg.write_text(cfg.read_text().replace('radius: 10', f'radius: {crop}'))
    res = {'types': label, 'crop_radius': crop or 10,
           'poses': sum(1 for _ in open(types))}
    rates = {'on': [], 'off': []}
    outs = {}
    try:
        _, model, _, _, dl = inference.get_model_and_test_dl(
            ck, str(types), str(root), 'pose', batch_size=args.batch, device_crop=True,
            loader_kwargs=dict(num_workers=4))
        model.set_math(args.math)
        # the loader alone: ligand parquets read by 4 threads
        t0 = time.perf_counter()
        n_read = sum(len(items) for items, _ in dl.prepared())
        res['ligand_read_poses_per_s'] = round(n_read / (time.perf_counter() - t0), 1)
        for rnd in range(args.rounds + 1):
            for mode in ('off', 'on'):
                # a fresh dataset state per run: no pocket carried over
                dl.dataset._pockets.clear()
                dl.dataset._rec_dev.clear()
                data.ComplexDataset.pocket_route = orig_route if mode == 'on' else off
                k1p_batches[0] = 0
                out = root / f'pred_{mode}.txt'
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                model.val(dl, out)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                if rnd:   # round 0 warms every shape
                    rates[mode].append(res['poses'] / dt)
                res[f'k1p_batches_{mode}'] = k1p_batches[0]
                outs[mode] = (out.parent / ('pose_' + out.name)).read_bytes()
    finally:
        Pocket.radius_graph = orig_graph
        data.ComplexDataset.pocket_route = orig_route
    res['batches'] = len(dl)
    res['poses_per_s'] = {k: round(max(v), 1) for k, v in rates.items()}
    res['poses_per_s_rounds'] = {k: [round(x, 1) for x in v] for k, v in rates.items()}
    res['predictions_identical'] = outs['on'] == outs['off']
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=128)
    ap.add_argument('--graph-steps', type=int, default=40)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--pool', type=int, default=1024)
    ap.add_argument('--many-poses', type=int, default=1100)
    ap.add_argument('--math', default='bf16x3')
    ap.add_argument('--skip-e2e', action='store_true')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    dev = torch.device('cuda')
    rng = np.random.default_rng(0)
    result = dict(gpu_info(), batch=args.batch, edge_radii=[4.0, 4.0],
                  graph_steps=args.graph_steps, rounds=args.rounds, graph=[], build=[],
                  e2e=[])
    ds = affinity_dataset()
    cases = [synthetic_case(800, args.pool, dev), synthetic_case(3000, args.pool, dev)]
    cases += [protein_case(ds, p, args.pool, dev, rng) for p in PROTEINS]
    for label, rec, ligs, nf, compact in cases:
        for radius in (np.inf, 10.0):
            case = graph_case(label, rec, ligs, nf, compact, radius, args, dev)
            print(json.dumps(case), file=sys.stderr)
            result['graph'].append(case)
    for name in sorted(p.name for p in AFF.iterdir()):
        i = [k for k, r in enumerate(ds.receptor_fnames) if r.startswith(name)][0]
        rec = ds.receptor_on_device(ds.receptor_fnames[i], dev)
        b = dict(receptor=name, **build_time(rec, 10, dev))
        print(json.dumps(b), file=sys.stderr)
        result['build'].append(b)
    if not args.skip_e2e:
        tmp = Path(tempfile.mkdtemp(prefix='pvs_route_'))
        try:
            many = make_types(tmp / 'many', args.many_poses, 1, rng, PROTEINS)
            single = make_types(tmp / 'single', 1, 16, rng)
            for label, types, crop in (
                    ('many poses per receptor, sorted', many, None),
                    ('many poses per receptor, sorted', many, 16),
                    ('one pose per receptor', single, None)):
                r = e2e_case(label, types, types.parent, args, crop)
                print(json.dumps(r), file=sys.stderr)
                result['e2e'].append(r)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    text = json.dumps(result, indent=1)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + '\n')
    print(text)


if __name__ == '__main__':
    main()
