"""Pocket screening: the K0 + K1 chain against K0 + K1p, on the same batches.

For each pocket (the 800-atom configs[4] pocket of `synthetic_pocket_poses`
and a ~3000-atom one) and each crop (none, 10 A), 128 poses a batch of
30-atom ligands:

* graph stage: K0's output of `--graph-steps` batches is kept; the graph
  builder alone then runs over all of them between two CUDA events, K1
  (`radius_graph_batch`, count + fill) and K1p (`Pocket.radius_graph`)
  alternating, `--rounds` times each; the best round is reported per step;
* end to end: K0 -> graph -> 8 x 64 `egnn` (bf16x3) -> scores, poses/s over
  `--steps` batches, the two chains alternating, `--rounds` times each;
* parity: the scores of both chains on every timed batch, bit for bit.

Prints one JSON document (and writes it to --out).
"""
import argparse
import json
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402
import pointvs_b200 as pv  # noqa: E402
from pointvs_b200 import data  # noqa: E402
from pointvs_b200.graph import radius_graph_batch  # noqa: E402
from pointvs_b200.synthetic import synthetic_pocket_poses  # noqa: E402

N_LIG, N_TYPES = 30, 12


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


def make_pocket(n_pocket, pool, dev):
    coords, _, feats, _ = synthetic_pocket_poses(0, pool, n_pocket, N_LIG)
    types = feats[:, :N_TYPES].argmax(1)
    per = N_LIG + n_pocket
    rec = (torch.from_numpy(coords[N_LIG:per].copy()).to(dev),
           torch.ones(n_pocket, dtype=torch.uint8, device=dev),
           torch.from_numpy((types[N_LIG:per] + N_TYPES).astype(np.int16)).to(dev))
    ligs = [data.Ligand(coords[p * per:p * per + N_LIG].copy(),
                        np.ones(N_LIG, dtype=np.uint8),
                        types[p * per:p * per + N_LIG].astype(np.int16))
            for p in range(pool)]
    torch.cuda.synchronize()
    return rec, ligs


def run_case(model, rec, ligs, radius, args, dev):
    pocket = pv.Pocket(rec, 4.0, 4.0)
    zeros = np.zeros(args.batch, dtype=np.int32)
    lig_count = [N_LIG] * args.batch
    pool = len(ligs)

    def batch_ligs(i):
        return [ligs[(i * args.batch + j) % pool] for j in range(args.batch)]

    def k1(crop):
        return radius_graph_batch(crop.coords, crop.bp, crop.complex_ptr_host, 4.0, 4.0,
                                  device=dev, edge_capacity='auto')

    def k1p(crop):
        return pocket.radius_graph(crop, lig_count, edge_capacity='auto')

    # ---- graph stage ----
    crops = [pocket.crop(batch_ligs(i), zeros, radius, N_TYPES)
             for i in range(args.graph_steps)]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    graph_ms = {'k1': [], 'k1p': []}
    edges = {'k1': 0, 'k1p': 0}
    for name, fn in (('k1', k1), ('k1p', k1p)):   # warm-up
        for c in crops[:3]:
            fn(c)
    torch.cuda.synchronize()
    for _ in range(args.rounds):
        for name, fn in (('k1', k1), ('k1p', k1p)):
            tot = torch.zeros(1, dtype=torch.int64, device=dev)
            ev[0].record()
            for c in crops:
                g = fn(c)
                tot += g.n_edges_dev
            ev[1].record()
            torch.cuda.synchronize()
            graph_ms[name].append(ev[0].elapsed_time(ev[1]) / len(crops))
            edges[name] = int(tot.item())
    assert edges['k1'] == edges['k1p'], edges
    atoms = sum(int(c.complex_ptr_host[-1]) for c in crops)
    del crops

    # ---- end to end ----
    def step(i, use_pocket):
        crop = pocket.crop(batch_ligs(i), zeros, radius, N_TYPES)
        csr = k1p(crop) if use_pocket else k1(crop)
        batch = pv.PackedBatch(crop.feats, crop.coords.float(), csr, crop.complex_ptr)
        with torch.no_grad():
            return model(batch).reshape(args.batch, -1), csr

    for i in range(4):
        step(i, False)
        step(i, True)
    torch.cuda.synchronize()
    e2e = {'k1': [], 'k1p': []}
    scores = {}
    for _ in range(args.rounds):
        for name in ('k1', 'k1p'):
            outs = torch.empty((args.steps, args.batch, 1), dtype=torch.float32).pin_memory()
            overflow = torch.zeros(1, dtype=torch.int32, device=dev)
            ev[0].record()
            for i in range(args.steps):
                out, csr = step(i, name == 'k1p')
                outs[i].copy_(out, non_blocking=True)
                overflow += csr._overflow
            ev[1].record()
            torch.cuda.synchronize()
            assert int(overflow.item()) == 0
            e2e[name].append(args.steps * args.batch / (ev[0].elapsed_time(ev[1]) * 1e-3))
            scores[name] = outs.numpy().copy()
    same = bool(np.array_equal(scores['k1'], scores['k1p']))
    n_graph = args.graph_steps * args.batch
    return {
        'pocket_atoms': int(rec[0].shape[0]),
        'crop_radius': None if not np.isfinite(radius) else radius,
        'atoms_per_complex': round(atoms / n_graph, 1),
        'edges_per_pose': round(edges['k1'] / n_graph, 1),
        'receptor_receptor_edges_cached': pocket.n_rr_edges,
        'graph_ms_per_batch': {k: round(min(v), 4) for k, v in graph_ms.items()},
        'graph_ms_per_batch_rounds': {k: [round(x, 4) for x in v]
                                      for k, v in graph_ms.items()},
        'graph_speedup': round(min(graph_ms['k1']) / min(graph_ms['k1p']), 3),
        'poses_per_s': {k: round(max(v), 1) for k, v in e2e.items()},
        'poses_per_s_rounds': {k: [round(x, 1) for x in v] for k, v in e2e.items()},
        'e2e_ratio_k1p_over_k1': round(max(e2e['k1p']) / max(e2e['k1']), 4),
        'scores_bitwise_equal': same,
        'scores_max_abs_diff': float(np.abs(scores['k1'] - scores['k1p']).max()),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=128)
    ap.add_argument('--steps', type=int, default=60)
    ap.add_argument('--graph-steps', type=int, default=60)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--pool', type=int, default=1024)
    ap.add_argument('--pockets', default='800,3000')
    ap.add_argument('--math', default='bf16x3')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    dev = torch.device('cuda')
    torch.manual_seed(0)
    model = pv.SartorrasEGNN(Path(tempfile.mkdtemp()), 0, 0, None, None, silent=True,
                             **bench.MODEL_KW).to(dev).eval()
    model.set_math(args.math)
    model.set_record_side_channels(False)
    model.record_embed_coords = False
    result = dict(gpu_info(), batch=args.batch, ligand_atoms=N_LIG, math=args.math,
                  model='egnn 8 x 64', edge_radii=[4.0, 4.0],
                  steps=args.steps, graph_steps=args.graph_steps, rounds=args.rounds,
                  cases=[])
    for n_pocket in (int(x) for x in args.pockets.split(',')):
        rec, ligs = make_pocket(n_pocket, args.pool, dev)
        for radius in (np.inf, 10.0):
            case = run_case(model, rec, ligs, radius, args, dev)
            print(json.dumps(case), file=sys.stderr)
            result['cases'].append(case)
    text = json.dumps(result, indent=1)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + '\n')
    print(text)


if __name__ == '__main__':
    main()
