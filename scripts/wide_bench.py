"""Scoring throughput at hidden width 128 (the 128-wide tensor-core forward)
beside the k = 64 model, on the bench workload: 8-layer `egnn` with the
BASELINE configs[3] options (bench.MODEL_KW), 128 complexes x 1000 atoms per
step, graph build + forward + score.

    python scripts/wide_bench.py [--steps 20] [--out wide_bench.json]

Per (k, math): complexes/s of the one-call scoring pass, and the edge and
node stages in microseconds per launch from CUDA events around each stage of
a separate per-layer pass (edge = edge kernel + split-node fix-up; node =
node MLP kernel; node_pre = P/Q), with the algorithmic TFLOP/s of each
(edge: 8k^2 + 12k FLOP per edge and layer, node: 6k^2 + 2k per node and
layer).  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

import bench  # noqa: E402
import pointvs_b200 as pv  # noqa: E402
from pointvs_b200 import egnn as egnn_mod  # noqa: E402
from pointvs_b200.synthetic import synthetic_batch  # noqa: E402


def flop_edge(k):
    return 8 * k * k + 12 * k


def flop_node(k):
    return 6 * k * k + 2 * k


class StageEvents:
    """STAGE_TIMER hook: events around each stage call of the per-layer path
    (stages 1 = node_pre, 2 = edge, 4 = node)."""
    split_stages = True

    def __init__(self):
        self.pairs = {1: [], 2: [], 4: []}
        self._begin = None

    def begin(self, stage):
        self._begin = torch.cuda.Event(enable_timing=True)
        self._begin.record()

    def end(self, stage):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.pairs[stage].append((self._begin, e))

    def us(self, stage):
        t = [a.elapsed_time(b) * 1e3 for a, b in self.pairs[stage]]
        return sum(t) / len(t)


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                        '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return {'name': torch.cuda.get_device_name(0),
            'nvidia_smi': q.stdout.strip() if q.returncode == 0 else None}


def run(k, math, steps, warmup, inputs):
    c, b, f, cptr = inputs
    torch.manual_seed(0)
    model = pv.SartorrasEGNN(Path('/tmp/pvs_wide_bench'), 0, 0, None, None,
                             silent=True, **dict(bench.MODEL_KW, k=k))
    model = model.cuda().eval().set_math(math)
    model.set_record_side_channels(False)
    model.record_embed_coords = False

    def step():
        batch = pv.PackedBatch.from_arrays(c, b, f, cptr, bench.EDGE_RADIUS,
                                           bench.EDGE_RADIUS, device='cuda',
                                           edge_capacity='auto')
        with torch.no_grad():
            return model(batch), batch

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    # stage times: one per-layer pass, outside the timed loop
    _, batch = step()
    n_edges = int(batch.edge_index.shape[1])
    n_nodes = int(c.shape[0])
    timer = StageEvents()
    egnn_mod.STAGE_TIMER = timer
    try:
        for _ in range(3):
            with torch.no_grad():
                model(batch)
    finally:
        egnn_mod.STAGE_TIMER = None
    torch.cuda.synchronize()
    edge_us, node_us, pre_us = timer.us(2), timer.us(4), timer.us(1)
    return {
        'k': k, 'math': math, 'complexes_per_s': (len(cptr) - 1) / dt,
        'ms_per_step': dt * 1e3, 'nodes': n_nodes, 'edges': n_edges,
        'edge_us_per_launch': edge_us, 'node_us_per_launch': node_us,
        'node_pre_us_per_launch': pre_us,
        'edge_tflops': n_edges * flop_edge(k) / (edge_us * 1e-6) / 1e12,
        'node_tflops': n_nodes * flop_node(k) / (node_us * 1e-6) / 1e12,
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--out', type=str, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('wide_bench needs a CUDA device')
    torch.cuda.set_device(0)
    coords, bp, feats, cptr = synthetic_batch(0, 128, 1000, 30)
    inputs = tuple(torch.from_numpy(a).cuda() for a in (coords, bp, feats)) + (cptr,)
    results = []
    for math in ('bf16x3', 'fp16x2', 'bf16'):
        for k in (64, 128):
            r = run(k, math, args.steps, args.warmup, inputs)
            print(json.dumps(r), flush=True)
            results.append(r)
    out = {'card': card(), 'workload': '128 x 1000-atom complexes, 8 layers, '
           'bench.MODEL_KW options, edge radius 4.0', 'steps': args.steps,
           'results': results}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w', encoding='utf-8') as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out['card']))


if __name__ == '__main__':
    main()
