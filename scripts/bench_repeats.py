#!/usr/bin/env python
"""Test-time repeats on one scene: ``RepeatEvaluator`` against R single-pass evaluations.

    python scripts/bench_repeats.py --out DIR [--repeats 1 5] [--iters 10] [--warmup 3]

Scene: the config-2 room of ``synth.room_points`` (ScanNet-shaped, ~200k voxels), MinkUNet18A (the architecture every
``ours_*`` config names) with a 768-d head, K = 20 text rows, feature_type 'ensemble', fp16 fused features on ~80 % of the
points.  Per R, three arms run alternately on the same R voxelisation matrices, timed with CUDA events after warm-up:
  (a) ``RepeatEvaluator.add_scene``: one forward over the R voxel sets, the fp16 score sum kept on the device;
  (b) R passes of voxelise / remap / forward / ``match_ensemble`` with ``store = pred + store`` in torch on the device;
  (c) arm (b) with the reference's host accumulation: ``pred.cpu()`` every repeat, added and reduced on the CPU.
Device-to-host bytes per scene come from one profiled scene per arm (memcpy records of a torch.profiler trace), outside
the timed loop.  Writes DIR/bench_repeats.json and prints it.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or 'not measured'
    except (OSError, subprocess.TimeoutExpired):
        power = 'not measured'
    return name, power


def d2h_bytes(fn):
    """Device-to-host bytes of one call of fn, from the memcpy records of a profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, 'trace.json')
        prof.export_chrome_trace(path)
        events = json.load(open(path)).get('traceEvents', [])
    return int(sum(e.get('args', {}).get('bytes', 0) for e in events
                   if e.get('cat') == 'gpu_memcpy' and 'DtoH' in e.get('name', '')))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--repeats', type=int, nargs='+', default=[1, 5])
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--k-text', type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit('bench_repeats.py measures on a CUDA device; none is visible')
    from openscene_b200 import matching, pipeline, synth
    from openscene_b200.engine import FusedMinkUNet
    from openscene_b200.fused_features import remap_fused_features
    from openscene_b200.metric import ConfusionMeter
    from openscene_b200.voxelize import Voxelizer, voxelize_points

    dev = torch.device('cuda:0')
    pts_np, voxel = synth.scene_points('config2_200k')
    n = len(pts_np)
    rng = np.random.RandomState(0)
    points = torch.from_numpy(pts_np).to(dev)
    gt = torch.from_numpy(rng.randint(0, 20, n)).to(dev)
    mask_full = torch.from_numpy(rng.rand(n) < 0.8).to(dev)
    feat = (torch.randn(int(mask_full.sum()), 768, device=dev) * 0.3).half()
    text = torch.from_numpy(synth.text_embeddings(a.k_text)).to(dev)
    engine = FusedMinkUNet(synth.build_model('MinkUNet18A', 768, seed=0).eval().to(dev))
    vox = Voxelizer(voxel_size=voxel, use_augmentation=True, scale_augmentation_bound=pipeline.LOADER_SCALE_BOUND,
                    rotation_augmentation_bound=pipeline.LOADER_ROTATION_BOUND)
    name, power = card()
    result = {'card': name, 'power_limit': power, 'scene': 'config2_200k', 'n_points': n, 'arch': 'MinkUNet18A', 'c': 768,
              'k_text': a.k_text, 'feature_type': 'ensemble', 'iters': a.iters, 'warmup': a.warmup, 'runs': []}

    for R in a.repeats:
        np.random.seed(R)
        mats = [(lambda m: m[1] @ m[0])(vox.get_transformation_matrix()) for _ in range(R)]
        ev = pipeline.RepeatEvaluator(engine, text, feature_type='ensemble', test_repeats=R, voxel_size=voxel)
        meters = [ConfusionMeter(20, dev) for _ in range(R)]
        n_vox = [int(voxelize_points(points, M)[0].shape[0]) for M in mats]

        def arm_a():
            return ev.add_scene(points, gt, fused=(feat, mask_full), matrices=mats)

        def solo(host):
            store = 0.0
            for r, M in enumerate(mats):
                cv, inds, inv, _ = voxelize_points(points, M)
                coords = torch.zeros((cv.shape[0], 4), dtype=torch.int32, device=dev)
                coords[:, 1:] = cv
                fv, _ = remap_fused_features(feat, mask_full, inds, split='val', device=dev)
                out = engine(coords, torch.ones((cv.shape[0], 3), device=dev))
                s, _, _, _ = matching.match_ensemble(out, fv, inv, text)
                store = (s.cpu() if host else s) + store
                lab = store.float().max(1)[1]
                meters[r].update(lab, gt)
            return lab.to(dev)

        arms = {'a_repeat_evaluator': arm_a, 'b_single_pass_device_sum': lambda: solo(False),
                'c_single_pass_host_sum': lambda: solo(True)}
        labels = {k: fn() for k, fn in arms.items()}
        for _ in range(a.warmup):
            for fn in arms.values():
                fn()
        times = {k: [] for k in arms}
        for _ in range(a.iters):
            for k, fn in arms.items():
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1))
        run = {'repeats': R, 'n_vox': n_vox, 'arms': {}}
        for k, fn in arms.items():
            t = np.array(times[k])
            run['arms'][k] = {'ms_per_scene': {'min': float(t.min()), 'median': float(np.median(t)), 'max': float(t.max())},
                              'points_per_s': float(n / (np.median(t) / 1e3)), 'd2h_bytes_per_scene': d2h_bytes(fn)}
        la = labels['a_repeat_evaluator']
        run['label_agreement_a_vs_b'] = float((la == labels['b_single_pass_device_sum']).float().mean())
        run['label_agreement_a_vs_c'] = float((la == labels['c_single_pass_host_sum']).float().mean())
        run['scores_bytes_n_pts_x_k'] = 2 * n * a.k_text
        result['runs'].append(run)
        print(json.dumps(run), flush=True)

    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, 'bench_repeats.json'), 'w') as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == '__main__':
    main()
