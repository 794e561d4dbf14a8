#!/usr/bin/env python
"""Benchmark of the OpenScene hot path on B200: MinkUNet34C forward + 768-d cosine matching.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference ...                     CPU restatement of the reference path (oracle/)
    python bench.py ... --dump-outputs DIR                   also write the last timed step's results as DIR/*.npy

A step = one synthetic ScanNet-shaped scene (BASELINE.json configs[1]: ~200k voxels) through
  coordinate hashing + stride sets + kernel maps  ->  MinkUNet34C forward (768-d head)  ->
  per-point L2-normalise + [N,768]x[768,20] cosine scores + argmax.
`value`  : voxels/s with coords/feats already in HBM (whole job, all ranks).
`e2e`    : same metric through the public API with pinned HOST buffers: H2D of coords/feats and D2H of the labels
           inside the timed region.
One scene per GPU with no data-path collective; every rank processes the same seed-0 scene, i.e. the work per GPU is
fixed as N grows (weak scaling; see scene_seed); timing = CUDA events, max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='osb200', choices=['osb200', 'reference'])
    ap.add_argument('--workload', default='config2_200k')
    ap.add_argument('--arch', default='MinkUNet34C')
    ap.add_argument('--k-text', type=int, default=None, help='text embeddings (default 20; 160 for config4_matterport, 16 for config5_lidar)')
    ap.add_argument('--match', default=None, choices=['cosine', 'ensemble'], help="matching step: cosine (default) or run/evaluate.py's ensemble path (default for config4_matterport)")
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--modules', action='store_true', help='time the module-by-module MinkowskiEngine surface instead of the fused engine')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last timed step returned as DIR/<name>.npy (see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


DUMP_ROWS = 8192          # rows of the wide per-voxel outputs kept by --dump-outputs (all rows of one scene: ~600 MB)


def voxel_outputs(features, scores, labels):
    """The per-voxel results of one step: every label, and features / scores at a fixed seeded sample of rows (rows.npy).
    The inputs are seeded too, so two builds run with the same arguments can be compared file by file."""
    rows = np.sort(np.random.RandomState(0).choice(len(labels), min(len(labels), DUMP_ROWS), replace=False))
    idx = torch.from_numpy(rows).to(features.device)
    return {'labels': labels.cpu().numpy(), 'rows': rows, 'features': features[idx].float().cpu().numpy(),
            'scores': scores[idx].float().cpu().numpy()}


def dump_outputs(path, arrays):
    """--dump-outputs: each array as <path>/<name>.npy, floating point as float32 (float64 stays float64), integers as
    float64 (exact); 64 MB at most in all."""
    conv = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        conv[name] = a.astype(np.float32 if a.dtype.kind == 'f' and a.dtype.itemsize <= 4 else np.float64)
    total = sum(a.nbytes for a in conv.values())
    assert total <= 64 << 20, f'--dump-outputs would write {total} bytes'
    os.makedirs(path, exist_ok=True)
    for name, a in conv.items():
        np.save(os.path.join(path, name + '.npy'), a)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """Clock evidence for the timed region (B200_PROFILING.md 'clocks' line) without perturbing it.

    * SM clock: measured ON THE DEVICE between timed steps by `osb_measure_sm_mhz` (cycles of clock64 per ns of
      %globaltimer over 20 us; a single-thread kernel outside every step's CUDA-event pair).
    * throttle reasons / max clock: NVML, read immediately before and immediately after the timed region.
    Why not NVML / nvidia-smi during the region: measured here, a query issued while kernels are in flight -- or even right
    after a drain -- intermittently stalls the GPU for 30-70 ms (per-step max 34-67 ms against a 4.6 ms median), and a
    background `nvidia-smi -lms` poller inflated ms/step by 45-100%."""
    REASONS = {'hw_slowdown': 0x8, 'sw_thermal_slowdown': 0x20, 'hw_thermal_slowdown': 0x40, 'sw_power_cap': 0x4}

    def __init__(self, index, dev):
        from openscene_b200 import _cabi
        self.cabi = _cabi
        self.buf = torch.zeros(64, dtype=torch.float32, device=dev)
        self.n = 0
        self.mx, self.reasons, self.ok = None, set(), False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:            # noqa: BLE001
            self.err = str(e)

    def sample(self):
        """enqueue one on-device clock measurement (asynchronous, ~20 us of GPU time)."""
        if self.n < 64:
            self.cabi.call('osb_measure_sm_mhz', self.cabi.c_void_p(self.buf.data_ptr() + 4 * self.n), self.cabi.stream_ptr())
            self.n += 1

    def nvml_reasons(self):
        if not self.ok:
            return
        try:
            r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            for name, bit in self.REASONS.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:                 # noqa: BLE001
            pass

    def stop(self):
        vals = sorted(self.buf[:self.n].cpu().tolist())
        out = {'sm_mhz': vals[len(vals) // 2] if vals else None, 'sm_max_mhz': self.mx, 'reasons': sorted(self.reasons),
               'samples': len(vals), 'how': 'sm_mhz: on-device clock64/globaltimer between timed steps; reasons: NVML right before '
                                            'and right after the timed region'}
        if not self.ok:
            out['reasons'] = ['nvml unavailable: ' + getattr(self, 'err', '')]
        return out


def algorithmic_bytes(census):
    """SURVEY.md 8d: per conv 4*N_in*Cin + 4*N_out*Cout + 4*K*Cin*Cout + 8*pairs."""
    total, flops = 0, 0
    for (name, pairs, cin, cout, n_in, n_out, K) in census:
        pairs = pairs if pairs is not None else 0
        total += 4 * n_in * cin + 4 * n_out * cout + 4 * K * cin * cout + 8 * pairs
        flops += 2 * pairs * cin * cout
    return total, flops


def crop_sample(coords, target):
    """Bounded CPU sample of the workload: the x-slab of the scene holding ~target voxels."""
    if len(coords) <= target:
        return coords
    xs = np.sort(coords[:, 1])
    cut = xs[target]
    return coords[coords[:, 1] < cut]


def cpu_pass(coords, arch, k_text, threads, keep=False):
    """One pass of the CPU restatement (oracle/) over `coords`: map building + forward + cosine matching.
    keep: leave (features, scores, labels) in cpu_pass.last."""
    from openscene_b200 import synth
    from oracle import matching as om
    from oracle import me_cpu
    torch.set_num_threads(threads)
    model = cpu_pass.cache.get(arch)
    if model is None:
        model = synth.build_model(arch, 768, seed=0, ME=me_cpu.as_module()).eval()
        cpu_pass.cache[arch] = model
    text = torch.from_numpy(synth.text_embeddings(k_text))
    feats = torch.ones(len(coords), 3)
    t0 = time.perf_counter()
    with torch.no_grad():
        out = model(me_cpu.SparseTensor(feats, torch.from_numpy(coords)))
        s = om._hmm(om._l2n(out), text)
        label = s.max(1)[1]
    dt = time.perf_counter() - t0
    if keep:
        cpu_pass.last = (out, s, label)
    return dt


cpu_pass.cache = {}


def host_threads():
    """Threads for the CPU arm: the setting that makes it fastest.  Measured on the B200 host (2 x 32-core Xeon 8562Y+,
    128 hardware threads) for this workload: 8 threads 42.4k voxels/s, 16 -> 42.9k, 32 -> 31.6k, 64 -> 14.6k (the many small
    per-offset GEMMs of gather-GEMM-scatter lose to synchronisation beyond one socket's worth of cores).  Default 16,
    override with OSB_CPU_THREADS."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    return max(1, min(n, int(os.environ.get('OSB_CPU_THREADS', 16))))


def scene_seed(rank):
    """Weak scaling = the work per GPU is fixed as N grows, so every rank processes the SAME scene (seed 0, the N=1 workload).
    With per-rank seeds the generator's scenes differ by up to +-8 % in voxel count (seeds 0..7 of config2_200k: 197382, 202435,
    188286, 180984, 195133, 211036, 200222, 207840) and every rank repeats its own scene for all K steps: the max-over-ranks
    time is then the largest scene's while `value` counts the mean -- a persistent imbalance a real run over many scenes per
    rank does not have (no per-step synchronisation in inference).  OSB_BENCH_SCENES=distinct restores one seed per rank."""
    return rank if os.environ.get('OSB_BENCH_SCENES', 'same') == 'distinct' else 0


def workload_config(args, n_vox):
    """The `config` object, identical in both arms (the driver compares them)."""
    return {'workload': f'{args.workload}: {n_vox} voxels/scene, one scene per GPU, {args.arch}, 768-d head, '
                        f'K_text={args.k_text}, ' + ('ensemble matching (2 cosine products + select + final product, run/evaluate.py:302-323)'
                                                      if getattr(args, 'match', 'cosine') == 'ensemble' else 'cosine (L2-normalised) scores') + ' + argmax',
            'points': 'stride-1 voxels fed to SparseTensor',
            'scenes': ('one generator seed per rank (OSB_BENCH_SCENES=distinct)' if os.environ.get('OSB_BENCH_SCENES', 'same') == 'distinct'
                       else 'every rank processes the same seed-0 scene: per-GPU work exactly fixed (weak scaling)'),
            'l2': 'GPU arm: L2 flushed (256 MiB memset) before every timed step; CPU arm: working set (~2 GB of activations) '
                  'far beyond the last-level cache'}


def run_reference(args, rank):
    """`--impl reference`: the reference's CPU path for this metric.  MinkowskiEngine itself is not installable
    offline (SURVEY.md 0.1), so this times oracle/ -- the PyTorch-CPU restatement of the same algorithm -- on the SAME
    scene as the GPU arm (the full workload; ~5 s per step for config2_200k on 16 host threads).  Only if the whole
    `--steps K --warmup W` run would exceed ~6 minutes is the per-step sample cut to an x-slab of the scene, and the line
    then says so (`same_config: false`)."""
    if rank != 0:
        return
    from openscene_b200 import synth
    scene = synth.scene(args.workload, seed=0)
    coords = scene
    threads = host_threads()
    t_probe = cpu_pass(coords, args.arch, args.k_text, threads)          # first pass: also the first warm-up
    budget_s, total = 360.0, args.steps + max(args.warmup, 1)
    if t_probe * total > budget_s:
        coords = crop_sample(scene, max(4000, int(len(coords) * budget_s / (t_probe * total))))
    for _ in range(max(args.warmup - 1, 1 if coords is not scene else 0)):
        cpu_pass(coords, args.arch, args.k_text, threads)
    ts = [cpu_pass(coords, args.arch, args.k_text, threads, keep=i == args.steps - 1) for i in range(args.steps)]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, voxel_outputs(*cpu_pass.last))
    tot = sum(ts)
    value = len(coords) * args.steps / tot
    full = len(coords) == len(scene)
    line = {'impl': 'reference', 'metric': 'voxels/s MinkUNet34C fwd + 768-d cosine-sim', 'value': value, 'unit': 'voxels/s',
            'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * tot / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args, len(scene)), 'same_config': full,
            'voxels_per_step': len(coords), 'voxels_per_step_gpu_arm': len(scene),
            'cpu_baseline': {'value': value, 'unit': 'voxels/s', 'cores': threads, 'kind': 'port',
                             'sample': (f'the full {args.workload} scene, {len(coords)} voxels per step' if full else
                                        f'x-slab crop of {args.workload}: {len(coords)} of {len(scene)} voxels per step '
                                        f'(a full-scene step takes {t_probe:.1f} s)'),
                             'note': 'PyTorch-CPU restatement of gather-GEMM-scatter (oracle/), not MinkowskiEngine itself'},
            'e2e': {'value': value, 'unit': 'voxels/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


def run_distill(args, rank, local, world):
    """`--workload config3_distill`: one step of run/distill.py:311-334 per rank -- random integer translation, forward with
    BatchNorm in train mode, row select by the supervision mask, cosine distillation loss against fp16 fused features,
    backward (dgrad + wgrad on tensor cores), DDP gradient all-reduce over NCCL (world > 1), Adam step.  One ScanNet-shaped
    scene per GPU (batch_size 8 over 8 GPUs, config/scannet/ours_openseg.yaml:14-16), MinkUNet18A unless --arch says otherwise,
    M = 20,000 supervised voxels per scene (scripts/feature_fusion/scannet_openseg.py:145-147)."""
    import torch.distributed as dist
    from openscene_b200 import _cabi, distill, synth
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    arch = args.arch if args.arch != 'MinkUNet34C' or os.environ.get('OSB_DISTILL_34C') else 'MinkUNet18A'
    coords_np = synth.scene('config2_200k', seed=scene_seed(rank))
    n0 = len(coords_np)
    g = torch.Generator().manual_seed(100 + rank)
    m_sup = min(20_000, n0)
    mask_h = torch.zeros(n0, dtype=torch.bool)
    mask_h[torch.randperm(n0, generator=g)[:m_sup]] = True
    feat3d_h = (torch.randn(m_sup, 768, generator=g) * 0.3).half().pin_memory()
    coords_h = torch.from_numpy(coords_np).pin_memory()
    feats_h = torch.ones(n0, 3).pin_memory()
    mask_h = mask_h.pin_memory()
    torch.manual_seed(0)
    model = synth.build_model(arch, 768, seed=0).train().to(dev)
    ddp = distill.wrap_ddp(model, dev)
    opt = torch.optim.Adam(ddp.parameters(), lr=1e-4)                  # run/distill.py:141
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    loss_host = torch.zeros(1).pin_memory()

    def step(sync=True):
        """H2D of the batch, the step, D2H of the loss: the call a user of run/distill.py makes per iteration."""
        c, f = coords_h.to(dev, non_blocking=True), feats_h.to(dev, non_blocking=True)
        t3, mk = feat3d_h.to(dev, non_blocking=True), mask_h.to(dev, non_blocking=True)
        ctx = ddp.no_sync() if (not sync and world > 1) else _null()
        with ctx:
            loss = distill.distill_step(ddp, opt, c, f, t3, mk, 'cosine', translate=True)
        loss_host.copy_(loss.reshape(1), non_blocking=True)
        return loss

    last = {}

    def timed(fn, k):
        import gc
        gc.collect(); gc.disable()
        evs = []
        for i in range(k):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); r = fn(); b.record()
            evs.append((a, b))
            if i == k - 1:
                last['loss'] = r
        torch.cuda.synchronize()
        gc.enable()
        seq = [a.elapsed_time(b) for a, b in evs]
        ts = sorted(seq)
        return sum(ts), {'min': ts[0], 'median': ts[len(ts) // 2], 'max': ts[-1], 'in_order': [round(t, 2) for t in seq[:64]]}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local, dev) if rank == 0 else None
    # at least 10 untimed steps: DDP rebuilds its buckets after the first iteration, NCCL sets its channels up lazily, and the
    # random translation changes the coarse-level sizes from step to step until the caching allocator has seen the range
    n_warm = max(args.warmup, 10)
    for _ in range(n_warm):
        step()
    barrier()
    l0 = _cabi.lib().osb_launch_count()
    if sampler:
        sampler.nvml_reasons(); torch.cuda.synchronize()
    ms, stats = timed(step, args.steps)
    if sampler:
        sampler.sample(); sampler.nvml_reasons()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'loss': last['loss'].reshape(1).cpu().numpy()})
    launches = _cabi.lib().osb_launch_count() - l0
    barrier()
    ms_nosync = None
    if world > 1:                                                      # the same step without the gradient all-reduce
        for _ in range(2):
            step(sync=False)
        barrier()
        ms_nosync, _ = timed(lambda: step(sync=False), max(3, args.steps // 2))
        ms_nosync /= max(3, args.steps // 2)
        barrier()
    stats_t = torch.tensor([ms, float(n0)], dtype=torch.float64, device=dev)
    if world > 1:
        allst = [torch.zeros_like(stats_t) for _ in range(world)]
        dist.all_gather(allst, stats_t)
        allst = torch.stack(allst).cpu()
    else:
        allst = stats_t.cpu().unsqueeze(0)
    t_all, total_vox = float(allst[:, 0].max()), float(allst[:, 1].sum())
    if rank == 0:
        n_par = sum(p.numel() for p in model.parameters())
        value = total_vox * args.steps / (t_all / 1e3)
        line = {'metric': 'voxels/s distillation step (fwd + cosine loss + bwd + Adam)', 'value': value, 'unit': 'voxels/s',
                'n_gpus': world, 'steps': args.steps, 'warmup': n_warm, 'ms_per_step': t_all / args.steps,
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'bf16x3 (split fp32 operands, fp32 accumulate); wgrad bf16x4', 'data': 'synthetic',
                'config': {'workload': f'config3_distill: one config2_200k scene ({n0} voxels) per GPU, {arch}, 768-d head, '
                                       f'{m_sup} supervised voxels, cosine loss, Adam, DDP/NCCL gradient all-reduce of '
                                       f'{n_par * 4 / 1e6:.0f} MB', 'points': 'stride-1 voxels fed to SparseTensor',
                           'scenes': ('one generator seed per rank' if scene_seed(1) else 'every rank trains on the same seed-0 scene '
                                      '(per-GPU work exactly fixed); supervision mask and target features differ per rank'),
                           'l2': 'flushed (256 MiB memset) before every timed step'},
                'e2e': {'value': value, 'unit': 'voxels/s', 'ms_per_step': t_all / args.steps,
                        'h2d_bytes_per_step': int(coords_h.numel() * 4 + feats_h.numel() * 4 + feat3d_h.numel() * 2 + mask_h.numel()),
                        'd2h_bytes_per_step': 4, 'note': 'the timed step IS the end-to-end call: H2D of the batch and D2H of the loss inside'},
                'gpu_launches': int(launches), 'clocks': sampler.stop() if sampler else None, 'step_ms_stats': stats,
                'allreduce': None if ms_nosync is None else {
                    'ms_per_step_with': t_all / args.steps, 'ms_per_step_without': ms_nosync,
                    'exposed_ms': t_all / args.steps - ms_nosync, 'bytes': n_par * 4,
                    'note': 'rank-0 step time under DDP.no_sync() vs the DDP step; the difference is the all-reduce time not hidden '
                            'behind backward'}}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


class _null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def main():
    args = parse()
    if args.workload == 'config3_distill' and args.impl != 'reference':
        return run_distill(args, int(os.environ.get('RANK', 0)), int(os.environ.get('LOCAL_RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)))
    if args.k_text is None:
        args.k_text = {'config4_matterport': 160, 'config5_lidar': 16}.get(args.workload, 20)
    if args.match is None:
        args.match = 'ensemble' if args.workload == 'config4_matterport' else 'cosine'
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        return run_reference(args, rank)

    import torch.distributed as dist
    from openscene_b200 import _cabi, engine, matching, synth, tc
    from openscene_b200 import me as ME
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    # ---- workload: one scene per rank (weak scaling), seeded by rank ---------------------------------
    coords_np = synth.scene(args.workload, seed=scene_seed(rank))
    n0 = len(coords_np)
    coords_host = torch.from_numpy(coords_np).pin_memory()
    feats_host = torch.ones(n0, 3).pin_memory()                      # dataset/feature_loader.py:184
    coords_dev, feats_dev = coords_host.to(dev), feats_host.to(dev)
    text = torch.from_numpy(synth.text_embeddings(args.k_text)).to(dev)
    model = synth.build_model(args.arch, 768, seed=0).eval().to(dev)
    eng = engine.FusedMinkUNet(model)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    feat2d = None
    if args.match == 'ensemble':                                    # fused 2-D features of the scene, fp16 as stored (fusion_util.py:87)
        g2 = torch.Generator(device=dev).manual_seed(11 + rank)
        feat2d = (torch.randn(n0, 768, device=dev, generator=g2) * 0.3).half()

    def match(out):
        if args.match == 'ensemble':                                 # run/evaluate.py:302-323: two cosine products, select, final product
            s_, l_, _, _ = matching.match_ensemble(out, feat2d, None, text)
            return s_, l_, None
        return matching._scores(out, None, text, normalize=True)

    def step_device():
        if args.modules:
            with torch.no_grad():                                    # as run/evaluate.py:260
                out = model(ME.SparseTensor(feats_dev, coords_dev))
        else:
            out = eng(coords_dev, feats_dev)
        return out, match(out)

    label_host = [torch.empty(n0, dtype=torch.int64).pin_memory() for _ in range(4)]   # ring of pinned result buffers
    e2e_i = [0]

    def step_e2e():
        """Public-API call with HOST buffers: H2D of this step's coords/feats from pinned memory, forward + matching,
        D2H of the labels into pinned memory -- all stream-ordered inside the step's event pair; the host only
        blocks on the results at the end of the timed region (a serving loop would consume them a step later)."""
        c = coords_host.to(dev, non_blocking=True)
        f = feats_host.to(dev, non_blocking=True)
        with torch.no_grad():
            out = model(ME.SparseTensor(f, c)) if args.modules else eng(c, f)
        _, label, _ = match(out)
        buf = label_host[e2e_i[0] % len(label_host)]
        e2e_i[0] += 1
        buf.copy_(label, non_blocking=True)
        return buf

    step_stats, last = {}, {}

    def timed(fn, k, sampler=None, tag=None):
        import gc
        evs = []
        gc.collect()
        gc.disable()                                                 # no collector pauses between enqueues
        try:
            for i in range(k):
                flush.zero_()                                        # L2 flush, outside the timed events
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); r = fn(); b.record()
                if tag and i == k - 1:
                    last[tag] = r                            # only the last step's result outlives its step
                del r
                evs.append((a, b))
                if sampler is not None and i in (k // 4, k // 2, (3 * k) // 4):
                    # on-device clock measurement, stream-ordered between two steps (outside their event pairs)
                    sampler.sample()
            torch.cuda.synchronize()
        finally:
            gc.enable()
        ts = sorted(a.elapsed_time(b) for a, b in evs)
        if tag:
            step_stats[tag] = {'min': ts[0], 'median': ts[len(ts) // 2], 'max': ts[-1]}
        return sum(ts)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local, dev) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    l0 = _cabi.lib().osb_launch_count()
    if sampler:
        sampler.nvml_reasons()                                 # throttle reasons right before ...
        torch.cuda.synchronize()
    ms_dev = timed(step_device, args.steps, sampler, tag='device')
    if sampler:
        sampler.nvml_reasons()                                 # ... and right after the timed region
    launches = _cabi.lib().osb_launch_count() - l0
    barrier()
    if args.dump_outputs and rank == 0:
        out, (scores, label, _) = last.pop('device')
        dump_outputs(args.dump_outputs, voxel_outputs(out, scores, label))
    last.clear()
    clocks = sampler.stop() if sampler else None
    for _ in range(2):
        step_e2e()
    barrier()
    ms_e2e = timed(step_e2e, args.steps, tag='e2e')
    barrier()

    # ---- the same step from RAW POINTS (dataset/voxelizer.py on the device): H2D of float32 points, voxelise (affine, floor,
    #      FNV key, first-occurrence unique), network, matching with the voxel->point expansion fused in, D2H of per-point labels
    ms_points, n_pts = None, 0
    if not args.modules:
        from openscene_b200.voxelize import voxelize_points
        pts_np, vsize = synth.scene_points(args.workload, seed=scene_seed(rank))
        n_pts = len(pts_np)
        pts_host = torch.from_numpy(pts_np.astype(np.float32)).pin_memory()
        Mv = np.eye(4); Mv[0, 0] = Mv[1, 1] = Mv[2, 2] = 1.0 / vsize
        plabel_host = torch.empty(n_pts, dtype=torch.int64).pin_memory()

        def step_points():
            p = pts_host.to(dev, non_blocking=True)
            cv, inds, inv, _ = voxelize_points(p, Mv)                 # SYNC inside: the voxel count comes back to the host
            c4 = torch.zeros((cv.shape[0], 4), dtype=torch.int32, device=dev)
            c4[:, 1:] = cv
            out = eng(c4, torch.ones(cv.shape[0], 3, device=dev))
            if args.match == 'ensemble':
                _, lab, _, _ = matching.match_ensemble(out, feat2d[:cv.shape[0]], inv, text)
            else:
                _, lab, _ = matching._scores(out, inv, text, normalize=True, want_scores=False)
            plabel_host.copy_(lab, non_blocking=True)
        # extra measurement: never fail the headline.  Every rank passes the SAME two barriers whether or not its own
        # attempt raised (a rank that skipped one would pair its next collective with the others' barrier).
        ok_points = True
        try:
            for _ in range(2):
                step_points()
        except Exception as e:                                        # noqa: BLE001
            ok_points = False
            print(f'[bench] e2e_points skipped: {e}', file=sys.stderr)
        barrier()
        if ok_points:
            try:
                ms_points = timed(step_points, min(args.steps, 20)) / min(args.steps, 20)
            except Exception as e:                                    # noqa: BLE001
                ms_points = None
                print(f'[bench] e2e_points skipped: {e}', file=sys.stderr)
        barrier()

    # ---- optional re-associated head (not the headline: the 768-d features are not materialised) -----
    ms_folded = None
    if not args.modules:
        folded = eng.fold_head(text.float())
        step_folded = lambda: eng.forward_scores(coords_dev, feats_dev, folded)
        for _ in range(2):
            step_folded()
        barrier()
        ms_folded = timed(step_folded, min(args.steps, 20)) / min(args.steps, 20)

    # ---- dominant kernel (k_conv_chain, or k_conv_tc with OSB_CHAIN=0) timed live with CUDA events on the launching stream -------------
    conv_ms, conv_calls = 0.0, 0
    if not args.modules:
        pend = []
        hooked_names = ('osb_conv_fwd_tc', 'osb_convtr_fwd_tc', 'osb_conv_chain_launch')   # every tensor-core convolution launch

        def make_hook(real_fn):
            def hooked(*a):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); r = real_fn(*a); e1.record()
                pend.append((e0, e1))
                return r
            return hooked
        reps = 3
        orig_lib = _cabi.lib
        hooks = {nm: make_hook(getattr(orig_lib(), nm)) for nm in hooked_names}

        class LibProxy:                    # the engine calls lib().<fn>(...) directly with raw addresses
            def __getattr__(self, name):
                return hooks[name] if name in hooks else getattr(orig_lib(), name)
        engine.C.lib = lambda: LibProxy()
        for _ in range(reps):
            flush.zero_()
            step_device()
        torch.cuda.synchronize()
        engine.C.lib = orig_lib
        conv_ms = sum(a.elapsed_time(b) for a, b in pend) / reps
        conv_calls = len(pend) // reps
        census = eng.conv_census(eng.last_cm)
        tc_rows = [r for r in census if r[0] != 'stem']
        conv_bytes, conv_flops = algorithmic_bytes(tc_rows)
        all_bytes, all_flops = algorithmic_bytes(census)

    # ---- gather over ranks: max time, sum of voxels -----------------------------------------------
    stats = torch.tensor([ms_dev, ms_e2e, float(n0)], dtype=torch.float64, device=dev)
    if world > 1:
        allst = [torch.zeros_like(stats) for _ in range(world)]
        dist.all_gather(allst, stats)
        allst = torch.stack(allst).cpu()
    else:
        allst = stats.cpu().unsqueeze(0)
    t_dev, t_e2e, total_vox = float(allst[:, 0].max()), float(allst[:, 1].max()), float(allst[:, 2].sum())
    if rank == 0:
        peak, peak_src = peaks()
        line = {
            'metric': 'voxels/s MinkUNet34C fwd + 768-d cosine-sim', 'value': total_vox * args.steps / (t_dev / 1e3),
            'unit': 'voxels/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': t_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16x3 (split fp32 operands, fp32 accumulate)', 'data': 'synthetic',
            'config': workload_config(args, n0), 'path': 'module surface' if args.modules else 'fused engine',
            'e2e': {'value': total_vox * args.steps / (t_e2e / 1e3), 'unit': 'voxels/s', 'ms_per_step': t_e2e / args.steps,
                    'h2d_bytes_per_step': int(coords_host.numel() * 4 + feats_host.numel() * 4), 'd2h_bytes_per_step': int(n0 * 8)},
            'gpu_launches': int(launches), 'clocks': clocks, 'step_ms_stats': step_stats,
        }
        if ms_points is not None:
            line['e2e_points'] = {'ms_per_step': ms_points, 'points_per_s': n_pts / (ms_points / 1e3), 'voxels_per_s': n0 / (ms_points / 1e3),
                                  'n_points': n_pts, 'h2d_bytes_per_step': n_pts * 12, 'd2h_bytes_per_step': n_pts * 8,
                                  'note': 'rank 0: float32 points from pinned host memory -> osb_voxelize -> engine -> matching through '
                                          'inds_reverse -> int64 labels per POINT back to pinned host memory'}
        if ms_folded is not None:
            line['extra'] = {'folded_head_ms_per_step': ms_folded,
                             'note': 'optional engine.forward_scores: final 1x1x1 conv re-associated with the text matrix '
                                     '(W W^T = L L^T, U = W T^T); same cosine scores, no 768-d features written; rank-0 time'}
        if not args.modules:
            ach = conv_bytes / (conv_ms * 1e-3) / 1e9
            traffic = None
            tpath = os.path.join(ROOT, 'profiles', 'traffic.json')     # dram bytes per launch from the committed ncu --set full capture
            if os.path.exists(tpath):
                traffic = json.load(open(tpath))
            line['roofline'] = {'bound': 'hbm', 'kernel': 'k_conv_chain' if eng.use_chain else 'k_conv_tc', 'achieved': ach, 'peak': peak, 'unit': 'GB/s',
                                'frac': ach / peak, 'traffic': traffic['dram_bytes_per_launch'] if traffic else None,
                                'traffic_note': traffic['note'] if traffic else None, 'peak_source': peak_src,
                                'launches_per_step': conv_calls, 'kernel_ms_per_step': conv_ms,
                                'algorithmic_bytes_per_step': conv_bytes, 'tflops': conv_flops / (conv_ms * 1e-3) / 1e12,
                                'step_algorithmic_bytes': all_bytes, 'step_gflop': all_flops / 1e9}
            try:      # second lens: bf16 MMA work behind the algorithmic fp32 flops (3 passes per product) vs the measured bf16 peak
                pk = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))).get('bf16_tflops')
                if pk:
                    tf3 = 3.0 * line['roofline']['tflops']
                    line['roofline']['tensor_lens'] = {
                        'bf16_tflops': tf3, 'peak': float(pk), 'frac': tf3 / float(pk),
                        'note': 'algorithmic pairs x 3 bf16 passes; the 128-row tiles also multiply the zero rows of missing '
                                'neighbours (about half of the rows at level 0), so the tensor pipe itself is ~2x busier: 52% '
                                'active on the level-0 layers (profiles/r01_ncu_full_conv_tc_96x96_k3_final.md, first-generation kernel)'}
            except Exception:
                pass
            # third lens: operand bytes the gather-per-offset algorithm pulls from L2 into the SMs (every 128-row tile re-reads
            # its rows for each kernel offset and a weight tile per stage and item) against the L2 throughput cap
            op_bytes = 0
            for (name, pairs, cin, cout, n_in, n_out, K) in tc_rows:
                cp = (cout + 15) // 16 * 16 if cout <= 256 else (cout + 255) // 256 * 256
                nt = min(cp, 256)
                m_tiles = (n_out + 127) // 128
                items = m_tiles if nt > 128 else (m_tiles + 1) // 2
                op_bytes += m_tiles * (cp // nt) * K * (cin // 32) * 128 * 128 + items * (cp // nt) * K * (cin // 32) * nt * 128
            sm_mhz = (clocks or {}).get('sm_mhz') or 1965
            cap = 6300.0 * sm_mhz * 1e6 / 1e9            # B/cycle full chip (B300_MICROARCH.md 'LTS throughput cap') x SM clock
            line['roofline']['l2_lens'] = {
                'operand_bytes_per_step': int(op_bytes), 'achieved_GBps': op_bytes / (conv_ms * 1e-3) / 1e9, 'cap_GBps': cap,
                'frac': op_bytes / (conv_ms * 1e-3) / 1e9 / cap,
                'note': 'split-bf16 rows (4 B per value) gathered once per kernel offset + pre-swizzled weight tiles; this L2->SM '
                        'stream, not HBM or the tensor pipe, is what the level-0/1 layers run against (profiles/r02_chain_roles.md)'}
        if world == 1 and not args.no_cpu_baseline:
            threads = host_threads()
            cpu_pass(coords_np, args.arch, args.k_text, threads)                   # warm-up pass (allocator, thread pool)
            dt = cpu_pass(coords_np, args.arch, args.k_text, threads)
            line['cpu_baseline'] = {'value': n0 / dt, 'unit': 'voxels/s', 'cores': threads, 'kind': 'port',
                                    'sample': f'the full scene of this run ({n0} voxels): one warm-up pass + one timed pass of {dt:.1f} s',
                                    'note': 'PyTorch-CPU restatement of gather-GEMM-scatter (oracle/), not MinkowskiEngine'}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
