#!/usr/bin/env python
"""Headline benchmark of the Mega-NeRF rendering hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host CPU cores

A "step" is one render_rays() pass over one batch of synthetic rays: BASELINE.json configs[1]
(MegaNeRF 8 x 256-wide sub-modules, 4096 rays x (64 coarse + 128 fine) samples, random-init weights).
With N > 1 (torchrun, one rank per GPU) rays are sharded: every rank renders its own 4096 rays with
replicated weights and the per-ray results (rgb + depth) are all-gathered over NCCL each step (weak scaling).

With N > 1 the per-GPU batch is BASELINE configs[2]'s shard (65 536 rays / 8 = 8192 rays per GPU) instead of configs[1]'s 4096.

Prints ONE JSON line on rank 0 (see the task contract): value = ray-samples/s with inputs resident in HBM
(device-timed with CUDA events), e2e = the same through the public API from pinned host buffers including
H2D/D2H, roofline for the dominant (MLP) kernel, cpu_baseline = the oracle port of the reference (`kind: "port"`) timed on
the host cores.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from argparse import Namespace

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_RAYS = 4096
COARSE, FINE = 64, 128
MARGIN = 1.15
# The graded line is 'c2' (BASELINE configs[1]).  'c4' / 'c5' are the other single-GPU-sized BASELINE shapes, selectable
# for diagnostics only (python bench.py --workload c4); their lines carry the same keys.
WORKLOADS = {
    'c2': dict(desc='BASELINE configs[1]: mega-nerf 8-submodule 256-ch', rays=4096, spec={}, grid=(2, 4), sh_deg=None,
               kernel='tc_mlp_tp_kernel'),
    # configs[2]: 65 536 rays per iteration over 8 GPUs = 8192 rays per GPU; the default when N > 1
    'c3': dict(desc='BASELINE configs[2] shard: mega-nerf 8-submodule 256-ch, 65536 rays / 8 GPUs', rays=8192, spec={}, grid=(2, 4),
               sh_deg=None, kernel='tc_mlp_tp_kernel'),
    'c4': dict(desc='BASELINE configs[3] shape: mega-nerf 25-submodule 512-ch', rays=4096, spec=dict(layer_dim=512), grid=(5, 5),
               sh_deg=None, kernel='tc_mlp_wide_kernel'),
    'c5': dict(desc='BASELINE configs[4]: mega-nerf-sh-3 (SH degree 2 head) 8-submodule 256-ch', rays=8192,
               spec=dict(pos_dir_dim=0, rgb_dim=27), grid=(2, 4), sh_deg=2, kernel='tc_mlp_tp_kernel'),
}
WL = WORKLOADS['c2']


def select_workload(name: str) -> None:
    global WL, N_RAYS
    WL = WORKLOADS[name]
    N_RAYS = WL['rays']
L2_FLUSH_BYTES = 256 << 20


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=d['bf16_tflops'], tflops_sustained=d.get('bf16_tflops_sustained'), hbm=d['hbm_gbs'], src='measured')
    return dict(tflops=1590.0, tflops_sustained=1400.0, hbm=6650.0, src='fallback')


def cpu_renderer(O, net, opts):
    """-> (fn(rays, idx) -> results, kind): the oracle port of the reference's render_rays."""
    return (lambda r, i: O.render_rays(net, None, r, i, opts, None, None, True, False, False)[0]), 'port'


def kernel_traffic(kernel: str, workload_name: str, precision: str):
    """DRAM traffic per launch of `kernel` from the committed ncu capture of this workload (profiles/kernel_traffic.json)."""
    p = os.path.join(ROOT, 'profiles', 'kernel_traffic.json')
    if not os.path.exists(p):
        return None
    try:
        for e in json.load(open(p)):
            if e['kernel'] == kernel and e['workload'] == workload_name and e['precision'] == precision:
                return e
    except Exception:  # noqa: BLE001
        pass
    return None


def workload(seed_shift: int = 0):
    from oracle import mn_oracle as O
    spec = O.NerfSpec(**WL['spec'])
    cents = O.grid_centroids(*WL['grid'])
    net = O.make_net('mega', spec, seed=0, n_sub=cents.shape[0], centroids=cents, boundary_margin=MARGIN, cluster_2d=True)
    rays = O.synthetic_rays(N_RAYS, seed=seed_shift)
    idx = O.synthetic_indices(N_RAYS, spec.appearance_count, seed=1 + seed_shift)
    opts = O.RenderOpts(coarse_samples=COARSE, fine_samples=FINE, use_cascade=False, perturb=1.0, pos_dir_dim=spec.pos_dir_dim,
                        sh_deg=WL['sh_deg'], model_chunk_size=32 * 1024)
    return spec, net, rays, idx, opts


def workload_string() -> str:
    """Identical in both arms (the driver compares the strings)."""
    return (f'{WL["desc"]}, {N_RAYS} rays x ({COARSE} coarse + {FINE} fine) samples per GPU, boundary_margin {MARGIN}, '
            'random-init weights, synthetic rays')


def flops_per_row(spec) -> int:
    L, ix = spec.layer_dim, spec.in_xyz
    f = 0
    for i in range(spec.layers):
        kin = ix if i == 0 else (L + ix if i in spec.skip_layers else L)
        f += 2 * kin * L
    f += 2 * L                                   # sigma
    if spec.has_dir_a:
        f += 2 * L * L                           # xyz_encoding_final
        f += 2 * (L + spec.in_dir + (spec.appearance_dim if not spec.affine_appearance else 0)) * (L // 2)
        f += 2 * (L // 2) * spec.rgb_dim
    else:
        f += 2 * L * spec.rgb_dim
    return f


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}', '--format=csv,noheader,nounits',
                                          '-lms', '20'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            # nvidia-smi needs ~0.1-0.3 s before its first row: wait for it, then drop the idle rows so that a short
            # timed region (a few 10-ms training steps) is still covered by samples taken under load
            t0 = time.time()
            while not self.rows and time.time() - t0 < 3.0:
                time.sleep(0.01)
            self.rows.clear()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(sm)}


def usable_cpus() -> int:
    """Host threads this process can really use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        q, p = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = min(n, max(1, int(int(q) / int(p))))
    except Exception:  # noqa: BLE001
        pass
    return max(1, n)


def cpu_rays_per_sec(render, rays, idx, n_probe: int = 64) -> float:
    """Quick probe of the CPU renderer's speed on this host, used to bound the timed CPU samples."""
    with torch.inference_mode():
        render(rays[:n_probe], idx[:n_probe])
        t0 = time.perf_counter()
        render(rays[:n_probe], idx[:n_probe])
        return n_probe / (time.perf_counter() - t0)


def run_reference(args, rank: int):
    """The reference algorithm on the host cores: the oracle port of mega_nerf.rendering.render_rays + mega_nerf.models
    (oracle/mn_oracle.py, kind "port")."""
    if rank != 0:
        return
    from oracle import mn_oracle as O
    torch.set_num_threads(usable_cpus())
    spec, net, rays, idx, opts = workload()
    render, kind = cpu_renderer(O, net, opts)
    rate = cpu_rays_per_sec(render, rays, idx)
    # bounded sample: the whole --steps/--warmup run should take about two minutes of CPU time
    sample = int(min(N_RAYS, max(64, rate * 120.0 / (args.steps + args.warmup)))) // 64 * 64
    r, i = rays[:sample], idx[:sample]
    times = []
    with torch.inference_mode():
        for s in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            render(r, i)
            if s >= args.warmup:
                times.append(time.perf_counter() - t0)
    tot = sum(times)
    value = sample * (COARSE + FINE) * args.steps / tot
    line = {
        'impl': 'reference', 'metric': 'ray-samples/sec (MLP+composite)', 'value': value, 'unit': 'samples/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * tot / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_string(), 'cpu_sample': f'each CPU step renders a {sample}-ray sample of it'},
        'cpu_baseline': {'value': value, 'unit': 'samples/s', 'cores': torch.get_num_threads(), 'kind': kind,
                         'sample': f'{sample} of {N_RAYS} rays per step, {args.steps} steps',
                         'what': 'oracle port of mega_nerf.rendering.render_rays + mega_nerf.models, torch CPU fp32, inference_mode'},
        'e2e': {'value': value, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def gpu_incumbent(O, net, rays_d, idx_d, opts, dev, steps: int = 5):
    """SURVEY.md §8d "GPU incumbent": the oracle restatement of the reference's render_rays over mega_nerf.models (cuBLAS
    GEMMs + ~10^3 ATen elementwise launches per step) through torch-CUDA on the SAME B200 in the three precisions the
    reference can run in - fp32, TF32, and autocast fp16 (its default, runner.py:243).  A baseline leg like cpu_baseline:
    reported next to the product's number, never on the product path.  Any failure is reported, not raised."""
    out = {'kind': 'port (oracle restatement under torch-CUDA eager, same GPU)', 'unit': 'samples/s', 'steps': steps}
    try:
        n = rays_d.shape[0]
        samples = n * (opts.coarse_samples + opts.fine_samples)
        netd = O.net_to(net, dev)
        render = lambda: O.render_rays(netd, None, rays_d, idx_d, opts, None, None, True, False, False)  # noqa: E731
        saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
        for name, tf32, amp in (('fp32', False, False), ('tf32', True, False), ('amp_fp16', True, True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32

            def step():
                with torch.inference_mode(), torch.autocast('cuda', dtype=torch.float16, enabled=amp):
                    render()
            for _ in range(2):
                step()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                step()
            b.record()
            torch.cuda.synchronize()
            ms = a.elapsed_time(b) / steps
            out[name] = {'value': samples / (ms * 1e-3), 'ms_per_step': ms}
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved
    except Exception as e:  # noqa: BLE001
        out['error'] = repr(e)[:300]
    return out


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: every array as out_dir/<name>.npy in float32, so that two builds can be compared output for output."""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items() if torch.is_tensor(v)}
    total = sum(a.nbytes for a in arrays.values())
    if total > 64 << 20:
        raise SystemExit(f'--dump-outputs: {total} bytes of outputs exceed 64 MiB')
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f'{k}.npy'), a)
    log(f'outputs of the last timed step: {sorted(arrays)} -> {out_dir}')


def log(msg):
    if os.environ.get('MN_BENCH_VERBOSE', '1') == '1':
        print(f'[bench {time.strftime("%H:%M:%S")}] {msg}', file=sys.stderr, flush=True)


def run_train(args, rank, local_rank, world):
    """One training step of the reference (runner.py:346-378, :244-274 without AMP): render_rays(get_depth=False,
    get_depth_variance=True) in train() mode, photometric MSE, backward, Adam step.  Rank-sharded rays, gradients
    all-reduced by DistributedDataParallel semantics are NOT part of this diagnostic (N = 1 only)."""
    import mega_nerf_b200 as M
    from mega_nerf_b200 import _cabi as K
    from mega_nerf_b200.synthetic import build_net
    if world != 1:
        raise SystemExit('--mode train is a single-GPU diagnostic')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    spec, net, rays_h, idx_h, opts = workload()
    hp = Namespace(**vars(opts))
    model = build_net(net, dev, trainable=True).train()
    M.set_train_precision(args.train_precision)
    opt = torch.optim.Adam(model.parameters(), lr=5e-4)
    rgbs_h = torch.rand(N_RAYS, 3, generator=torch.Generator().manual_seed(9))
    rays_pin, idx_pin, rgbs_pin = rays_h.pin_memory(), idx_h.pin_memory(), rgbs_h.pin_memory()
    loss_pin = torch.empty(1).pin_memory()
    rays_d, idx_d, rgbs_d = rays_h.to(dev), idx_h.to(dev), rgbs_h.to(dev)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    h, L = K.ctx(dev), K.lib()

    def step(r, i, t):
        res, _ = M.render_rays(model, None, r, i, hp, None, None, False, True, False)
        loss = torch.nn.functional.mse_loss(res['rgb_fine'], t)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        return loss

    def step_resident():
        step(rays_d, idx_d, rgbs_d)

    def step_e2e():
        loss = step(rays_pin.to(dev, non_blocking=True), idx_pin.to(dev, non_blocking=True), rgbs_pin.to(dev, non_blocking=True))
        loss_pin.copy_(loss.detach().view(1), non_blocking=True)

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        torch.cuda.synchronize()
        for a, b in evs:
            flush.fill_(1)
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs)

    for _ in range(args.warmup):
        step_resident()
        step_e2e()
    torch.cuda.synchronize()
    l0 = L.mn_launch_count(h)
    step_resident()
    launches_per_step = L.mn_launch_count(h) - l0
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms = timed(step_resident, args.steps)
    ms_e2e = timed(step_e2e, args.steps)
    K.check(L.mn_profile_enable(h, 1), h)
    timed(step_resident, args.steps)
    tot_ms, n_l = C.c_double(), C.c_longlong()
    K.check(L.mn_profile_read(h, C.byref(tot_ms), C.byref(n_l)), h)
    K.check(L.mn_profile_enable(h, 0), h)
    clocks = sampler.stop()
    slots, _ = model._native().stats(dev)
    mult = slots / (N_RAYS * FINE)
    on_tc = model._native().train_on_tensor_cores()
    other = None
    if args.train_precision == 'tc_f16':
        # the fp32 (parity-mode) step on the same box for comparison, a few steps
        M.set_train_precision('fp32')
        for _ in range(2):
            step_resident()
        other = timed(step_resident, max(2, args.steps // 4)) / max(2, args.steps // 4)
        M.set_train_precision(args.train_precision)
    pk = peaks()
    samples = N_RAYS * (COARSE + FINE)
    flops_step = 3 * samples * mult * flops_per_row(spec)          # forward + data gradients + weight gradients
    kms = tot_ms.value / args.steps
    achieved = flops_step / (kms * 1e-3) / 1e12 if kms > 0 else 0.0
    line = {
        'metric': 'training ray-samples/sec (forward + backward + Adam)', 'value': samples * args.steps / (ms * 1e-3),
        'unit': 'samples/s', 'n_gpus': 1, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f16 operands / f32 accumulate' if on_tc else 'f32', 'data': 'synthetic',
        'config': {'workload': f'{WL["desc"]}, {N_RAYS} rays x ({COARSE} coarse + {FINE} fine), train() mode (jitter, density '
                               f'noise, random resampling), boundary_margin {MARGIN} (m = {mult:.3f}), MSE vs random colours, Adam',
                   'parallelism': 'single GPU',
                   'precision': ('tc_f16: recording forward, data gradients and weight gradients on tcgen05 (fp16 operands, fp32 accumulate)'
                                 if on_tc else 'fp32 (CUDA-core kernels, the parity mode)'),
                   'fp32_parity_mode_ms_per_step': other,
                   'launch': 'eager', 'l2': f'flushed between timed iterations ({L2_FLUSH_BYTES >> 20} MiB write)'},
        'e2e': {'value': samples * args.steps / (ms_e2e * 1e-3), 'unit': 'samples/s', 'ms_per_step': ms_e2e / args.steps,
                'h2d_bytes_per_step': (rays_pin.numel() + idx_pin.numel() + rgbs_pin.numel()) * 4, 'd2h_bytes_per_step': 4},
        'gpu_launches': int(launches_per_step * args.steps),
        'clocks': clocks,
        'roofline': {'bound': 'tensor', 'kernel': ('tc_mlp_pp_kernel<TRAIN_FWD> + tc_mlp_pp_kernel<DGRAD> + tc_wgrad_kernel' if on_tc else
                                                    'mlp_simt_kernel<SAVE> + mlp_bwd_data_kernel + mlp_bwd_weight_kernel'),
                     'achieved': achieved, 'peak': pk['tflops'], 'unit': 'TFLOP/s', 'frac': achieved / pk['tflops'],
                     'peak_source': pk['src'], 'traffic': None, 'kernel_ms_per_step': kms,
                     'note': ('forward + backward MLP kernels timed by CUDA events on the launching stream; 3 x forward FLOPs'
                              if on_tc else 'GEMM-shaped work on the fp32 FMA pipe: the fraction is against the tensor-core peak on purpose')},
    }
    print(json.dumps(line), flush=True)


def run_cluster(args, local_rank):
    """scripts/create_cluster_masks.py:155-201 on its default chunk (ray_chunk_size 48k rays, ray_samples 1000) with the 8
    centroids of the C2 grid: rays/s of mn_cluster_min_dist_ratios, device-timed, next to the restatement on the host cores
    (bounded sample).  The kernel reads 32 B/ray and writes (4K + K) B/ray, so HBM is irrelevant (a few GB/s): the work is
    S x K distance evaluations per ray (sqrt + div each), i.e. it is bound by the fp32 / SFU issue rate; `roofline`
    reports distance evaluations per second against 148 SMs x 128 lanes x clock / ~12 issue slots per evaluation."""
    import mega_nerf_b200 as M  # noqa: F401
    from mega_nerf_b200 import cluster_masks as CM
    from oracle import mn_oracle as O
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    n, S = 48 * 1024, 1000
    rays_h = O.synthetic_rays(n, seed=0, far=1.2)
    cent = O.grid_centroids(2, 4)
    zs = torch.linspace(0, 1, S)
    rays_d, cent_d, zs_d = rays_h.to(dev), cent.to(dev), zs.to(dev)
    rays_pin = rays_h.pin_memory()
    mask_pin = torch.empty(8, n, dtype=torch.uint8).pin_memory()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        torch.cuda.synchronize()
        for a, b in evs:
            flush.fill_(1)
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs)

    def resident():
        CM.min_dist_ratios(rays_d, zs_d, cent_d, True, MARGIN)

    def e2e():
        _, m = CM.min_dist_ratios(rays_pin.to(dev, non_blocking=True), zs_d, cent_d, True, MARGIN)
        mask_pin.copy_(m, non_blocking=True)

    for _ in range(args.warmup):
        resident()
        e2e()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms = timed(resident, args.steps) / args.steps
    ms_e2e = timed(e2e, args.steps) / args.steps
    clocks = sampler.stop()
    torch.set_num_threads(usable_cpus())
    n_cpu = 2048
    with torch.inference_mode():
        t0 = time.perf_counter()
        O.cluster_min_dist_ratios(rays_h[:n_cpu], zs, cent, True)
        dt = time.perf_counter() - t0
    evals = n * S * 8
    sm_mhz = clocks.get('sm_mhz') or 1965.0
    peak = 148 * 128 * sm_mhz * 1e6 / 12.0
    line = {'metric': 'cluster-mask rays/sec (1000 samples x 8 centroids per ray)', 'value': n / (ms * 1e-3), 'unit': 'rays/s',
            'n_gpus': 1, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': f'create_cluster_masks.py default chunk: {n} rays x {S} samples, 2x4 centroid grid, cluster_2d, margin {MARGIN}',
                       'l2': f'flushed between timed iterations ({L2_FLUSH_BYTES >> 20} MiB write)'},
            'e2e': {'value': n / (ms_e2e * 1e-3), 'unit': 'rays/s', 'ms_per_step': ms_e2e, 'h2d_bytes_per_step': rays_pin.numel() * 4,
                    'd2h_bytes_per_step': mask_pin.numel()},
            'gpu_launches': args.steps, 'clocks': clocks,
            'roofline': {'bound': 'hbm', 'note': 'HBM traffic is ~2 MB per launch; the kernel is issue-bound (sqrt + div per distance)',
                         'achieved': (n * 32 + n * 8 * 5) / (ms * 1e-3) / 1e9, 'peak': peaks()['hbm'], 'unit': 'GB/s',
                         'frac': (n * 32 + n * 8 * 5) / (ms * 1e-3) / 1e9 / peaks()['hbm'], 'traffic': None,
                         'distance_evals_per_s': evals / (ms * 1e-3), 'issue_bound_estimate_evals_per_s': peak},
            'cpu_baseline': {'value': n_cpu / dt, 'unit': 'rays/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                             'sample': f'first {n_cpu} rays of the same chunk ({dt:.1f} s)'}}
    print(json.dumps(line), flush=True)


def main():
    import faulthandler
    faulthandler.dump_traceback_later(240, repeat=True, file=sys.stderr)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--precision', default=os.environ.get('MN_B200_PRECISION', 'tc_f16'))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-gpu-incumbent', action='store_true', help='skip timing the restatement under torch-CUDA eager')
    ap.add_argument('--workload', default=None, choices=sorted(WORKLOADS),
                    help="default: 'c2' (BASELINE configs[1], 4096 rays) on one GPU, 'c3' (configs[2]: 8192 rays per GPU) when N > 1")
    ap.add_argument('--no-graph', action='store_true', help='issue every step eagerly instead of replaying a CUDA graph')
    ap.add_argument('--margin', type=float, default=MARGIN, help='boundary_margin of the mixture: 1.15 = reference eval default (graded), '
                                                                 '1.0 = hard routing, m = 1 (SURVEY.md §8d)')
    ap.add_argument('--parallelism', default='rays', choices=['rays', 'experts'],
                    help="N > 1: 'rays' = ray-sharded with replicated weights (default, graded); 'experts' = additionally "
                         "owner-computes sub-modules (sub-module k on rank k mod N, two all-to-alls per model query; eager launches)")
    ap.add_argument('--gather', default='nccl', choices=['nccl', 'peer'],
                    help="N > 1: how the per-ray results are exchanged: 'nccl' = torch.cat + all_gather_into_tensor (default, graded); "
                         "'peer' = one kernel of ours storing into every rank's symmetric buffer over NVLink (mega_nerf_b200.dist.PeerGather)")
    ap.add_argument('--train-precision', default='tc_f16', choices=['fp32', 'tc_f16'], help="--mode train: arithmetic of the recording forward "
                    "and the backward pass ('fp32' = CUDA-core parity mode)")
    ap.add_argument('--mode', default='render', choices=['render', 'train', 'cluster'],
                    help="'render' = the graded line; 'train' = one optimisation step (forward + backward + Adam) of the same "
                         "workload through the recording path (SURVEY.md §8f-1); 'cluster' = the cluster-mask kernel on one "
                         "48k-ray chunk x 1000 samples (SURVEY.md §8f-3); both diagnostics only")
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='render mode: write the results of the last timed step (and, when N > 1, the all-gathered '
                         '[rays, 4] buffer) as DIR/<name>.npy in float32; the inputs are seeded, identical from run to run')
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != 'b200' or args.mode != 'render'):
        ap.error('--dump-outputs applies to the render mode of --impl b200')
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.workload is None:
        args.workload = 'c2' if max(world, args.gpus) == 1 else 'c3'
    select_workload(args.workload)
    globals()['MARGIN'] = args.margin
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.impl == 'reference':
        run_reference(args, rank)
        return
    if args.mode == 'train':
        run_train(args, rank, local_rank, world)
        return
    if args.mode == 'cluster':
        run_cluster(args, local_rank)
        return

    import torch.distributed as dist
    import mega_nerf_b200 as M
    from mega_nerf_b200 import _cabi as K
    from oracle import mn_oracle as O            # cpu_baseline / parity sample only
    from mega_nerf_b200.synthetic import build_net

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)

    spec, net, rays_h, idx_h, opts = workload(seed_shift=rank)
    hp = Namespace(**vars(opts))
    model = build_net(net, dev)
    M.set_precision(args.precision)
    experts = args.parallelism == 'experts' and world > 1
    if experts:
        from mega_nerf_b200 import expert_parallel as EP
        EP.enable(model)
        args.no_graph = True                      # host-sized all-to-alls are not graph-capturable
    rays_d, idx_d = rays_h.to(dev), idx_h.to(dev)
    rays_pin, idx_pin = rays_h.pin_memory(), idx_h.pin_memory()
    out_pin = torch.empty(N_RAYS, 4).pin_memory()
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    gather_buf = torch.empty(world * N_RAYS, 4, device=dev) if world > 1 else None
    pg = None
    if world > 1 and args.gather == 'peer':
        from mega_nerf_b200.dist import PeerGather
        pg = PeerGather(world * N_RAYS, dev)

    def exchange(res):
        """every rank ends up with all ranks' (rgb, depth) rows"""
        if world == 1:
            return
        if pg is not None:
            pg.gather(res['rgb_fine'], res['depth_fine'], rank * N_RAYS)
        else:
            dist.all_gather_into_tensor(gather_buf, torch.cat([res['rgb_fine'], res['depth_fine'].unsqueeze(-1)], -1))
    h = K.ctx(dev)
    L = K.lib()

    graphed = None      # the public CUDA-graph replay of render_rays (mega_nerf_b200/graph.py); set after the eager warm-up

    def step_eager():
        res, _ = M.render_rays(model, None, rays_d, idx_d, hp, None, None, True, False, False)
        exchange(res)
        return res

    def step_resident():
        if graphed is None:
            return step_eager()
        res = graphed(rays_d, idx_d)                 # device-resident inputs -> static buffers (D2D) -> graph replay
        if graphed.post is None:
            exchange(res)
        return res

    def step_e2e():
        if graphed is None:
            r = rays_pin.to(dev, non_blocking=True)
            i = idx_pin.to(dev, non_blocking=True)
            res, _ = M.render_rays(model, None, r, i, hp, None, None, True, False, False)
        else:
            res = graphed(rays_pin, idx_pin)         # pinned host inputs -> static device buffers (H2D) -> graph replay
        packed = torch.cat([res['rgb_fine'], res['depth_fine'].unsqueeze(-1)], -1)
        if world > 1 and not (graphed is not None and graphed.post is not None):
            if pg is not None:
                pg.gather(res['rgb_fine'], res['depth_fine'], rank * N_RAYS)
            else:
                dist.all_gather_into_tensor(gather_buf, packed)
        out_pin.copy_(packed, non_blocking=True)

    last = {}                                   # what the most recent timed step returned

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        for a, b in evs:
            flush.fill_(1)                      # L2 flush between timed iterations (not timed)
            a.record()
            last['out'] = fn()
            b.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    log('workload built; warm-up')
    for _ in range(args.warmup):
        step_resident()
        step_e2e()
    torch.cuda.synchronize()
    launches0 = L.mn_launch_count(h)
    step_eager()
    launches_per_step = L.mn_launch_count(h) - launches0      # kernels of ours per step (the graph replays the same list)
    if not args.no_graph:
        try:
            # the per-step exchange (pack + all-gather) is captured with the render: one graph launch per step at any N
            graphed = M.GraphedRenderRays(model, hp, N_RAYS, dev, with_indices=True, get_depth=True,
                                          post=exchange if (world > 1 and pg is None) else None)
            graphed.capture(rays_d, idx_d)
            for _ in range(args.warmup):
                step_resident()
                step_e2e()
            torch.cuda.synchronize()
        except Exception as e:  # noqa: BLE001
            log(f'CUDA graph capture failed ({e!r}); running eagerly')
            graphed = None
    log(f'warm-up done (cuda graph: {graphed is not None})')

    # ---- device-resident throughput (the `value`) with clocks sampled during the timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total = timed(step_resident, args.steps)
    if args.dump_outputs and rank == 0:
        # copied now: the next graph replay overwrites the static result buffers
        outs = dict(last['out'])
        if world > 1:
            outs['gathered'] = pg.buf if pg is not None else gather_buf
        dump_outputs(args.dump_outputs, outs)
    launches = launches_per_step * args.steps
    samples_per_step = N_RAYS * (COARSE + FINE) * world
    value = samples_per_step * args.steps / (ms_total * 1e-3)

    log(f'resident: {ms_total / args.steps:.3f} ms/step')
    # ---- end to end through the public API from pinned host memory
    ms_e2e = timed(step_e2e, args.steps)
    e2e_value = samples_per_step * args.steps / (ms_e2e * 1e-3)

    log(f'e2e: {ms_e2e / args.steps:.3f} ms/step')
    # ---- MLP kernel duration by CUDA events on the launching stream (roofline)
    nat = model._native()
    K.check(L.mn_profile_enable(h, 1), h)
    timed(step_eager, args.steps)
    tot_ms, n_l = C.c_double(), C.c_longlong()
    K.check(L.mn_profile_read(h, C.byref(tot_ms), C.byref(n_l)), h)
    K.check(L.mn_profile_enable(h, 0), h)
    clocks = sampler.stop() if rank == 0 else None      # sampled over the resident, e2e and kernel-timing sections

    def pairs_of_last_query():
        # routed (sample, sub-module) pairs of the most recent model query, read back from the device counters
        return model._ep.last_pairs if experts else nat.stats(dev)[0]
    pairs_fine = pairs_of_last_query()                    # the last query of a step is the fine pass
    # the coarse pass of the two-pass render issues exactly the query of a coarse-only render of the same rays
    hp_coarse = Namespace(**{**vars(hp), 'fine_samples': 0})
    with torch.no_grad():
        M.render_rays(model, None, rays_d, idx_d, hp_coarse, None, None, True, False, False)
    pairs_coarse = pairs_of_last_query()
    m_coarse, m_fine = pairs_coarse / (N_RAYS * COARSE), pairs_fine / (N_RAYS * FINE)
    mult = (pairs_coarse + pairs_fine) / (N_RAYS * (COARSE + FINE))
    pk = peaks()
    fl_row = flops_per_row(spec)
    # per step: coarse + fine launches; algorithmic flops = routed pairs of BOTH passes (each measured) * flops_row
    flops_step = (pairs_coarse + pairs_fine) * fl_row
    kernel_ms_per_step = tot_ms.value / args.steps
    achieved = flops_step / (kernel_ms_per_step * 1e-3) / 1e12 if kernel_ms_per_step > 0 else 0.0
    passes = {'fp32': 1, 'tc_f16': 1, 'tc_f16x3': 3}[args.precision]
    kernel_name = {'fp32': 'mlp_simt_kernel', 'tc_f16': WL['kernel'], 'tc_f16x3': 'tc_mlp_kernel<split>'}[args.precision]
    if kernel_name == 'tc_mlp_tp_kernel' and os.environ.get('MN_TC_TP', '1') == '0':
        kernel_name = 'tc_mlp_pp_kernel'          # A/B switch of libmn_b200.so: the shared-memory ping-pong kernel
    traffic = kernel_traffic(kernel_name, args.workload if world == 1 else 'c3', args.precision)

    log(f'mlp kernel: {kernel_ms_per_step:.3f} ms/step, m={mult:.3f}')
    # ---- parity against the CPU checker (not timed).  Every rank checks (a) the first N_PAR of its own rays through the
    # single-GPU call and, when N > 1, (b) its OWN copy of the gathered buffer: the rows of its own segment and of its right
    # neighbour's segment (that rank's seeded rays are regenerated here); the maxima are all-reduced.
    N_PAR = 128
    torch.set_num_threads(max(1, usable_cpus() // max(1, min(world, 8))))

    def check_rows(rays_c, idx_c):
        with torch.inference_mode():
            ref, _ = O.render_rays(net, None, rays_c, idx_c, opts, None, None, True, False, False)
        return ref['rgb_fine'], ref['depth_fine']

    def rel(a, b):
        return float((a.double().cpu() - b.double()).abs().max() / b.double().abs().max())
    ref_rgb, ref_depth = check_rows(rays_h[:N_PAR], idx_h[:N_PAR])
    with torch.no_grad():
        got, _ = M.render_rays(model, None, rays_d[:N_PAR], idx_d[:N_PAR], hp, None, None, True, False, False)
    par_rgb, par_depth = rel(got['rgb_fine'], ref_rgb), rel(got['depth_fine'], ref_depth)
    par_g_rgb = par_g_depth = None
    if world > 1:
        step_resident()                                     # one more exchange: every rank holds the buffer of THESE inputs
        torch.cuda.synchronize()
        gbuf = (pg.buf if pg is not None else gather_buf).cpu()
        nb = (rank + 1) % world
        _, _, rays_nb, idx_nb, _ = workload(seed_shift=nb)
        nb_rgb, nb_depth = check_rows(rays_nb[:N_PAR], idx_nb[:N_PAR])
        own, oth = gbuf[rank * N_RAYS: rank * N_RAYS + N_PAR], gbuf[nb * N_RAYS: nb * N_RAYS + N_PAR]
        t = torch.tensor([max(rel(own[:, :3], ref_rgb), rel(oth[:, :3], nb_rgb)),
                          max(rel(own[:, 3], ref_depth), rel(oth[:, 3], nb_depth)), par_rgb, par_depth],
                         device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        par_g_rgb, par_g_depth, par_rgb, par_depth = [float(v) for v in t.tolist()]
    if experts:
        EP.disable(model)
    if rank == 0:
        log(f'parity: rgb {par_rgb:.2e} depth {par_depth:.2e}' + (f' gathered rgb {par_g_rgb:.2e} depth {par_g_depth:.2e}' if world > 1 else ''))
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            # the reference algorithm's CPU path (oracle port) on a bounded sample of the same batch
            torch.set_num_threads(usable_cpus())
            render_cpu, cpu_kind = cpu_renderer(O, net, opts)
            rate = cpu_rays_per_sec(render_cpu, rays_h, idx_h)
            n_cpu = int(min(N_RAYS, max(64, rate * 15.0))) // 64 * 64         # ~15 s of CPU work
            with torch.inference_mode():
                t0 = time.perf_counter()
                render_cpu(rays_h[:n_cpu], idx_h[:n_cpu])
                dt = time.perf_counter() - t0
            cpu = {'value': n_cpu * (COARSE + FINE) / dt, 'unit': 'samples/s', 'cores': torch.get_num_threads(),
                   'kind': cpu_kind, 'sample': f'first {n_cpu} of the {N_RAYS} rays of the same batch ({dt:.1f} s), after a 64-ray probe'}
            log(f'cpu baseline ({cpu_kind}): {cpu["value"]:.3e} samples/s on {cpu["cores"]} threads')

        line = {
            'metric': 'ray-samples/sec (MLP+composite)', 'value': value, 'unit': 'samples/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_total / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': {'fp32': 'f32', 'tc_f16': 'f16 operands / f32 accumulate', 'tc_f16x3': 'f16x3 split / f32 accumulate'}[args.precision],
            'data': 'synthetic',
            'config': {'workload': workload_string(),
                       'per_gpu_rays': N_RAYS,
                       'sub_modules_per_sample': {'coarse_pass': m_coarse, 'fine_pass': m_fine, 'step': mult,
                                                  'how': 'routed (sample, sub-module) pairs of each pass read back from the device counters'},
                       'parallelism': (f'ray-sharded x{world} + owner-computes sub-modules (k mod {world}), 2 all-to-alls per query, '
                                       f'1 all-gather of [rays,4] per step' if experts else
                                       f'ray-sharded x{world}, weights replicated, 1 all-gather of [rays,4] per step'
                                       + (' as peer-memory stores (PeerGather)' if pg is not None else '')) if world > 1 else 'single GPU',
                       'precision': args.precision,
                       'launch': 'one CUDA graph replay per step (mega_nerf_b200.GraphedRenderRays)' if graphed is not None else 'eager launches',
                       'l2': f'flushed between timed iterations ({L2_FLUSH_BYTES >> 20} MiB write)',
                       'rays_per_sec': value / (COARSE + FINE)},
            'e2e': {'value': e2e_value, 'unit': 'samples/s', 'ms_per_step': ms_e2e / args.steps,
                    'h2d_bytes_per_step': rays_pin.numel() * 4 + idx_pin.numel() * 4, 'd2h_bytes_per_step': out_pin.numel() * 4},
            'gpu_launches': int(launches),
            'clocks': clocks,
            'roofline': {'bound': 'tensor',
                         'kernel': kernel_name,
                         'achieved': achieved, 'peak': pk['tflops'], 'unit': 'TFLOP/s', 'frac': achieved / pk['tflops'],
                         'frac_of_sustained_peak': achieved / pk['tflops_sustained'] if pk['tflops_sustained'] else None,
                         'peak_source': pk['src'],
                         # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel on this workload, from the committed
                         # `ncu --set full` capture (profiles/kernel_traffic.json, written by scripts/ncu_extract.py from the
                         # .ncu-rep next to it); null when no capture of this (kernel, workload, precision) is committed
                         'traffic': traffic['dram_bytes'] if traffic else None,
                         'traffic_detail': traffic,
                         'algorithmic_flops_per_row': fl_row, 'mma_passes_per_algorithmic': passes,
                         'kernel_ms_per_step': kernel_ms_per_step, 'launches_per_step': n_l.value / args.steps},
            'parity': {'max_rel_rgb_vs_oracle': par_rgb, 'max_rel_depth_vs_oracle': par_depth, 'rays_checked_per_rank': N_PAR,
                       'max_rel_rgb_gathered': par_g_rgb, 'max_rel_depth_gathered': par_g_depth,
                       'gathered_check': (f'every rank compares its own copy of the all-gathered [rays,4] buffer (own segment + right '
                                          f"neighbour's segment, {N_PAR} rays each) with the CPU oracle; max over the {world} ranks")
                       if world > 1 else None,
                       'tolerance': 1e-4, 'pass': bool(max(par_rgb, par_g_rgb or 0.0) <= 1e-4),
                       'note': ('tc_f16 rounds both MMA operands to fp16 (what the reference itself does on a GPU under autocast): rendered '
                                'rgb passes the 1e-4 north-star tolerance on this random-init workload with ~2x headroom; tc_f16x3 '
                                '(3 MMA passes, <= 1e-5 per MLP row) is the parity-grade tensor mode, fp32 the CUDA-core one')
                       if args.precision == 'tc_f16' else None},
        }
        if cpu is not None:
            line['cpu_baseline'] = cpu
        if world == 1 and not args.no_gpu_incumbent:
            line['gpu_incumbent'] = gpu_incumbent(O, net, rays_d, idx_d, opts, dev)
            log(f'gpu incumbent: {line["gpu_incumbent"]}')
        print(json.dumps(line), flush=True)
    if world > 1:
        # The per-step all-gather lives inside a captured CUDA graph; tearing the NCCL communicator down while graphs that
        # reference it are alive blocked in destroy_process_group() for minutes on the 2-GPU box.  Drop the graph, drain the
        # device, agree that everybody is done, then leave without the collective teardown (the line is already printed).
        graphed = None
        import gc
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == '__main__':
    main()
