#!/usr/bin/env python
"""Headline benchmark: galaxies/s of Unrolled-ADMM(8) (UnrolledADMMGaussian, ResUNet nc 32..256) on 48x48 stamps.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--stamps S] [--n-iters 8]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic stamps per GPU (BASELINE.json configs[1]: 10,000
synthetic 48x48 stamps at SNR 100, the test.py --n_gal 10000 shape): model(obs, psf, alpha) through the
reference-shaped nn.Module -> C ABI -> sm_100a kernels, followed by the per-galaxy moment ellipticities and (N > 1)
their NCCL all-gather.  Weak scaling: every rank processes its own `stamps` galaxies per step, no data-path collective.

Printed JSON (rank 0, one line): `value` = whole-job galaxies/s with inputs resident in HBM; `e2e` = the same call with
pinned HOST inputs (H2D of obs/psf/alpha and D2H of the deconvolved stamps + ellipticities inside the timed region);
`roofline` = the dominant kernel family (k_conv_umma and the chain kernels k_l1_chain / k_l2_chain, tcgen05 tap-GEMM) timed live per launch with CUDA events, algorithmic
FLOPs / time against the measured bf16 peak of MEASURED_PEAKS.json; `cpu_baseline` = the CPU oracle (bit-exact port of
the reference's torch code) timed on this box's host cores on a bounded sample.

--impl reference: times the reference's own CPU implementation of the path (the oracle port; /root/reference does not
exist on the GPU box) on the host cores with all threads; rank 0 only.  It imports only torch, the oracle and the
torch-only generator module gdsynth: libgdeconv.so is never mapped in that process.

--dump-outputs DIR: after the timed steps, write what the last timed step of the headline path computed, as float32 .npy
files: DIR/deconvolved.npy (rank 0's deconvolved stamps [S,1,48,48]) and DIR/ellipticities.npy (the gathered moment
ellipticities [S,2]).  Arrays longer than 4096 stamps / 2^21 galaxies are cut to a fixed seeded sample of that many rows in
index order (at most 55 MB in all).  Inputs and weights are seeded, so two builds run with the same arguments can be compared
file for file.

--config 3|4|5 run the other BASELINE.json configs (one JSON line per measurement; the default line, config 2, is unchanged):
  3  Unrolled-ADMM(8) on --total (1,000,000) stamps, STRONG scaling: the total is sharded by galaxy over the ranks, every shard
     is generated on its own GPU, and one step = forward over the whole shard + moment ellipticities + NCCL all-gather;
  4  Richardson-Lucy(10/50/100), Wiener, Tikhonov-Laplacian and Tikhonet_Laplacian on --total stamps, sharded the same way;
  5  PSF-mismatch sweep (test_psf.py:237-242 shape): 10 shear + 10 seeing errors x --sweep-stamps (100,000) stamps, sharded.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.join(ROOT, 'galaxy-deconv_b200'), ROOT, os.path.join(ROOT, 'tools')]

import torch  # noqa: E402

STAMP_BYTES_IN = 2 * 48 * 48 * 4 + 4
STAMP_BYTES_OUT = 48 * 48 * 4 + 8


def flops_per_stamp_g(n):
    """SURVEY.md section 8d: F_G(n) = n*1,248,362,496 + 5,742,720 + 128*n (conv + linear MACs*2; FFTs excluded)."""
    return n * 1248362496 + 5742720 + 128 * n


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        p = json.load(open(path))
        return dict(hbm=p['hbm_gbs'], tensor_burst=p['bf16_tflops'], tensor_sustained=p.get('bf16_tflops_sustained', p['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    except Exception:
        return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.rows.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            f = [c.strip() for c in r.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx or None, reasons=sorted(reasons), samples=len(sm))


def seeded_rows(t, k, seed=0):
    """t itself if it has at most k rows, else k of its rows picked by a fixed seed, in index order."""
    if t.shape[0] <= k:
        return t
    idx = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(seed))[:k].sort().values
    return t[idx.to(t.device)]


def cpu_reference(n_iters, sample, batch, steps, warmup):
    """The reference's CPU implementation of the path (oracle port, bit-exact vs the reference) on the host cores."""
    import oracle.ref_models as O
    from gdsynth import make_batch            # torch-only module: the reference arm never loads libgdeconv.so
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    m = O.UnrolledADMMGaussian(n_iters).eval()
    m.load_state_dict(O.seeded_state_dict(lambda: O.UnrolledADMMGaussian(n_iters), 12))
    b = make_batch(0, sample, 100.0)
    times = []
    with torch.no_grad():
        for s in range(warmup + steps):
            t0 = time.perf_counter()
            for i in range(0, sample, batch):
                m(b['obs'][i:i + batch], b['psf'][i:i + batch], b['alpha'][i:i + batch])
            if s >= warmup:
                times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return dict(value=sample / dt, unit='galaxies/s', cores=cores, kind='port',
                sample=f'{sample} synthetic stamps (SNR 100), batch {batch}, {steps} timed pass(es), torch {torch.__version__} CPU, {cores} threads',
                ms_per_step=dt * 1e3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--stamps', type=int, default=10000, help='stamps per GPU per step')
    ap.add_argument('--n-iters', type=int, default=8)
    ap.add_argument('--precision', default=None)
    ap.add_argument('--cpu-sample', type=int, default=512, help='stamps per pass of the cpu_baseline leg (BASELINE.md section 3: N = 512)')
    ap.add_argument('--config', type=int, default=2, choices=[2, 3, 4, 5], help='BASELINE.json configs index (2 = headline)')
    ap.add_argument('--total', type=int, default=1000000, help='configs 3/4: total stamps over all ranks')
    ap.add_argument('--sweep-stamps', type=int, default=100000, help='config 5: stamps per sweep point over all ranks')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or args.config != 2):
        ap.error('--dump-outputs covers the headline path only (--impl b200, --config 2)')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    metric = f'galaxies/sec Unrolled-ADMM({args.n_iters}) 48x48'
    cfg = dict(workload=f'UnrolledADMMGaussian({args.n_iters}) on {args.stamps} synthetic 48x48 stamps (SNR 100, Moffat PSF) per GPU per step '
                        f'(BASELINE configs[1], test.py --n_gal 10000 shape), seeded random weights',
               stamps_per_gpu=args.stamps, n_iters=args.n_iters, parallelism=f'galaxy-sharded x{world}',
               l2='inputs+outputs of a step (%.0f MB) exceed the 126 MB L2' % (args.stamps * (STAMP_BYTES_IN + STAMP_BYTES_OUT) / 1e6))

    if args.impl == 'reference':
        if rank != 0:
            return
        # a step = one pass over a bounded sample of the workload, sized so that steps + warm-up stay within ~2 minutes
        per_step = max(64, min(512, int(15000 / max(1, args.steps + args.warmup)) // 64 * 64))
        r = cpu_reference(args.n_iters, per_step, 64, max(1, args.steps), max(0, args.warmup))
        print(json.dumps(dict(metric=metric, value=r['value'], unit='galaxies/s', n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                              ms_per_step=r['ms_per_step'], higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
                              data='synthetic', impl='reference', config=cfg,
                              cpu_baseline={k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
                              e2e=dict(value=r['value'], unit='galaxies/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))))
        return

    import torch.distributed as dist
    from gdeconv import engine, moments_e
    from gdeconv._lib import lib
    from gdeconv.shard import gather_ellipticities, shard_range
    from gdsynth import make_batch
    from models.unrolled_admm_gaussian import UnrolledADMMGaussian
    import oracle.ref_models as O          # only for the seeded weights and the cpu_baseline leg

    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU path)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    if args.precision:
        os.environ['GDECONV_PRECISION'] = args.precision
    precision = engine.default_precision()

    model = UnrolledADMMGaussian(args.n_iters).eval()
    model.load_state_dict(O.seeded_state_dict(lambda: O.UnrolledADMMGaussian(args.n_iters), 12))
    model = model.to(dev)
    if args.config != 2:
        from bench_configs import run_config
        run_config(args, model, dev, rank, world, peaks())
        if world > 1:
            dist.destroy_process_group()
        return
    n_total = args.stamps * world
    lo, hi = shard_range(n_total, rank, world)
    data = make_batch(lo, hi - lo, 100.0, device=dev)
    obs, psf, alpha = data['obs'], data['psf'], data['alpha']
    host = {k: data[k].cpu().pin_memory() for k in ('obs', 'psf', 'alpha')}
    out_host = torch.empty(hi - lo, 1, 48, 48).pin_memory()
    e_host = torch.empty(n_total, 2).pin_memory()

    def step_device():
        out = model(obs, psf, alpha)
        return out, gather_ellipticities(moments_e(out), n_total)

    def step_e2e():
        # the public host-batch call: chunk-pipelined H2D / compute / D2H inside the engine (one cudaMemcpyAsync per tensor and
        # chunk on two copy streams), then the ellipticity gather and its D2H
        _, e_loc = model.deconvolve_host(host['obs'], host['psf'], host['alpha'], out=out_host, want_e=True, device=dev)
        e = gather_ellipticities(e_loc, n_total)
        e_host.copy_(e, non_blocking=True)

    def timed(fn, steps, warmup):
        """-> (ms per step, launches in the timed steps, what the last timed step returned).  The warm-up keeps each step's
        result alive through the next step exactly like the timed loop, so the allocator holds both before timing starts."""
        last = None
        for _ in range(warmup):
            last = fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l0 = lib.gd_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = fn()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps, int(lib.gd_launch_count() - l0), last

    with ClockSampler(local) as clk:
        ms_step, launches, (out_last, e_last) = timed(step_device, args.steps, max(3, args.warmup))
    clocks = clk.summary()
    dump = None
    if args.dump_outputs and rank == 0:
        dump = dict(deconvolved=seeded_rows(out_last, 4096).float().cpu(), ellipticities=seeded_rows(e_last, 1 << 21).float().cpu())
    del out_last, e_last
    ms_e2e, _, _ = timed(step_e2e, args.steps, max(3, args.warmup))

    # dominant kernel, live: every k_conv_umma / k_rb_umma launch of one more step bracketed by CUDA events on its stream
    roof = None
    P = peaks()
    if precision == 'fp16_umma':
        # (chunks run back to back on ONE stream for this step, so that each launch's events bracket that kernel alone)
        torch.cuda.synchronize()
        streams_env = os.environ.get('GDECONV_STREAMS')
        os.environ['GDECONV_STREAMS'] = '1'
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        lib.gd_profile_begin()
        p0.record()
        step_device()
        p1.record()
        ms_k, fl_k, n_k = C.c_double(), C.c_double(), C.c_uint64()
        lib.gd_profile_end(C.byref(ms_k), C.byref(fl_k), C.byref(n_k))
        torch.cuda.synchronize()
        ms_profile_step = p0.elapsed_time(p1)
        if streams_env is None:
            del os.environ['GDECONV_STREAMS']
        else:
            os.environ['GDECONV_STREAMS'] = streams_env
        if ms_k.value > 0:
            ach = fl_k.value / (ms_k.value * 1e-3) / 1e12
            traffic, traffic_note = None, 'no ncu capture found under profiles/'
            try:        # DRAM bytes per launch from the committed ncu capture of the same kernel (per launch, like `achieved`)
                tpath = next(q for q in (os.path.join(ROOT, 'profiles', f) for f in ('roofline_traffic_r02.json', 'roofline_traffic_r01.json')) if os.path.exists(q))
                tj = json.load(open(tpath))
                per_chunk = engine._chunk_for(hi - lo)
                traffic = tj['avg_traffic_bytes_per_launch'] * min(per_chunk, hi - lo) / tj['stamps_per_launch']
                traffic_note = 'ncu dram__bytes_read+write per tcgen05 conv launch (profiles/%s), scaled by stamps per launch' % os.path.basename(tpath)
            except Exception:
                pass
            roof = dict(bound='tensor', achieved=ach, peak=P['tensor_sustained'], unit='TFLOP/s', frac=ach / P['tensor_sustained'], traffic=traffic,
                        traffic_note=traffic_note,
                        kernel='k_conv_umma + k_l1_chain + k_l2_chain (tcgen05 tap-GEMM convolutions; the chain kernels run 4-5 convs per launch)', launches_per_step=int(n_k.value), avg_launch_us=ms_k.value * 1e3 / max(1, n_k.value),
                        kernel_share_of_step=ms_k.value / ms_profile_step, profiled_step_ms=ms_profile_step, flops_per_launch_avg=fl_k.value / max(1, n_k.value),
                        peak_source=P['source'] + ', sustained bf16 (kernel timed inside a long step); burst = %.1f' % P['tensor_burst'])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    gal_s = n_total / (ms_step * 1e-3)
    F = flops_per_stamp_g(args.n_iters)
    line = dict(metric=metric, value=gal_s, unit='galaxies/s', n_gpus=world, steps=args.steps, warmup=max(3, args.warmup), ms_per_step=ms_step,
                higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f16' if precision.startswith('fp16') else 'f32',
                data='synthetic', config=dict(cfg, precision=precision, chunk=engine._chunk_for(hi - lo), streams=engine.n_streams()),
                e2e=dict(value=n_total / (ms_e2e * 1e-3), unit='galaxies/s', h2d_bytes_per_step=(hi - lo) * STAMP_BYTES_IN,
                         d2h_bytes_per_step=(hi - lo) * 48 * 48 * 4 + n_total * 8, ms_per_step=ms_e2e),
                gpu_launches=launches, clocks=clocks,
                whole_step_roofline=dict(flops_per_stamp=F, achieved_tflops=gal_s * F / 1e12 / world, frac_of_sustained=gal_s * F / 1e12 / world / P['tensor_sustained'],
                                         frac_of_burst=gal_s * F / 1e12 / world / P['tensor_burst'], hbm_bytes_per_stamp=27652))
    if roof:
        line['roofline'] = roof
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference(args.n_iters, args.cpu_sample, 64, 3, 1)
        line['cpu_baseline'] = {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')}
    if dump:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in dump.items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), t.numpy())
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
