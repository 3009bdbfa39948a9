#!/usr/bin/env python
"""Stamps/s of the two synthetic-stamp generators on one GPU, and how closely they agree.

  torch   gdsynth.make_batch on the device in 20,000-stamp pieces copied into one output per key: tools/bench_configs.py
          _make_shard, which is how configs 3, 4 and 5 generate their inputs
  device  gdeconv.make_batch_device: one fused kernel (k_synth, csrc/synth.cu) writing the outputs directly

Workloads: all four keys for --stamps stamps (configs 3 / 4), and the mismatched model PSF alone with psf_shear_err=0.03
for --psf-stamps stamps (one config-5 sweep point).  Each arm is warmed up on its workload, then passes over the whole
workload repeat until the window reaches --min-seconds; the time is read from CUDA events.  The outputs (up to 37 GB for
1,000,000 stamps) are far larger than the L2.  Parity: make_batch_device against gdsynth.make_batch on the CPU, the fp32
reference of tests/test_synth_device.py, on --parity stamps: max per-stamp rel-L2 of obs / psf / gt, and the max alpha
deviation over max(|alpha|, RMS(obs)).  The card's name and power limit are read in the same run.

    python tools/synth_bench.py [--stamps 1000000] [--psf-stamps 100000] [--parity 4096] [--min-seconds 1]

Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, 'galaxy-deconv_b200'), ROOT, os.path.join(ROOT, 'tools')]

import torch  # noqa: E402


def card(dev):
    info = dict(name=torch.cuda.get_device_name(dev), power_limit_w=None, max_sm_clock_mhz=None)
    try:
        out = subprocess.run(['nvidia-smi', '-i', str(dev.index), '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader,nounits'],
                             capture_output=True, text=True, timeout=60).stdout.strip().split(',')
        info.update(name=out[0].strip(), power_limit_w=float(out[1]), max_sm_clock_mhz=float(out[2]))
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return info


def rate(fn, n, min_seconds):
    """stamps/s of fn() generating n stamps: one warm-up pass, then whole passes until the CUDA-event window is >= min_seconds."""
    out = fn()
    del out
    torch.cuda.synchronize()
    passes, ms = 0, 0.0
    while ms < min_seconds * 1e3:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        del out
        ms += e0.elapsed_time(e1)
        passes += 1
    return dict(stamps_per_s=passes * n / (ms * 1e-3), seconds=ms * 1e-3, passes=passes)


def compare(workload, n, torch_fn, device_fn, min_seconds):
    t = rate(torch_fn, n, min_seconds)
    torch.cuda.empty_cache()
    d = rate(device_fn, n, min_seconds)
    torch.cuda.empty_cache()
    return dict(workload=workload, stamps=n, torch=t, device=d, speedup=d['stamps_per_s'] / t['stamps_per_s'])


def rel_l2(a, b):
    """per-stamp relative L2 error of a against the reference b"""
    a, b = a.double().flatten(1), b.double().flatten(1)
    return (a - b).norm(dim=1) / b.norm(dim=1).clamp_min(1e-30)


def parity(n):
    import gdsynth
    from gdeconv import make_batch_device
    res = {}
    for name, kw in (('snr100', dict(snr=100.0)), ('mixed_shear0.03', dict(snr='mixed', psf_shear_err=0.03))):
        ref = gdsynth.make_batch(0, n, **kw)
        got = {k: v.cpu() for k, v in make_batch_device(0, n, **kw).items()}
        a_ref = ref['alpha'].flatten()
        rms = ref['obs'].flatten(1).pow(2).mean(1).sqrt()
        res[name] = dict({k: float(rel_l2(got[k], ref[k]).max()) for k in ('obs', 'psf', 'gt')},
                         alpha=float(((got['alpha'].flatten() - a_ref).abs() / torch.maximum(a_ref.abs(), rms)).max()))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--stamps', type=int, default=1_000_000)
    ap.add_argument('--psf-stamps', type=int, default=100_000)
    ap.add_argument('--parity', type=int, default=4096)
    ap.add_argument('--min-seconds', type=float, default=1.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('synth_bench needs a CUDA device')
    from bench_configs import PIECE, _make_shard
    from gdeconv import make_batch_device
    dev = torch.device('cuda', torch.cuda.current_device())
    t0 = time.time()
    keys = ('obs', 'psf', 'alpha', 'gt')
    rows = [compare('all keys (obs, psf, alpha, gt), SNR 100', args.stamps,
                    lambda: _make_shard(0, args.stamps, dev, keys=keys), lambda: make_batch_device(0, args.stamps, 100.0, device=dev),
                    args.min_seconds),
            compare('model PSF only, psf_shear_err=0.03', args.psf_stamps,
                    lambda: _make_shard(0, args.psf_stamps, dev, keys=('psf',), psf_shear_err=0.03),
                    lambda: make_batch_device(0, args.psf_stamps, 100.0, device=dev, psf_shear_err=0.03, keys=('psf',)),
                    args.min_seconds)]
    print(json.dumps(dict(metric='synthetic stamps/s', card=card(dev), torch=torch.__version__, torch_piece=PIECE, rows=rows,
                          parity_vs_cpu_reference=dict(stamps=args.parity, **parity(args.parity)), wall_seconds=time.time() - t0)))


if __name__ == '__main__':
    main()
