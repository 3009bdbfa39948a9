#!/usr/bin/env python
"""Stamps/s of the two shape estimators on one GPU, how the adaptive one ends, and (as context) how well each recovers the
true shapes after a Wiener deconvolution.

  adaptive_moments   gdeconv.adaptive_moments: k_adaptive_moments (csrc/shape.cu), one warp per stamp
  moments_e          gdeconv.moments_e: k_moments, min-max normalised unweighted moments (the training-loss metric)
  torch_reference    oracle/adaptive_moments.py in fp32 on the same GPU, in --piece-stamp pieces: the library-free baseline

Workloads: --stamps gt stamps and --stamps SNR-100 obs stamps from gdeconv.make_batch_device (9.2 GB each for 1,000,000 stamps,
far beyond the L2).  Each arm is warmed up on its workload, then passes over the whole workload repeat until the CUDA-event window
reaches --min-seconds.  For each workload: the mean number of passes and the count of each status of gd_adaptive_moments.
Context, not a gate: on --wiener-stamps SNR-100 stamps deconvolved with the (weight-free) Wiener filter, the median and 90th
percentile of |e - e_gt| for both estimators (adaptive: stamps OK in both measurements).  The card's name and power limit are
read in the same run.

    python tools/shape_bench.py [--stamps 1000000] [--wiener-stamps 100000] [--piece-stamps 100000] [--min-seconds 1]

Prints one JSON line.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, 'galaxy-deconv_b200'), ROOT, os.path.join(ROOT, 'tools')]

import torch  # noqa: E402

from synth_bench import card, rate  # noqa: E402

STATUS = ('OK', 'MAXITER', 'FLUX', 'MOMENTS', 'CENTROID')


def pieces(fn, x, piece):
    """fn over x in pieces of `piece` stamps; the results are dropped once the piece is done, as a caller of the reference would"""
    for i in range(0, x.shape[0], piece):
        fn(x[i:i + piece])


def workload(name, x, args):
    from gdeconv import adaptive_moments, moments_e
    from oracle.adaptive_moments import adaptive_moments as reference
    n = x.shape[0]
    res = adaptive_moments(x)
    counts = torch.bincount(res['status'].long(), minlength=len(STATUS)).tolist()
    row = dict(workload=name, stamps=n, mean_passes=float(res['n_iter'].double().mean()), status_counts=dict(zip(STATUS, counts)))
    del res
    row['adaptive_moments'] = rate(lambda: adaptive_moments(x), n, args.min_seconds)
    row['moments_e'] = rate(lambda: moments_e(x), n, args.min_seconds)
    row['torch_reference'] = rate(lambda: pieces(reference, x, args.piece_stamps), n, args.min_seconds)
    torch.cuda.empty_cache()
    row['speedup_vs_torch_reference'] = row['adaptive_moments']['stamps_per_s'] / row['torch_reference']['stamps_per_s']
    return row


def wiener_context(n):
    from gdeconv import adaptive_moments, make_batch_device, moments_e
    from models.Wiener import Wiener
    b = make_batch_device(0, n, 100.0)
    w = Wiener()(b['obs'], b['psf'], b['alpha'])
    q = lambda d: dict(median=float(d.median()), p90=float(d.quantile(0.9)), stamps=int(d.numel()))
    de_mom = (moments_e(w) - moments_e(b['gt'])).norm(dim=1).double().cpu()
    a_w, a_gt = adaptive_moments(w), adaptive_moments(b['gt'])
    both = (a_w['status'] == 0) & (a_gt['status'] == 0)
    de_ad = (a_w['e'][both] - a_gt['e'][both]).norm(dim=1).double().cpu()
    return dict(stamps=n, snr=100.0, moments_e=q(de_mom), adaptive_moments=q(de_ad))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--stamps', type=int, default=1_000_000)
    ap.add_argument('--wiener-stamps', type=int, default=100_000)
    ap.add_argument('--piece-stamps', type=int, default=100_000)
    ap.add_argument('--min-seconds', type=float, default=1.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('shape_bench needs a CUDA device')
    from gdeconv import make_batch_device
    dev = torch.device('cuda', torch.cuda.current_device())
    t0 = time.time()
    rows = []
    for key, name in (('gt', 'gt (noise-free galaxies)'), ('obs', 'obs, SNR 100')):
        x = make_batch_device(0, args.stamps, 100.0, device=dev, keys=(key,))[key]
        rows.append(workload(name, x, args))
        del x
        torch.cuda.empty_cache()
    print(json.dumps(dict(metric='shape measurements stamps/s', card=card(dev), torch=torch.__version__, torch_reference_piece=args.piece_stamps,
                          rows=rows, wiener_context=wiener_context(args.wiener_stamps), wall_seconds=time.time() - t0)))


if __name__ == '__main__':
    main()
