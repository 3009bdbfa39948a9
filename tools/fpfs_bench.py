#!/usr/bin/env python
"""Stamps/s of FPFS shear estimation on one GPU, and (as context) the reference's SNR table of shear errors in its own shape.

  device           gdeconv.fpfs: k_fpfs (csrc/fpfs.cu), without a PSF (one 2-D transform per stamp) and with a per-stamp PSF (two)
  torch_reference  oracle/fpfs.py in fp32 on the same GPU, in --piece-stamps pieces: the library-free baseline

Workload: --stamps SNR-100 obs stamps and their PSFs from gdeconv.make_batch_device (9.2 GB each for 1,000,000 stamps, far
beyond the L2).  Each arm is warmed up on its workload, then passes over the whole workload repeat until the CUDA-event window
reaches --min-seconds.  Compulsory traffic: 9,252 B per stamp without a PSF (the image read, 9 result floats written), 18,468 B
with one.

SNR table (context, not a gate): for each SNR, --table-stamps stamps from make_batch_device; the median over stamps of
|g - g_gt| (the norm of the two-component difference of the per-galaxy shears e / R, sigma 3.5, const 0), where g_gt is gt
measured with no PSF, for No_Deconv (obs, no PSF), FPFS (obs, its true PSF), Wiener, Tikhonov-Laplacian (lam 1) and RL(10)
(their outputs, no PSF), as the reference's evaluation does (test.py:67-87).  The learned models are left out: their weights
here are seeded, not trained.  Stamps with a NaN shear are counted and left out of the median.  The card's name and power
limit are read in the same run.

    python tools/fpfs_bench.py [--stamps 1000000] [--piece-stamps 100000] [--table-stamps 10000] [--min-seconds 1]

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

SNRS = (20, 40, 60, 80, 100, 150, 200, 300)
BYTES = {False: 2304 * 4 + 9 * 4, True: 2 * 2304 * 4 + 9 * 4}


def pieces(fn, x, psf, piece):
    for i in range(0, x.shape[0], piece):
        fn(x[i:i + piece], None if psf is None else psf[i:i + piece])


def throughput(args, dev):
    from gdeconv import fpfs, make_batch_device
    from oracle.fpfs import fpfs as reference
    b = make_batch_device(0, args.stamps, 100.0, device=dev, keys=('obs', 'psf'))
    rows = []
    for with_psf in (False, True):
        x, p = b['obs'], b['psf'] if with_psf else None
        row = dict(workload=f"obs, SNR 100, {'per-stamp PSF' if with_psf else 'no PSF'}", stamps=args.stamps, bytes_per_stamp=BYTES[with_psf])
        row['device'] = rate(lambda: fpfs(x, p), args.stamps, args.min_seconds)
        row['device']['achieved_TBps'] = row['device']['stamps_per_s'] * BYTES[with_psf] / 1e12
        row['torch_reference'] = rate(lambda: pieces(reference, x, p, args.piece_stamps), args.stamps, args.min_seconds)
        torch.cuda.empty_cache()
        row['speedup_vs_torch_reference'] = row['device']['stamps_per_s'] / row['torch_reference']['stamps_per_s']
        rows.append(row)
    return rows


def snr_table(n, dev):
    from gdeconv import fpfs, make_batch_device
    from models.Richard_Lucy import Richard_Lucy
    from models.Tikhonet import Tikhonov
    from models.Wiener import Wiener
    table = []
    for snr in SNRS:
        b = make_batch_device(0, n, float(snr), device=dev)
        g_gt = fpfs(b['gt'])['g']
        outs = dict(No_Deconv=fpfs(b['obs'])['g'], FPFS=fpfs(b['obs'], b['psf'])['g'],
                    Wiener=fpfs(Wiener()(b['obs'], b['psf'], b['alpha']))['g'],
                    Tikhonov_Laplacian=fpfs(Tikhonov('Laplacian')(b['obs'], b['psf'], b['alpha'], 1.0))['g'],
                    RL10=fpfs(Richard_Lucy(10)(b['obs'], b['psf']))['g'])
        row = dict(snr=snr, stamps=n)
        for k, g in outs.items():
            d = (g - g_gt).norm(dim=1).double().cpu()
            ok = d.isfinite()
            row[k] = dict(median_abs_dg=float(d[ok].median()), nan=int((~ok).sum()))
        table.append(row)
    return table


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--stamps', type=int, default=1_000_000)
    ap.add_argument('--piece-stamps', type=int, default=100_000)
    ap.add_argument('--table-stamps', type=int, default=10_000)
    ap.add_argument('--min-seconds', type=float, default=1.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('fpfs_bench needs a CUDA device')
    dev = torch.device('cuda', torch.cuda.current_device())
    t0 = time.time()
    rows = throughput(args, dev)
    torch.cuda.empty_cache()
    print(json.dumps(dict(metric='FPFS shear estimates stamps/s', card=card(dev), torch=torch.__version__, torch_reference_piece=args.piece_stamps,
                          rows=rows, snr_table=snr_table(args.table_stamps, dev), wall_seconds=time.time() - t0)))


if __name__ == '__main__':
    main()
