#!/usr/bin/env python
"""Stamps/s of metacalibration on one GPU, and (as context) a table of shear errors at three SNRs.

  device           gdeconv.metacal: k_metacal (csrc/metacal.cu) with no PSF, one PSF for the batch and a per-stamp PSF
  device_fixnoise  the same with fix-noise (k_metacal_fixnoise), the noise field generated at gdsynth.SIGMA
  torch_reference  oracle/metacal.py in fp32 on the same GPU, in --piece-stamps pieces, on --ref-stamps stamps: the
                   library-free baseline

Workload: --stamps SNR-100 obs stamps and their PSFs from gdeconv.make_batch_device (9.2 GB each for 1,000,000 stamps, far
beyond the L2).  Each arm is warmed up on its workload, then passes over the whole workload repeat until the CUDA-event window
reaches --min-seconds.  FMAs per stamp are those of the direct DTFT, counted from shapes: 4 sheared spectra x 1,105 half-plane
targets x (48 x 48 x 2 + 48 x 4) per image transformed (the stamp, and a per-stamp PSF); fix-noise adds the noise field's
DTFT at all 5 x 1,105 (shear, target) pairs.  The grid transforms and the shapes are left out.

Table (context, not a gate): for SNR 20, 100 and 300, --table-stamps stamps from make_batch_device; the median over stamps of
|g - g_gt| (the norm of the two-component difference of the per-galaxy shears), where g_gt is metacal of gt with no PSF, for
metacal of obs with its PSF (without and with generated fix-noise at gdsynth.SIGMA), and metacal with no PSF of the Wiener
(without and with caller fix-noise Wiener(sigma N)) and RL(10) outputs.  Stamps with a NaN shear (a status other
than OK on one of the five images) are counted and left out of the median.  The card's name and power limit are read in the
same run.

Noisy rings (context): the noise-bias study of tests/test_metacal_fixnoise.py at --ring-groups rings of SNR 50 per g: m at
g = (0.02, -0.01), c at g = 0 and their jackknife errors, with and without fix-noise.

    python tools/metacal_bench.py [--stamps 1000000] [--ref-stamps 20000] [--piece-stamps 2000] [--table-stamps 10000] [--min-seconds 1]
                                  [--ring-groups 200000]

Prints one JSON line.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, 'galaxy-deconv_b200'), ROOT, os.path.join(ROOT, 'tools'), os.path.join(ROOT, 'tests')]

import torch  # noqa: E402

from synth_bench import card, rate  # noqa: E402
from test_metacal_fixnoise import SIGMA, noise_bias  # noqa: E402

SNRS = (20, 100, 300)
TARGETS = 4 * 1105
FMA_PER_IMAGE = TARGETS * (48 * 48 * 2 + 48 * 4)
FMA_FIXNOISE = 5 * 1105 * (48 * 48 * 2 + 48 * 4)


def pieces(fn, x, psf, piece):
    for i in range(0, x.shape[0], piece):
        fn(x[i:i + piece], psf if psf is None or psf.shape[0] == 1 else psf[i:i + piece])


def throughput(args, dev):
    from gdeconv import make_batch_device, metacal
    from oracle.metacal import metacal as reference
    b = make_batch_device(0, args.stamps, 100.0, device=dev, keys=('obs', 'psf'))
    rows = []
    for mode in ('no PSF', 'one PSF', 'per-stamp PSF'):
        x = b['obs']
        p = None if mode == 'no PSF' else b['psf'][:1] if mode == 'one PSF' else b['psf']
        fma = FMA_PER_IMAGE * (2 if mode == 'per-stamp PSF' else 1)
        row = dict(workload=f'obs, SNR 100, {mode}', stamps=args.stamps, dtft_fma_per_stamp=fma)
        row['device'] = rate(lambda: metacal(x, p), args.stamps, args.min_seconds)
        row['device']['achieved_TFMA_per_s'] = row['device']['stamps_per_s'] * fma / 1e12
        row['dtft_fma_per_stamp_fixnoise'] = fma + FMA_FIXNOISE
        row['device_fixnoise'] = rate(lambda: metacal(x, p, noise_sigma=SIGMA), args.stamps, args.min_seconds)
        row['device_fixnoise']['achieved_TFMA_per_s'] = row['device_fixnoise']['stamps_per_s'] * (fma + FMA_FIXNOISE) / 1e12
        n = args.ref_stamps
        xr, pr = x[:n], None if p is None else p[:n] if p.shape[0] > 1 else p
        row['torch_reference'] = rate(lambda: pieces(reference, xr, pr, args.piece_stamps), n, args.min_seconds)
        row['torch_reference']['stamps'] = n
        torch.cuda.empty_cache()
        row['speedup_vs_torch_reference'] = row['device']['stamps_per_s'] / row['torch_reference']['stamps_per_s']
        rows.append(row)
    return rows


def snr_table(n, dev):
    from gdeconv import make_batch_device, metacal
    from models.Richard_Lucy import Richard_Lucy
    from models.Wiener import Wiener
    table = []
    for snr in SNRS:
        b = make_batch_device(0, n, float(snr), device=dev)
        g_gt = metacal(b['gt'])['g']
        wn = Wiener()(SIGMA * torch.randn(b['obs'].shape, device=dev, generator=torch.Generator(dev).manual_seed(snr)), b['psf'], b['alpha'])
        outs = dict(metacal_obs_with_psf=metacal(b['obs'], b['psf'])['g'],
                    metacal_obs_with_psf_fixnoise=metacal(b['obs'], b['psf'], noise_sigma=SIGMA, seed=snr)['g'],
                    Wiener=metacal(Wiener()(b['obs'], b['psf'], b['alpha']))['g'],
                    Wiener_fixnoise=metacal(Wiener()(b['obs'], b['psf'], b['alpha']), noise=wn)['g'],
                    RL10=metacal(Richard_Lucy(10)(b['obs'], b['psf']))['g'])
        row = dict(snr=snr, stamps=n, gt_nan=int(g_gt.isnan().any(1).sum()))
        for k, g in outs.items():
            d = (g - g_gt).norm(dim=1).double().cpu()
            ok = d.isfinite()
            row[k] = dict(median_abs_dg=float(d[ok].median()), nan=int((~ok).sum()))
        table.append(row)
    return table


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--stamps', type=int, default=1_000_000)
    ap.add_argument('--ref-stamps', type=int, default=20_000)
    ap.add_argument('--piece-stamps', type=int, default=2_000)
    ap.add_argument('--table-stamps', type=int, default=10_000)
    ap.add_argument('--min-seconds', type=float, default=1.0)
    ap.add_argument('--ring-groups', type=int, default=200_000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('metacal_bench needs a CUDA device')
    dev = torch.device('cuda', torch.cuda.current_device())
    t0 = time.time()
    rows = throughput(args, dev)
    torch.cuda.empty_cache()
    print(json.dumps(dict(metric='metacalibration stamps/s', card=card(dev), torch=torch.__version__, torch_reference_piece=args.piece_stamps,
                          rows=rows, snr_table=snr_table(args.table_stamps, dev),
                          noisy_rings_snr50=noise_bias(args.ring_groups), wall_seconds=time.time() - t0)))


if __name__ == '__main__':
    main()
