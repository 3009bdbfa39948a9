"""Metacalibration of 48x48 stamps in plain torch: the reference of gd_metacal / gdeconv.metacal.

The definition is the one stated in galaxy-deconv_b200/csrc/metacal_core.cuh (Huff & Mandelbaum 2017; Sheldon & Huff 2017).
Pixel p = 48 r + c sits at X = c - 24, Y = r - 24; on the grid k = 2 pi (u, v) / 48 (u, v the fftfreq integers, kx along
columns), with I~(q) = sum I[r,c] exp(-i (qx X + qy Y)), A_g = [[1+g1, g2], [g2, 1-g1]] / sqrt(1 - g1^2 - g2^2) and
G~(k) = exp(-sigma^2 |k|^2 / 2), image j of the shears (0,0), (+d,0), (-d,0), (0,+d), (0,-d) is Re ifft2(M_j (-1)^(u+v)) with
M_j(k) = I~(A_j k) G~(k) / P(A_j k), P = p~ / p~(0) (0 where |P|^2 < 1e-8, and on the Nyquist row and column; no PSF: P = 1).
Every spectrum, the noshear one included, is the direct DTFT, factorised by rows: a sum over the columns of each row, then over
the rows.  The shapes are oracle/adaptive_moments.py's; R[:, i, j] = (e_i(+d_j) - e_i(-d_j)) / (2 d), g = R^-1 e(noshear).
Batched over stamps, device- and dtype-agnostic: the tests run it in float64.
"""
import math

import torch

from oracle.adaptive_moments import OK, adaptive_moments

STAMP = 48
PSF_FLOOR = 1e-8
SHEARS = ((0.0, 0.0), (1.0, 0.0), (-1.0, 0.0), (0.0, 1.0), (0.0, -1.0))   # in units of delta


def _grid(device, dtype):
    f = torch.fft.fftfreq(STAMP, 1.0 / STAMP, device=device, dtype=dtype)
    v, u = torch.meshgrid(f, f, indexing='ij')                      # rows carry v (ky), columns u (kx)
    return u, v


def dtft(img, g, chunk=64):
    """I~(A_g k) of img [B,48,48] on the fft grid of k -> complex [B,48,48]"""
    B, dev, dt = img.shape[0], img.device, img.dtype
    u, v = _grid(dev, dt)
    g1, g2 = g
    n = 1 / math.sqrt(1 - g1 * g1 - g2 * g2)
    w = 2 * math.pi / STAMP
    qx = (w * n * ((1 + g1) * u + g2 * v)).reshape(-1, 1)
    qy = (w * n * (g2 * u + (1 - g1) * v)).reshape(-1, 1)
    X = torch.arange(STAMP, device=dev, dtype=dt) - STAMP // 2
    ex, ey = torch.exp(-1j * qx * X), torch.exp(-1j * qy * X)       # [2304, 48]: over columns, over rows
    out = []
    for i in range(0, B, chunk):
        T = torch.einsum('brc,kc->bkr', img[i:i + chunk].to(ex.dtype), ex)   # the sum over the columns of each row
        out.append((T * ey).sum(-1))                                          # then over the rows
    return torch.cat(out).reshape(B, STAMP, STAMP) if out else torch.zeros(0, STAMP, STAMP, dtype=ex.dtype, device=dev)


def metacal_images(img, psf=None, delta=0.01, reconv_sigma=2.5):
    """img [B,(1,)48,48]; psf None or [1 or B,(1,)48,48] -> the five images [B,5,48,48] (noshear, 1p, 1m, 2p, 2m), img's dtype"""
    img = img.reshape(-1, STAMP, STAMP)
    dev, dt = img.device, img.dtype
    u, v = _grid(dev, dt)
    w = 2 * math.pi / STAMP
    gam = torch.exp(-0.5 * reconv_sigma ** 2 * w * w * (u * u + v * v))
    nyq = (u == -STAMP // 2) | (v == -STAMP // 2)
    sign = 1 - 2 * ((u + v).remainder(2))
    if psf is not None:
        psf = psf.reshape(-1, STAMP, STAMP).to(dt)
        p0 = psf.sum((1, 2)).reshape(-1, 1, 1)
    outs = []
    for s in SHEARS:
        g = (delta * s[0], delta * s[1])
        M = dtft(img, g) * gam
        if psf is not None:
            P = dtft(psf, g) / p0
            bad = P.real ** 2 + P.imag ** 2 < PSF_FLOOR
            M = torch.where(bad, torch.zeros((), dtype=M.dtype, device=dev), M / torch.where(bad, torch.ones((), dtype=P.dtype, device=dev), P))
        M = torch.where(nyq, torch.zeros((), dtype=M.dtype, device=dev), M) * sign
        outs.append(torch.fft.ifft2(M).real)
    return torch.stack(outs, 1)


def response(e, delta):
    """e [B,5,2] -> R [B,2,2], R[:, i, j] = (e_i(+delta_j) - e_i(-delta_j)) / (2 delta)"""
    return torch.stack([e[:, 1] - e[:, 2], e[:, 3] - e[:, 4]], 2) / (2 * delta)


def ensemble_shear(e, R, status):
    """<R>^-1 <e(noshear)> over the stamps whose five statuses are OK -> [2]"""
    ok = (status == OK).all(1)
    return torch.linalg.solve(R[ok].mean(0), e[ok, 0].mean(0))


def metacal(img, psf=None, delta=0.01, reconv_sigma=2.5, guess_sigma=3.0):
    """-> dict(images [B,5,48,48], e [B,5,2], status [B,5], n_iter [B,5], R [B,2,2], g [B,2]) as gdeconv.metacal"""
    ims = metacal_images(img, psf, delta, reconv_sigma)
    B = ims.shape[0]
    r = adaptive_moments(ims.reshape(-1, STAMP, STAMP), guess_sigma)
    e = r['e'].reshape(B, 5, 2)
    status, n_iter = r['status'].reshape(B, 5), r['n_iter'].reshape(B, 5)
    R = response(e, delta)
    e0, det = e[:, 0], R[:, 0, 0] * R[:, 1, 1] - R[:, 0, 1] * R[:, 1, 0]
    g = torch.stack([R[:, 1, 1] * e0[:, 0] - R[:, 0, 1] * e0[:, 1], R[:, 0, 0] * e0[:, 1] - R[:, 1, 0] * e0[:, 0]], 1) / det[:, None]
    g = torch.where((status == OK).all(1)[:, None], g, torch.full_like(g, float('nan')))
    return dict(images=ims, e=e, status=status, n_iter=n_iter, R=R, g=g)
