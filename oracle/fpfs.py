"""FPFS shear estimation of 48x48 stamps in plain torch: the reference of gd_fpfs / gdeconv.fpfs.

The estimator (Li, Li & Mandelbaum 2018, MNRAS 481, 4445) is the one stated in galaxy-deconv_b200/csrc/fpfs_core.cuh.  On the
grid k = 2 pi (u, v) / 48 (u, v the fftfreq integers, kx along columns) with r^2 = sigma^2 |k|^2 and G = exp(-r^2/2), the
deconvolved power D = |FT img|^2 / P, P = |FT psf|^2 / |FT psf(0)|^2 (cells with P < 1e-8 give 0; no PSF: P = 1), is projected on
    M00 = sum D G / (sigma sqrt(pi)),                       M22c, M22s = sum D r^2 (cos 2phi, sin 2phi) G / (sigma sqrt(2 pi)),
    M40 = sum D (r^4 - 4 r^2 + 2)/2 G / (sigma sqrt(pi)),   M42c, M42s = -sum D r^2 (3 - r^2) (cos 2phi, sin 2phi) G / (sigma sqrt(6 pi))
over all 2304 cells, and w = M00 + const, e1 = -M22c/w, e2 = -M22s/w, e41 = -M42c/w, e42 = -M42s/w,
R = (M00 - M40)/(sqrt(2) w) + sqrt(6)/2 (e1 e41 + e2 e42).  Batched over stamps, device- and dtype-agnostic: the tests run it in
float64 on the CPU.  Pixel p = 48 r + c is at x = c, y = r.
"""
import math

import torch

STAMP = 48
PSF_FLOOR = 1e-8


def basis(sigma, device='cpu', dtype=torch.float64):
    """the six per-cell basis functions [6,48,48] (M00, M22c, M22s, M40, M42c, M42s), normalisation included, on the
    torch.fft.fft2 grid of a 48x48 stamp"""
    f = torch.fft.fftfreq(STAMP, 1.0 / STAMP, device=device, dtype=dtype)
    kx, ky = (2 * math.pi / STAMP) * f[None, :], (2 * math.pi / STAMP) * f[:, None]
    s2 = float(sigma) ** 2
    a, b = s2 * kx * kx, s2 * ky * ky                  # r^2 = a + b, r^2 cos 2phi = a - b, r^2 sin 2phi = 2 sigma^2 kx ky
    r2, c2, t2 = a + b, a - b, 2 * s2 * kx * ky
    G = torch.exp(-0.5 * r2)
    n0, n2, n4 = 1 / (sigma * math.sqrt(math.pi)), 1 / (sigma * math.sqrt(2 * math.pi)), -1 / (sigma * math.sqrt(6 * math.pi))
    return torch.stack([n0 * G, n2 * c2 * G, n2 * t2 * G, n0 * 0.5 * (r2 * r2 - 4 * r2 + 2) * G,
                        n4 * (3 - r2) * c2 * G, n4 * (3 - r2) * t2 * G])


def fpfs(img, psf=None, sigma=3.5, const=0.0):
    """img [B,48,48] or [B,1,48,48]; psf None (a delta PSF) or [1 or B,(1,)48,48] -> dict(modes [B,6] (M00, M22c, M22s, M40,
    M42c, M42s), e [B,2], R [B], g [B,2] = e / R), in img's dtype.  e and R are NaN where w <= 0; everything is NaN for a stamp
    whose PSF does not sum to a positive value."""
    img = img.reshape(-1, STAMP, STAMP)
    B, dev, dt = img.shape[0], img.device, img.dtype
    F = torch.fft.fft2(img)
    D = F.real ** 2 + F.imag ** 2
    bad = torch.zeros(B, dtype=torch.bool, device=dev)
    if psf is not None:
        psf = psf.reshape(-1, STAMP, STAMP).to(dt)
        H = torch.fft.fft2(psf)
        hh = H.real ** 2 + H.imag ** 2
        P = hh / hh[:, :1, :1]
        D = torch.where(P >= PSF_FLOOR, D / P, torch.zeros((), device=dev, dtype=dt))
        bad = (~(psf.sum((1, 2)) > 0)).expand(B)
    modes = torch.einsum('bij,mij->bm', D, basis(sigma, dev, dt))
    modes = torch.where(bad[:, None], torch.full_like(modes, float('nan')), modes)
    M00, M22c, M22s, M40, M42c, M42s = modes.unbind(1)
    w = M00 + const
    w = torch.where(w > 0, w, torch.full_like(w, float('nan')))
    e1, e2, e41, e42 = -M22c / w, -M22s / w, -M42c / w, -M42s / w
    R = (M00 - M40) / (math.sqrt(2) * w) + math.sqrt(6) / 2 * (e1 * e41 + e2 * e42)
    e = torch.stack([e1, e2], 1)
    return dict(modes=modes, e=e, R=R, g=e / R[:, None])
