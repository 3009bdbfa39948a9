"""Adaptive second moments of 48x48 stamps in plain torch: the reference of gd_adaptive_moments / gdeconv.adaptive_moments.

The estimator is the one stated in galaxy-deconv_b200/csrc/shape_core.cuh (Bernstein & Jarvis 2002; Hirata & Seljak 2003):
an elliptical Gaussian weight w = exp(-rho^2/2), rho^2 = (Myy dx^2 - 2 Mxy dx dy + Mxx dy^2) / det(M), started at (24, 24) with
M = guess_sigma^2 I and iterated until the centroid and M reproduce the weighted centroid and twice the weighted central second
moments.  Batched over stamps; stamps that have stopped are dropped from the working set.  Device- and dtype-agnostic: the
tests run it in float64 on the CPU.  Pixel p = 48 r + c is at x = c, y = r.
"""
import torch

STAMP = 48
START = 24.0
MAX_PASSES = 100
TOL = 1e-5
MAX_TRACE = 2.0 * 24 ** 2
MAX_SHIFT = 15.0
OK, MAXITER, FLUX, MOMENTS, CENTROID = 0, 1, 2, 3, 4


def adaptive_moments(img, guess_sigma=3.0, max_passes=MAX_PASSES):
    """img [B,48,48] or [B,1,48,48] -> dict(flux [B], centroid [B,2] (x, y), M [B,3] (Mxx, Mxy, Myy), e [B,2], sigma [B],
    status [B] int32, n_iter [B] int32), floats in img's dtype, NaN wherever status is not OK.  ``max_passes`` other than the
    estimator's 100 only serves to find out how a stamp that ran out of passes would have ended."""
    img = img.reshape(-1, STAMP * STAMP)
    B, dev, dt = img.shape[0], img.device, img.dtype
    r = torch.arange(STAMP, device=dev, dtype=dt).repeat_interleave(STAMP)
    c = torch.arange(STAMP, device=dev, dtype=dt).repeat(STAMP)
    x0 = torch.full((B,), START, device=dev, dtype=dt)
    y0 = x0.clone()
    mxx = torch.full((B,), float(guess_sigma) ** 2, device=dev, dtype=dt)
    mxy = torch.zeros(B, device=dev, dtype=dt)
    myy = mxx.clone()
    flux = torch.full((B,), float('nan'), device=dev, dtype=dt)
    status = torch.full((B,), MAXITER, device=dev, dtype=torch.int32)
    n_iter = torch.full((B,), max_passes, device=dev, dtype=torch.int32)
    act = torch.arange(B, device=dev)                     # stamps still iterating
    for k in range(1, max_passes + 1):
        if act.numel() == 0:
            break
        I = img[act]
        ax0, ay0, axx, axy, ayy = x0[act], y0[act], mxx[act], mxy[act], myy[act]
        dx = c - ax0[:, None]
        dy = r - ay0[:, None]
        D = axx * ayy - axy * axy
        rho2 = (ayy[:, None] * dx * dx - 2 * axy[:, None] * dx * dy + axx[:, None] * dy * dy) / D[:, None]
        v = I * torch.exp(-0.5 * rho2)
        A = v.sum(1)
        Bx, By = (v * dx).sum(1), (v * dy).sum(1)
        Cxx, Cxy, Cyy = (v * dx * dx).sum(1), (v * dx * dy).sum(1), (v * dy * dy).sum(1)
        bad_flux = ~(A > 0)
        mx, my = Bx / A, By / A
        nxx = 2 * (Cxx / A - mx * mx)
        nxy = 2 * (Cxy / A - mx * my)
        nyy = 2 * (Cyy / A - my * my)
        bad_mom = ~((nxx > 0) & (nyy > 0) & (nxx * nyy - nxy * nxy > 0)) | (nxx + nyy > MAX_TRACE)
        nx0, ny0 = ax0 + mx, ay0 + my
        bad_cen = ((nx0 - START).abs() > MAX_SHIFT) | ((ny0 - START).abs() > MAX_SHIFT)
        t = 0.5 * (nxx + nyy)
        conv = (torch.maximum(mx.abs(), my.abs()) <= TOL * t.sqrt()) & \
               (torch.maximum(torch.maximum((nxx - axx).abs(), (nxy - axy).abs()), (nyy - ayy).abs()) <= TOL * t)
        st = torch.where(bad_flux, FLUX, torch.where(bad_mom, MOMENTS, torch.where(bad_cen, CENTROID, torch.where(conv, OK, -1))))
        go = (st == -1) | (st == OK)                      # the update is taken on these
        idx = act[go]
        x0[idx], y0[idx], mxx[idx], mxy[idx], myy[idx] = nx0[go], ny0[go], nxx[go], nxy[go], nyy[go]
        stop = st != -1
        sidx = act[stop]
        status[sidx] = st[stop].to(torch.int32)
        n_iter[sidx] = k
        ok = st == OK
        flux[act[ok]] = 2 * A[ok]
        act = act[~stop]
    good = status == OK
    nan = torch.tensor(float('nan'), device=dev, dtype=dt)
    keep = lambda t: torch.where(good, t, nan)
    mxx, mxy, myy, x0, y0 = keep(mxx), keep(mxy), keep(myy), keep(x0), keep(y0)
    tr = mxx + myy
    M = torch.stack([mxx, mxy, myy], 1)
    return dict(flux=keep(flux), centroid=torch.stack([x0, y0], 1), M=M, e=torch.stack([(mxx - myy) / tr, 2 * mxy / tr], 1),
                sigma=(mxx * myy - mxy * mxy).pow(0.25), status=status, n_iter=n_iter)
