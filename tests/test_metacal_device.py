"""Metacalibration (gd_metacal / gdeconv.metacal, csrc/metacal.cu) against the float64 torch reference (oracle/metacal.py) and
against analytic answers.

CPU: the reference against analytic sheared and reconvolved Gaussians, the analytic response and rings; the images of
csrc/metacal_core.cuh compiled for the host in the kernel's order (tests/cpu/test_metacal_core.cpp) against the reference; the C
ABI and the Python entry point validate without a device; the library holds k_metacal, which does not spill.
GPU: the kernel against the reference on 2,048 stamps per kind, its shapes against gd_adaptive_moments bit for bit, per-stamp
independence from the batch and from how the PSF is passed, empty batches, NaN stamps, the caller's stream and rings."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT

import gdsynth as G
from oracle.adaptive_moments import OK
from oracle.metacal import PSF_FLOOR, SHEARS, dtft, ensemble_shear, metacal as reference, metacal_images

NPIX = 48 * 48
CSRC = os.path.join(ROOT, 'galaxy-deconv_b200', 'csrc')
NVCC = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
EYE = torch.eye(2, dtype=torch.float64)


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def gaussian(S, mu=(24.0, 24.0)):
    """unit-flux Gaussians of covariance S [n,2,2] (x, y), point-sampled at pixel centres -> float64 [n,48,48]"""
    y, x = torch.meshgrid(torch.arange(48, dtype=torch.float64), torch.arange(48, dtype=torch.float64), indexing='ij')
    Si = torch.linalg.inv(S)
    dx, dy = x[None] - mu[0], y[None] - mu[1]
    q = Si[:, 0, 0, None, None] * dx * dx + 2 * Si[:, 0, 1, None, None] * dx * dy + Si[:, 1, 1, None, None] * dy * dy
    return torch.exp(-0.5 * q) / (2 * math.pi * torch.linalg.det(S).sqrt()[:, None, None])


def shear_matrix(g1, g2):
    return torch.tensor([[1 + g1, g2], [g2, 1 - g1]], dtype=torch.float64)


def unit_shear(g1, g2):
    return shear_matrix(g1, g2) / math.sqrt(1 - g1 * g1 - g2 * g2)


def elliptical_covariances(sig, e, th, g=(0.0, 0.0)):
    """covariances of Gaussians of size det^(1/4) = sig, distortion |e| at angle th, then sheared by g"""
    a2, b2 = sig ** 2 * ((1 + e) / (1 - e)).sqrt(), sig ** 2 * ((1 - e) / (1 + e)).sqrt()
    ct, st = th.cos(), th.sin()
    S = torch.stack([torch.stack([a2 * ct ** 2 + b2 * st ** 2, (a2 - b2) * ct * st], -1),
                     torch.stack([(a2 - b2) * ct * st, a2 * st ** 2 + b2 * ct ** 2], -1)], -2)
    A = shear_matrix(*g)
    return A @ S @ A.T


def gaussians(n=256, seed=5):
    """elliptical Gaussians: size 1.5-4 px, |e| <= 0.5, any orientation, centre within 1 px of (24, 24), flux 10-1e5 (fp32)"""
    gen = torch.Generator().manual_seed(seed)
    u = lambda: torch.rand(n, generator=gen, dtype=torch.float64)
    S = elliptical_covariances(1.5 + 2.5 * u(), 0.5 * u(), math.pi * u())
    mu = (24 + 2 * (u() - 0.5)[:, None, None], 24 + 2 * (u() - 0.5)[:, None, None])
    return (10.0 ** (1 + 4 * u())[:, None, None] * gaussian(S, mu)).float()


def circular_convolve(x, psf):
    """x [n,48,48] convolved circularly with psf [n,48,48] centred at pixel (24, 24), in float64"""
    psf = torch.roll(psf.double(), (-24, -24), (-2, -1))
    return torch.fft.ifft2(torch.fft.fft2(x.double()) * torch.fft.fft2(psf)).real


def unit_psfs(idx):
    p = G.make_psf(idx, 'cpu').double()
    return p / p.sum((1, 2), keepdim=True)


def ring(g, n_rings=64, seed=9):
    """4-orientation rings of elliptical Gaussians (size 2-4 px, |e| <= 0.5) sheared by g and convolved with gdsynth PSFs:
    (stamps fp32 [4 n_rings,48,48], psf fp32 [4 n_rings,48,48])"""
    gen = torch.Generator().manual_seed(seed)
    u = lambda: torch.rand(n_rings, generator=gen, dtype=torch.float64)
    sig, e, th = 2 + 2 * u(), 0.5 * u(), math.pi * u()
    rot = torch.arange(4, dtype=torch.float64) * (math.pi / 4)
    S = elliptical_covariances(sig.repeat_interleave(4), e.repeat_interleave(4), (th[:, None] + rot).flatten(), g)
    psf = unit_psfs(torch.arange(4 * n_rings))
    return (1e3 * circular_convolve(gaussian(S), psf)).float(), psf.float()


def _ref(x, psf=None, device='cpu', **kw):
    r = reference(x.detach().to(device).double(), None if psf is None else psf.detach().to(device).double(), **kw)
    return {k: v.cpu() for k, v in r.items()}


def rel_l2(a, b):
    a, b = a.double().flatten(2), b.double().flatten(2)
    return (a - b).norm(dim=2) / b.norm(dim=2)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference against analytic answers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('psf_sigma', [None, 1.5])
def test_reference_images_are_the_analytic_sheared_reconvolved_gaussians(psf_sigma):
    t = lambda *v: torch.tensor(v, dtype=torch.float64)
    S = elliptical_covariances(t(2.5, 3.0), t(0.0, 0.3), t(0.0, 0.7)) if psf_sigma is None else \
        elliptical_covariances(t(2.0, 2.5), t(0.0, 0.3), t(0.0, 0.7))   # small enough not to wrap around the stamp
    rs, d = (1.0, 0.01) if psf_sigma is None else (1.5, 0.02)
    x = gaussian(S if psf_sigma is None else S + psf_sigma ** 2 * EYE)
    psf = None if psf_sigma is None else gaussian((psf_sigma ** 2 * EYE)[None])
    ims = metacal_images(x, psf, d, rs)
    for j, g in enumerate([(0, 0), (d, 0), (-d, 0), (0, d), (0, -d)]):
        A = unit_shear(*g)
        want = gaussian(A @ S @ A + rs * rs * EYE)
        err = float(((ims[:, j] - want).abs().amax((1, 2)) / want.amax((1, 2))).max())
        assert err <= 1e-10, (j, err)


def test_reference_response_of_a_round_gaussian():
    s, rs, d = 2.5, 1.0, 0.01
    r = reference(gaussian((s * s * EYE)[None]), None, d, rs)

    def e1(g):
        a, b = s * s * (1 + g) ** 2 / (1 - g * g) + rs * rs, s * s * (1 - g) ** 2 / (1 - g * g) + rs * rs
        return (a - b) / (a + b)

    want = (e1(d) - e1(-d)) / (2 * d)
    R = r['R'][0]
    assert r['status'].eq(OK).all()
    assert abs(float(R[0, 0]) - want) <= 1e-4 and abs(float(R[1, 1]) - want) <= 1e-4, (R, want)
    assert float(R[0, 1].abs()) <= 1e-6 and float(R[1, 0].abs()) <= 1e-6 and float(r['e'][0, 0].abs().max()) <= 1e-6


@pytest.mark.parametrize('g,m_tol', [((0.02, -0.01), 2e-3), ((-0.03, 0.05), 8e-3)])
def test_reference_recovers_shear_on_rings(g, m_tol):
    x, psf = ring(g)
    r = _ref(x, psf)
    got = ensemble_shear(r['e'], r['R'], r['status']).tolist()
    m = [got[i] / g[i] - 1 for i in range(2)]
    print(f'\ng={g}: {got} m={m}')
    assert max(abs(v) for v in m) <= m_tol, (got, m)


def test_reference_has_no_additive_bias_on_rings():
    x, psf = ring((0.0, 0.0))
    r = _ref(x, psf)
    c = ensemble_shear(r['e'], r['R'], r['status']).abs().max().item()
    print(f'\nc={c}')
    assert c <= 1e-5, c


# ---------------------------------------------------------------------------------------------------------------------
# CPU: host-compiled core
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def host_core(tmp_path_factory):
    if not os.path.exists(NVCC):
        pytest.skip('nvcc not found')
    d = tmp_path_factory.mktemp('metacal_core')
    exe = str(d / 'test_metacal_core')
    r = subprocess.run([NVCC, '-O2', '-std=c++17', '-Wno-deprecated-gpu-targets', '-I', CSRC,
                        os.path.join(ROOT, 'tests', 'cpu', 'test_metacal_core.cpp'), '-o', exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return exe, d


def run_host(host_core, stamps, psf=None, delta=0.01, reconv_sigma=2.5):
    exe, d = host_core
    d = d / f'run{len(os.listdir(d))}'
    d.mkdir()
    stamps.detach().cpu().float().contiguous().numpy().tofile(d / 'stamps.f32')
    if psf is not None:
        psf.detach().cpu().float().contiguous().numpy().tofile(d / 'psf.f32')
    r = subprocess.run([exe, str(d), repr(float(delta)), repr(float(reconv_sigma))], capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0 and r.stdout.strip().endswith('OK'), r.stdout[-2000:] + r.stderr[-2000:]
    return torch.from_numpy(np.fromfile(d / 'images.f32', dtype=np.float32).reshape(-1, 5, 48, 48))


@pytest.fixture(scope='module')
def synth_stamps():
    """48 gdsynth stamps: gt (noise-free), obs at SNR 20, 100 and 300, and their PSFs"""
    b = {snr: G.make_batch(0, 48, snr) for snr in (20.0, 100.0, 300.0)}
    return dict(gt=b[100.0]['gt'], **{f'obs{int(s)}': b[s]['obs'] for s in b}, psf_of=b[100.0]['psf'])


@pytest.mark.parametrize('kind,with_psf', [('gaussians', False), ('gaussians', True), ('gt', False), ('gt', True), ('obs20', False),
                                           ('obs20', True), ('obs100', False), ('obs100', True), ('obs300', False), ('obs300', True)])
def test_host_core_matches_reference(host_core, synth_stamps, kind, with_psf):
    x = gaussians(48) if kind == 'gaussians' else synth_stamps[kind]
    x = x.reshape(-1, 48, 48)
    psf = synth_stamps['psf_of'][:x.shape[0]] if with_psf else None
    got = run_host(host_core, x, psf)
    want = metacal_images(x.double(), None if psf is None else psf.double(), 0.01, 2.5)
    err = rel_l2(got, want)
    print(f'\n{kind} psf={with_psf}: rel-L2 max {float(err.max()):.3e} median {float(err.median()):.3e}')
    assert float(err.max()) <= 2e-6


def test_host_core_broadcast_psf_and_options(host_core, synth_stamps):
    x, psf = synth_stamps['obs100'][:8].reshape(-1, 48, 48), synth_stamps['psf_of'][3:4]
    got = run_host(host_core, x, psf, 0.05, 3.0)
    assert torch.equal(got, run_host(host_core, x, psf.expand(8, -1, -1, -1), 0.05, 3.0))
    assert float(rel_l2(got, metacal_images(x.double(), psf.double(), 0.05, 3.0)).max()) <= 2e-6


# ---------------------------------------------------------------------------------------------------------------------
# CPU: validation and build
# ---------------------------------------------------------------------------------------------------------------------
def test_metacal_validates_without_a_device():
    from gdeconv import _lib
    lib = _lib.lib
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    nan, inf = float('nan'), float('inf')
    cases = [  # (img, psf, psf_batch, batch, delta, reconv_sigma, guess_sigma, images, shape, info)
        (p, None, 0, -1, 0.01, 2.5, 3.0, p, p, p),
        (None, None, 0, 2, 0.01, 2.5, 3.0, p, p, p),
        (p, None, 0, 2, 0.01, 2.5, 3.0, p, None, p),
        (p, None, 0, 2, 0.01, 2.5, 3.0, p, p, None),
        (p, None, 0, 0, 0.01, 2.5, 3.0, p, None, p),
        (p, None, 1, 2, 0.01, 2.5, 3.0, p, p, p),          # psf_batch without a psf
        (p, p, 0, 2, 0.01, 2.5, 3.0, p, p, p),             # a psf without psf_batch
        (p, p, 3, 2, 0.01, 2.5, 3.0, p, p, p),
        (p, p, 2, 3, 0.01, 2.5, 3.0, p, p, p),
        (p, p, -1, 2, 0.01, 2.5, 3.0, p, p, p),
    ] + [(p, None, 0, 2, d, 2.5, 3.0, p, p, p) for d in (0.0, -0.01, 0.1001, nan, inf)] \
      + [(p, None, 0, 2, 0.01, s, 3.0, p, p, p) for s in (0.0, -1.0, 24.5, nan, inf)] \
      + [(p, None, 0, 2, 0.01, 2.5, s, p, p, p) for s in (0.0, -1.0, 24.5, nan, inf)]
    for case in cases:
        rc = lib.gd_metacal(*case, None)
        assert rc == -1, (case, rc)                       # GD_EBADSHAPE
        assert b'gd_metacal' in lib.gd_last_error(), 'gd_last_error() must explain the rejection'
    assert lib.gd_metacal(None, None, 0, 0, 0.01, 2.5, 3.0, None, p, p, None) == 0
    assert lib.gd_metacal(None, p, 1, 0, 0.1, 24.0, 24.0, None, p, p, None) == 0


def test_metacal_rejects_bad_tensors():
    from gdeconv import metacal
    for t in (torch.rand(2, 1, 48, 48), torch.rand(2, 1, 48, 48, dtype=torch.float64), torch.rand(2, 48, 48)):
        with pytest.raises(RuntimeError, match='no CPU path'):
            metacal(t)
    with pytest.raises(TypeError):
        metacal(np.zeros((2, 1, 48, 48), np.float32))


def test_library_contains_the_metacal_kernel():
    from gdeconv import _lib
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    sass = subprocess.run([cuobjdump, '-sass', _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert 'k_metacal' in sass and 'sm_100a' in sass


def test_metacal_kernel_does_not_spill(tmp_path):
    if not os.path.exists(NVCC):
        pytest.skip('nvcc not found')
    r = subprocess.run([NVCC, '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-std=c++17', '--expt-relaxed-constexpr', '-Xptxas', '-v',
                        '-c', os.path.join(CSRC, 'metacal.cu'), '-o', str(tmp_path / 'metacal.o')], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    m = re.search(r"Compiling entry function '\w*k_metacal\w*'.*?(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                  r.stdout + r.stderr, re.S)
    assert m, (r.stdout + r.stderr)[-2000:]
    assert m.groups() == ('0', '0', '0'), m.group(0)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _gpu(x, psf=None, **kw):
    from gdeconv import metacal
    return metacal(x.reshape(-1, 1, 48, 48).cuda(), None if psf is None else psf.reshape(-1, 1, 48, 48).cuda(), **kw)


def _device_stamps(kind, snr, n=2048, start=30000):
    from gdeconv import make_batch_device
    from models.Wiener import Wiener
    b = make_batch_device(start, n, snr, device='cuda:0')
    if kind == 'wiener':
        return Wiener()(b['obs'], b['psf'], b['alpha']), None
    if kind == 'gaussians':
        return gaussians(n).reshape(-1, 1, 48, 48).cuda(), None
    return b[kind], b['psf']


def near_floor(psf, delta=0.01):
    """[B,5] bool: image j of the stamp has a cell whose PSF power |P(A_j k)|^2 is within 1e-3 of the 1e-8 floor.  There fp32
    and float64 can decide the floor differently, and a cell kept by one and zeroed by the other moves the image by up to ~1e-5
    rel-L2 (measured: 5.0e-6 on one of 10,240 SNR-20 images, the host build of the core agreeing with the kernel)."""
    psf = psf.reshape(-1, 48, 48).double()
    p0 = psf.sum((1, 2)).reshape(-1, 1, 1)
    flags = []
    for s in SHEARS:
        P = dtft(psf, (delta * s[0], delta * s[1])) / p0
        h = (P.real ** 2 + P.imag ** 2) / PSF_FLOOR
        flags.append(((h - 1).abs() <= 1e-3).flatten(1).any(1))
    return torch.stack(flags, 1).cpu()


def check_against_reference(got, want, psf=None):
    """images rel-L2 <= 2e-6 (<= 2e-5 on an image with a PSF cell at the floor, see near_floor), statuses identical,
    |de| <= 2e-5 on every OK image, |dR| <= 2e-3; returns maxima and medians"""
    err = rel_l2(got['images'].reshape(-1, 5, NPIX).cpu(), want['images'].reshape(-1, 5, NPIX))
    at_floor = near_floor(psf) if psf is not None else torch.zeros_like(err, dtype=torch.bool)
    st = got['status'].cpu()
    assert torch.equal(st, want['status'].to(st.dtype)), int((st != want['status']).sum())
    ok = st == OK
    de = (got['e'].cpu().double() - want['e'])[ok].abs()
    allok = ok.all(1)
    dR = (got['R'].cpu().double() - want['R'])[allok].abs()
    stats = dict(img_rel_l2=(float(err[~at_floor].max()), float(err.median())), de=(float(de.max()), float(de.median())),
                 dR=(float(dR.max()), float(dR.median())), ok_images=int(ok.sum()), ok_stamps=int(allok.sum()),
                 at_floor_images=int(at_floor.sum()), at_floor_max=float(err[at_floor].max()) if at_floor.any() else 0.0)
    assert stats['img_rel_l2'][0] <= 2e-6 and stats['at_floor_max'] <= 2e-5, stats
    assert stats['de'][0] <= 2e-5 and stats['dR'][0] <= 2e-3, stats
    return stats


@pytest.mark.gpu
@pytest.mark.parametrize('kind,snr,with_psf', [('gaussians', 100.0, False), ('gt', 100.0, False), ('obs', 20.0, True), ('obs', 100.0, True),
                                               ('obs', 300.0, True), ('wiener', 100.0, False)])
def test_kernel_matches_reference(kind, snr, with_psf):
    x, psf = _device_stamps(kind, snr)
    psf = psf if with_psf else None
    got = _gpu(x, psf, images=True)
    want = _ref(x, psf, device='cuda:0')
    print(f'\n{kind} snr={snr} psf={with_psf}:', check_against_reference(got, want, psf))


def _bits(r, i=slice(None)):
    return torch.cat([r['e'][i].reshape(-1).view(torch.int32), r['status'][i].reshape(-1), r['n_iter'][i].reshape(-1),
                      r['images'][i].reshape(-1).view(torch.int32)])


@pytest.mark.gpu
def test_shapes_are_adaptive_moments_of_the_images():
    """the shape and info records equal gd_adaptive_moments on the returned images bit for bit, and do not depend on whether
    the images are written"""
    from gdeconv import make_batch_device
    from gdeconv._lib import lib
    from gdeconv.engine import _ptr, _stream
    b = make_batch_device(0, 500, 'mixed', device='cuda:0')
    x, st = b['obs'], _stream(torch.device('cuda:0'))
    for p in (None, b['psf'][:1], b['psf']):
        ims = torch.empty(500, 5, NPIX, device='cuda:0')
        records = []
        for out in (ims, None):
            shape = torch.empty(500, 5, 8, device='cuda:0')
            info = torch.empty(500, 5, 2, dtype=torch.int32, device='cuda:0')
            assert lib.gd_metacal(_ptr(x), _ptr(p), 0 if p is None else p.shape[0], 500, 0.01, 2.5, 3.0, _ptr(out), _ptr(shape),
                                  _ptr(info), st) == 0
            records.append((shape, info))
        am_shape = torch.empty(2500, 8, device='cuda:0')
        am_info = torch.empty(2500, 2, dtype=torch.int32, device='cuda:0')
        assert lib.gd_adaptive_moments(_ptr(ims), 2500, 3.0, _ptr(am_shape), _ptr(am_info), st) == 0
        torch.cuda.synchronize()
        for shape, info in records:
            assert torch.equal(shape.reshape(-1, 8).view(torch.int32), am_shape.view(torch.int32))
            assert torch.equal(info.reshape(-1, 2), am_info)


@pytest.mark.gpu
def test_a_stamp_does_not_depend_on_its_batch_or_psf_form():
    from gdeconv import metacal, make_batch_device
    b = make_batch_device(0, 1200, 'mixed', device='cuda:0')
    x, psf = b['obs'], b['psf']
    for p in (None, psf):
        full = metacal(x, p, images=True)
        one = metacal(x[1000:1001], None if p is None else p[1000:1001], images=True)
        sub = metacal(x[990:1027], None if p is None else p[990:1027], images=True)
        shifted = metacal(torch.cat([x[:3], x[1000:1001], x[5:41]]), None if p is None else torch.cat([p[:3], p[1000:1001], p[5:41]]),
                          images=True)
        want = _bits(full, 1000)
        assert torch.equal(_bits(one, 0), want) and torch.equal(_bits(sub, 10), want) and torch.equal(_bits(shifted, 3), want)
    p1 = psf[7:8]
    assert torch.equal(_bits(metacal(x[:300], p1, images=True)), _bits(metacal(x[:300], p1.expand(300, -1, -1, -1).contiguous(), images=True)))
    with pytest.raises(ValueError):
        metacal(x, psf[:2])
    with pytest.raises(RuntimeError, match='delta'):
        metacal(x, delta=0.0)
    with pytest.raises(RuntimeError, match='reconv_sigma'):
        metacal(x, reconv_sigma=float('nan'))


@pytest.mark.gpu
def test_empty_batch_and_nan_stamps():
    from gdeconv import launch_count, metacal, make_batch_device
    n0 = launch_count()
    for p in (None, torch.rand(1, 1, 48, 48, device='cuda:0'), torch.empty(0, 1, 48, 48, device='cuda:0')):
        got = metacal(torch.empty(0, 1, 48, 48, device='cuda:0'), p, images=True)
        for k, s in dict(e=(0, 5, 2), status=(0, 5), n_iter=(0, 5), R=(0, 2, 2), g=(0, 2), images=(0, 5, 1, 48, 48)).items():
            assert tuple(got[k].shape) == s and got[k].is_cuda, k
    assert launch_count() == n0
    b = make_batch_device(0, 40, 100.0, device='cuda:0')
    for p in (None, b['psf']):
        want = metacal(b['obs'], p, images=True)
        x = b['obs'].clone()
        x[17, 0, 5, 9] = float('nan')
        got = metacal(x, p, images=True)
        assert (got['status'][17] == 2).all() and got['g'][17].isnan().all()          # GD_SHAPE_FLUX
        keep = torch.arange(40, device='cuda:0') != 17
        assert torch.equal(_bits(got, keep), _bits(want, keep))


@pytest.mark.gpu
def test_runs_on_the_current_stream():
    """The input is written on a side stream after a delay; only that stream is synchronised: a kernel on any other stream
    would read the zeros that were there before."""
    from gdeconv import metacal, make_batch_device
    b = make_batch_device(0, 2048, 100.0, device='cuda:0')
    want = metacal(b['obs'], b['psf'], images=True)
    buf = torch.zeros_like(b['obs'])
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device='cuda:0')
    with torch.cuda.stream(s):
        torch.cuda._sleep(20_000_000)
        buf.copy_(b['obs'])
        got = metacal(buf, b['psf'], images=True)
    s.synchronize()
    assert torch.equal(_bits(got), _bits(want))


@pytest.mark.gpu
@pytest.mark.parametrize('g,m_tol', [((0.02, -0.01), 2e-3), ((-0.03, 0.05), 8e-3)])
def test_shear_recovery_on_rings(g, m_tol):
    x, psf = ring(g)
    got = _gpu(x, psf)
    want = _ref(x, psf, device='cuda:0')
    gd = ensemble_shear(got['e'].cpu().double(), got['R'].cpu().double(), got['status'].cpu())
    gr = ensemble_shear(want['e'], want['R'], want['status'])
    print(f'\ng={g}: device {gd.tolist()}, reference {gr.tolist()}')
    assert float(((gd - gr).abs() / gr.abs()).max()) <= 1e-4, (gd, gr)
    assert max(abs(float(gd[i]) / g[i] - 1) for i in range(2)) <= m_tol, gd
