"""FPFS shear estimation (gd_fpfs / gdeconv.fpfs, csrc/fpfs.cu) against the float64 torch reference (oracle/fpfs.py) and against
analytic answers.

CPU: the reference against the shear response of round Gaussians, its PSF correction and a ring test; the estimator of
csrc/fpfs_core.cuh compiled for the host with the kernel's transforms and summation order (tests/cpu/test_fpfs_core.cpp) against
the reference; the C ABI and the Python entry point validate without a device; the library holds k_fpfs, which does not spill.
GPU: the kernel against the reference on 4,096 stamps per kind, the PSF arguments, per-stamp independence from the batch, empty
batches, NaN rows, the caller's stream and shear recovery on rings."""
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
from oracle.fpfs import fpfs as reference

NPIX = 48 * 48
CSRC = os.path.join(ROOT, 'galaxy-deconv_b200', 'csrc')
NVCC = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'


# ---------------------------------------------------------------------------------------------------------------------
# inputs and gates
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


def elliptical_covariances(sig, e, th, g=(0.0, 0.0)):
    """covariances of Gaussians of size det^(1/4) = sig, distortion |e| at angle th, then sheared by g"""
    a2, b2 = sig ** 2 * ((1 + e) / (1 - e)).sqrt(), sig ** 2 * ((1 - e) / (1 + e)).sqrt()
    ct, st = th.cos(), th.sin()
    S = torch.stack([torch.stack([a2 * ct ** 2 + b2 * st ** 2, (a2 - b2) * ct * st], -1),
                     torch.stack([(a2 - b2) * ct * st, a2 * st ** 2 + b2 * ct ** 2], -1)], -2)
    A = shear_matrix(*g)
    return A @ S @ A.T


def gaussians(n=256, seed=5):
    """elliptical Gaussians: size 1.5-5 px, |e| <= 0.6, any orientation, centre within 1.5 px of (24, 24), flux 10-1e5 (fp32)"""
    gen = torch.Generator().manual_seed(seed)
    u = lambda: torch.rand(n, generator=gen, dtype=torch.float64)
    S = elliptical_covariances(1.5 + 3.5 * u(), 0.6 * u(), math.pi * u())
    mu = (24 + 3 * (u() - 0.5)[:, None, None], 24 + 3 * (u() - 0.5)[:, None, None])
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


def ensemble_shear(r):
    return (r['e'].double().sum(0) / r['R'].double().sum()).tolist()


def ell(r):
    return torch.cat([r['e'], r['R'][:, None]], 1).double().cpu()


def check_against_reference(got, ref, tol):
    """|de1|, |de2|, |dR| <= tol on every stamp; returns the maxima and medians"""
    d = (ell(got) - ell(ref)).abs()
    assert not d.isnan().any(), 'NaN where the reference has a number (or the reverse)'
    stats = dict(max=d.max(0).values.tolist(), median=d.median(0).values.tolist())
    assert d.max() <= tol, stats
    return stats


def _ref(x, psf=None, **kw):
    return reference(x.detach().cpu().double(), None if psf is None else psf.detach().cpu().double(), **kw)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference against analytic answers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('sigma', [2.0, 3.0, 4.0])
@pytest.mark.parametrize('sig_gal', [1.5, 3.0, 5.0])
def test_reference_response_is_the_shear_derivative(sig_gal, sigma):
    h = 1e-4
    S0 = (sig_gal ** 2 * torch.eye(2, dtype=torch.float64))[None]
    sheared = lambda g1, g2: reference(gaussian(shear_matrix(g1, g2) @ S0 @ shear_matrix(g1, g2).T), sigma=sigma)['e'][0]
    r = reference(gaussian(S0), sigma=sigma)
    R = float(r['R'][0])
    de1 = float(sheared(h, 0)[0] - sheared(-h, 0)[0]) / (2 * h)
    de2 = float(sheared(0, h)[1] - sheared(0, -h)[1]) / (2 * h)
    assert abs(R - de1) <= 1e-4 * abs(de1) and abs(R - de2) <= 1e-4 * abs(de2), (R, de1, de2)
    assert float(r['e'].abs().max()) <= 1e-9


def test_reference_sign_convention():
    t = lambda v: torch.tensor([v], dtype=torch.float64)
    x_long, y_long, diag = (reference(gaussian(elliptical_covariances(t(3.0), t(0.3), t(th)))) for th in (0.0, math.pi / 2, math.pi / 4))
    assert float(x_long['e'][0, 0]) > 0.05 and float(y_long['e'][0, 0]) < -0.05 and float(diag['e'][0, 1]) > 0.05


def test_reference_removes_the_psf():
    """a stamp convolved with a PSF and measured with it gives the modes of the unconvolved stamp measured with none"""
    idx = torch.arange(16)
    x = torch.cat([gaussians(8).double(), G.make_galaxy(idx[:8], 'cpu').double()])
    psf = unit_psfs(idx + 100)
    want = reference(x, sigma=3.5)
    got = reference(circular_convolve(x, psf), psf, sigma=3.5)
    rel = float(((got['modes'] - want['modes']).abs() / want['modes'][:, :1]).max())
    assert rel <= 1e-9, rel
    # the PSF's normalisation does not matter
    got16 = reference(circular_convolve(x, psf), psf / 16, sigma=3.5)
    assert float(((got16['modes'] - want['modes']).abs() / want['modes'][:, :1]).max()) <= 1e-9


@pytest.mark.parametrize('g', [(0.02, 0.0), (0.0, -0.01)])
def test_reference_recovers_shear_on_rings(g):
    x, psf = ring(g)
    got = ensemble_shear(_ref(x, psf))
    i = 0 if g[0] else 1
    assert abs(got[i] / g[i] - 1) <= 0.03 and abs(got[1 - i]) <= 1e-5, got


# ---------------------------------------------------------------------------------------------------------------------
# CPU: host-compiled core
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def host_core(tmp_path_factory):
    if not os.path.exists(NVCC):
        pytest.skip('nvcc not found')
    d = tmp_path_factory.mktemp('fpfs_core')
    exe = str(d / 'test_fpfs_core')
    r = subprocess.run([NVCC, '-O2', '-std=c++17', '-Wno-deprecated-gpu-targets', '-I', CSRC,
                        os.path.join(ROOT, 'tests', 'cpu', 'test_fpfs_core.cpp'), '-o', exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return exe, d


def run_host(host_core, stamps, psf=None, sigma=3.5, const=0.0):
    exe, d = host_core
    d = d / f'run{len(os.listdir(d))}'
    d.mkdir()
    stamps.detach().cpu().float().contiguous().numpy().tofile(d / 'stamps.f32')
    if psf is not None:
        psf.detach().cpu().float().contiguous().numpy().tofile(d / 'psf.f32')
    r = subprocess.run([exe, str(d), repr(float(sigma)), repr(float(const))], capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0 and r.stdout.strip().endswith('OK'), r.stdout[-2000:] + r.stderr[-2000:]
    modes = torch.from_numpy(np.fromfile(d / 'modes.f32', dtype=np.float32).reshape(-1, 6))
    e = torch.from_numpy(np.fromfile(d / 'ell.f32', dtype=np.float32).reshape(-1, 3))
    return dict(modes=modes, e=e[:, :2], R=e[:, 2])


@pytest.fixture(scope='module')
def synth_stamps():
    """512 gdsynth stamps: gt and psf (noise-free), obs at SNR 20, 100 and 300 with their PSFs"""
    b = {snr: G.make_batch(0, 512, snr) for snr in (20.0, 100.0, 300.0)}
    return dict(gt=b[100.0]['gt'], psf=b[100.0]['psf'], **{f'obs{int(s)}': b[s]['obs'] for s in b}, psf_of=b[100.0]['psf'])


@pytest.mark.parametrize('kind,with_psf', [('gaussians', False), ('gaussians', True), ('gt', False), ('psf', False), ('obs20', False),
                                           ('obs20', True), ('obs100', False), ('obs100', True), ('obs300', False), ('obs300', True)])
def test_host_core_matches_reference(host_core, synth_stamps, kind, with_psf):
    x = gaussians() if kind == 'gaussians' else synth_stamps[kind]
    psf = synth_stamps['psf_of'][:x.shape[0]] if with_psf else None
    print(f'\n{kind} psf={with_psf}:', check_against_reference(run_host(host_core, x, psf), _ref(x, psf), 1e-5))


def test_host_core_options(host_core, synth_stamps):
    """a broadcast PSF, another sigma and a non-zero const"""
    x, psf = synth_stamps['obs100'][:64], synth_stamps['psf_of'][:1]
    check_against_reference(run_host(host_core, x, psf), _ref(x, psf.expand(64, -1, -1, -1)), 1e-5)
    check_against_reference(run_host(host_core, x, sigma=2.5, const=1e6), _ref(x, sigma=2.5, const=1e6), 1e-5)


def test_nan_rows_host_core_and_reference(host_core):
    x = gaussians(3)
    x[1] = 0
    for got in (run_host(host_core, x), _ref(x)):
        bad = ell(got).isnan().any(1)
        assert bad.tolist() == [False, True, False], bad
        assert torch.equal(got['modes'][1].double(), torch.zeros(6, dtype=torch.float64))
    psf = G.make_batch(0, 3)['psf'].clone()
    psf[2] *= -1
    for got in (run_host(host_core, x, psf), _ref(x, psf)):
        assert ell(got).isnan().any(1).tolist() == [False, True, True]
        assert got['modes'].isnan().all(1).tolist() == [False, False, True]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: validation and build
# ---------------------------------------------------------------------------------------------------------------------
def test_fpfs_validates_without_a_device():
    from gdeconv import _lib
    lib = _lib.lib
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    cases = [  # (img, psf, psf_batch, batch, sigma, const, modes, ell)
        (p, None, 0, -1, 3.5, 0.0, p, p),
        (None, None, 0, 2, 3.5, 0.0, p, p),
        (p, None, 0, 2, 3.5, 0.0, p, None),
        (p, None, 1, 2, 3.5, 0.0, p, p),          # psf_batch without a psf
        (p, p, 0, 2, 3.5, 0.0, p, p),             # a psf without psf_batch
        (p, p, 3, 2, 3.5, 0.0, p, p),
        (p, p, 2, 3, 3.5, 0.0, p, p),
        (p, p, -1, 2, 3.5, 0.0, p, p),
        (p, None, 0, 0, 0.0, 0.0, p, p),
        (p, None, 0, 2, -1.0, 0.0, p, p),
        (p, None, 0, 2, float('nan'), 0.0, p, p),
        (p, None, 0, 2, float('inf'), 0.0, p, p),
        (p, None, 0, 2, 24.5, 0.0, p, p),
        (p, None, 0, 2, 3.5, -1.0, p, p),
        (p, None, 0, 2, 3.5, float('nan'), p, p),
        (p, None, 0, 2, 3.5, float('inf'), p, p),
    ]
    for case in cases:
        rc = lib.gd_fpfs(*case, None)
        assert rc == -1, (case, rc)                       # GD_EBADSHAPE
        assert b'gd_fpfs' in lib.gd_last_error(), 'gd_last_error() must explain the rejection'
    assert lib.gd_fpfs(None, None, 0, 0, 3.5, 0.0, None, None, None) == 0
    assert lib.gd_fpfs(None, p, 1, 0, 24.0, 0.0, None, None, None) == 0


def test_fpfs_rejects_cpu_tensors():
    from gdeconv import fpfs
    for t in (torch.rand(2, 1, 48, 48), torch.rand(2, 1, 48, 48, dtype=torch.float64), torch.rand(2, 48, 48)):
        with pytest.raises(RuntimeError, match='no CPU path'):
            fpfs(t)
    with pytest.raises(TypeError):
        fpfs(np.zeros((2, 1, 48, 48), np.float32))


def test_library_contains_the_fpfs_kernel():
    from gdeconv import _lib
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    sass = subprocess.run([cuobjdump, '-sass', _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert 'k_fpfs' in sass and 'sm_100a' in sass


def test_fpfs_kernel_does_not_spill(tmp_path):
    if not os.path.exists(NVCC):
        pytest.skip('nvcc not found')
    r = subprocess.run([NVCC, '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-std=c++17', '--expt-relaxed-constexpr', '-Xptxas', '-v',
                        '-c', os.path.join(CSRC, 'fpfs.cu'), '-o', str(tmp_path / 'fpfs.o')], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    m = re.search(r"Compiling entry function '\w*k_fpfs\w*'.*?(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                  r.stdout + r.stderr, re.S)
    assert m, (r.stdout + r.stderr)[-2000:]
    assert m.groups() == ('0', '0', '0'), m.group(0)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _gpu(x, psf=None, **kw):
    from gdeconv import fpfs
    return fpfs(x.reshape(-1, 1, 48, 48).cuda(), None if psf is None else psf.reshape(-1, 1, 48, 48).cuda(), **kw)


def _device_stamps(kind, snr, n=4096, start=30000):
    from gdeconv import make_batch_device
    from models.Wiener import Wiener
    b = make_batch_device(start, n, snr, device='cuda:0')
    if kind == 'wiener':
        return Wiener()(b['obs'], b['psf'], b['alpha']), None
    return b[kind], b['psf']


@pytest.mark.gpu
def test_kernel_matches_reference_on_gaussians():
    x = gaussians(4096)
    print('\ngaussians:', check_against_reference(_gpu(x), _ref(x), 1e-4))


@pytest.mark.gpu
@pytest.mark.parametrize('kind,snr,with_psf', [('gt', 100.0, False), ('obs', 20.0, True), ('obs', 20.0, False), ('obs', 100.0, True),
                                               ('obs', 100.0, False), ('obs', 300.0, True), ('obs', 300.0, False), ('wiener', 100.0, False)])
def test_kernel_matches_reference(kind, snr, with_psf):
    x, psf = _device_stamps(kind, snr)
    psf = psf if with_psf else None
    print(f'\n{kind} snr={snr} psf={with_psf}:', check_against_reference(_gpu(x, psf), _ref(x, psf), 1e-4))


def _bits(r, i=slice(None)):
    return torch.cat([r['modes'][i].reshape(-1), r['e'][i].reshape(-1), r['R'][i].reshape(-1)]).view(torch.int32)


@pytest.mark.gpu
def test_psf_arguments():
    from gdeconv import fpfs, make_batch_device
    b = make_batch_device(0, 300, 100.0, device='cuda:0')
    x, p1 = b['obs'], b['psf'][7:8]
    assert torch.equal(_bits(fpfs(x, p1)), _bits(fpfs(x, p1.expand(300, -1, -1, -1).contiguous())))
    assert torch.equal(_bits(fpfs(x, b['psf'])), _bits(fpfs(x, b['psf'], sigma=3.5, const=0.0)))
    assert torch.equal(_bits(fpfs(x)), _bits(fpfs(x, None, 3.5, 0.0)))
    with pytest.raises(ValueError):
        fpfs(x, b['psf'][:2])
    with pytest.raises(TypeError):
        fpfs(x, b['psf'].double())
    with pytest.raises(RuntimeError, match='no CPU path'):
        fpfs(x, b['psf'].cpu())
    with pytest.raises(RuntimeError, match='sigma'):
        fpfs(x, sigma=0.0)
    with pytest.raises(RuntimeError, match='const'):
        fpfs(x, const=-1.0)


@pytest.mark.gpu
def test_a_stamp_does_not_depend_on_its_batch():
    from gdeconv import fpfs, make_batch_device
    b = make_batch_device(0, 4096, 'mixed', device='cuda:0')
    x, psf = b['obs'], b['psf']
    for p in (None, psf):
        full = fpfs(x, p)
        one = fpfs(x[3000:3001], None if p is None else p[3000:3001])
        sub = fpfs(x[2990:3027], None if p is None else p[2990:3027])
        shifted = fpfs(torch.cat([x[:3], x[3000:3001], x[5:41]]), None if p is None else torch.cat([p[:3], p[3000:3001], p[5:41]]))
        want = _bits(full, 3000)
        assert torch.equal(_bits(one, 0), want) and torch.equal(_bits(sub, 10), want) and torch.equal(_bits(shifted, 3), want)
        assert sub['R'].shape == (37,) and not full['R'].isnan().any()


@pytest.mark.gpu
def test_empty_batch_and_nan_rows():
    from gdeconv import fpfs, launch_count, make_batch_device
    n0 = launch_count()
    for p in (None, torch.rand(1, 1, 48, 48, device='cuda:0'), torch.empty(0, 1, 48, 48, device='cuda:0')):
        got = fpfs(torch.empty(0, 1, 48, 48, device='cuda:0'), p)
        for k, s in dict(modes=(0, 6), e=(0, 2), R=(0,), g=(0, 2)).items():
            assert tuple(got[k].shape) == s and got[k].is_cuda, k
    assert launch_count() == n0
    b = make_batch_device(0, 40, 100.0, device='cuda:0')
    x = b['obs'].clone()
    x[17] = 0
    psf = b['psf'].clone()
    psf[23] *= -1
    got = fpfs(x)
    assert got['e'].isnan().any(1).nonzero().flatten().tolist() == [17] and got['R'].isnan().nonzero().flatten().tolist() == [17]
    assert not got['modes'].isnan().any() and float(got['modes'][17].abs().max()) == 0.0
    got = fpfs(x, psf)
    assert got['R'].isnan().nonzero().flatten().tolist() == [17, 23]
    assert got['modes'].isnan().all(1).nonzero().flatten().tolist() == [23]
    assert float(fpfs(x, const=1.0)['modes'][17].abs().max()) == 0.0 and not fpfs(x, const=1.0)['R'].isnan().any()


@pytest.mark.gpu
def test_runs_on_the_current_stream():
    """The input is written on a side stream after a delay; only that stream is synchronised: a kernel on any other stream
    would read the zeros that were there before."""
    from gdeconv import fpfs, make_batch_device
    b = make_batch_device(0, 4096, 100.0, device='cuda:0')
    want = fpfs(b['obs'], b['psf'])
    buf = torch.zeros_like(b['obs'])
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device='cuda:0')
    with torch.cuda.stream(s):
        torch.cuda._sleep(20_000_000)
        buf.copy_(b['obs'])
        got = fpfs(buf, b['psf'])
    s.synchronize()
    assert torch.equal(_bits(got), _bits(want))


@pytest.mark.gpu
@pytest.mark.parametrize('g', [(0.02, 0.0), (0.0, -0.01)])
def test_shear_recovery_on_rings(g):
    x, psf = ring(g)
    got, want = ensemble_shear(_gpu(x, psf)), ensemble_shear(_ref(x, psf))
    i = 0 if g[0] else 1
    print(f'\ng={g}: device {got}, reference {want}')
    assert max(abs(a - b) for a, b in zip(got, want)) <= 1e-5, (got, want)
    assert abs(got[i] / g[i] - 1) <= 0.03 and abs(got[1 - i]) <= 1e-5, got
