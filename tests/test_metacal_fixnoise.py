"""Fix-noise metacalibration (gd_metacal_fixnoise / gdeconv.metacal(noise_sigma=..., noise=...), csrc/metacal_fixnoise.cu) against
a float64 torch reference defined here on top of oracle/metacal.py: it rotates the noise literally with torch.rot90 and puts it
through oracle/metacal.py's metacal_images, so it reaches the images by another route than the kernel's folded spectrum.

CPU: the reference is linear in the noise and reduces to metacal_images without it; the folded spectrum of csrc/metacal_core.cuh,
written here in float64, equals the literal rot90 definition; the host build of the core (tests/cpu/test_metacal_fixnoise_core.cpp)
matches the reference and its generated field is gdsynth's hash; the C ABI and the Python entry point validate; the kernels
compile without spills (their 32-byte stack frame is cosf's large-argument reduction, as in k_synth).
GPU: the kernel against the reference, noise_sigma = 0 against gd_metacal, generated against caller noise, per-stamp
independence, edge cases, and the noise bias on rings of noisy galaxies."""
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
from oracle.adaptive_moments import OK, adaptive_moments
from oracle.metacal import PSF_FLOOR, SHEARS, STAMP, _grid, dtft, metacal as metacal_oracle, metacal_images, response
from test_metacal_device import check_against_reference, gaussian, gaussians, rel_l2

NPIX = 48 * 48
CSRC = os.path.join(ROOT, 'galaxy-deconv_b200', 'csrc')
NVCC = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
SIGMA = float(np.float32(G.SIGMA))
FIXNOISE_STREAM = 60                                  # streams 60 / 61 of gdsynth's counter hash


# ---------------------------------------------------------------------------------------------------------------------
# the fix-noise reference
# ---------------------------------------------------------------------------------------------------------------------
def fixnoise_field(start, count, seed, sigma):
    """the generated fix-noise fields of stamps start .. start + count - 1 -> fp32 [count,48,48]: sigma N(idx, p), N the standard
    normal of gdsynth._hashed_normal on streams 60 / 61; sigma a float or [1] / [count] (a non-finite sigma gives NaN)"""
    idx = torch.arange(int(start), int(start) + int(count), dtype=torch.int64)
    n = G._hashed_normal(idx, NPIX, FIXNOISE_STREAM, int(seed))
    s = torch.as_tensor(sigma, dtype=torch.float32).reshape(-1, 1).cpu()
    s = torch.where(s.isfinite(), s, torch.full_like(s, float('nan')))
    return (s * n).reshape(-1, STAMP, STAMP)


def fixnoise_images(noise, psf=None, delta=0.01, reconv_sigma=2.5):
    """rot90^-1(T_j(rot90(noise))) of noise [B,(1,)48,48] -> [B,5,48,48]: the term fix-noise adds to image j"""
    rot = torch.rot90(noise.reshape(-1, STAMP, STAMP), 1, dims=(-2, -1))
    return torch.rot90(metacal_images(rot, psf, delta, reconv_sigma), -1, dims=(-2, -1))


def reference(img, psf=None, delta=0.01, reconv_sigma=2.5, guess_sigma=3.0, noise=None):
    """oracle/metacal.py's metacal; with noise [B,(1,)48,48] (img's dtype and device) the fix-noise images
    T_j(img) + rot90^-1(T_j(rot90(noise))), measured and combined into R and g as oracle/metacal.py does"""
    if noise is None:
        return metacal_oracle(img, psf, delta, reconv_sigma, guess_sigma)
    ims = metacal_images(img, psf, delta, reconv_sigma)
    ims = ims + fixnoise_images(noise.to(ims.dtype), psf, delta, reconv_sigma)
    B = ims.shape[0]
    r = adaptive_moments(ims.reshape(-1, STAMP, STAMP), guess_sigma)
    e = r['e'].reshape(B, 5, 2)
    status, n_iter = r['status'].reshape(B, 5), r['n_iter'].reshape(B, 5)
    R = response(e, delta)
    e0, det = e[:, 0], R[:, 0, 0] * R[:, 1, 1] - R[:, 0, 1] * R[:, 1, 0]
    g = torch.stack([R[:, 1, 1] * e0[:, 0] - R[:, 0, 1] * e0[:, 1], R[:, 0, 0] * e0[:, 1] - R[:, 1, 0] * e0[:, 0]], 1) / det[:, None]
    g = torch.where((status == OK).all(1)[:, None], g, torch.full_like(g, float('nan')))
    return dict(images=ims, e=e, status=status, n_iter=n_iter, R=R, g=g)


def _psfs(kind, n):
    if kind is None:
        return None
    if kind == 'gaussian':
        s = torch.linspace(1.2, 2.5, n, dtype=torch.float64)
        return gaussian(torch.stack([torch.diag(torch.stack([a * a, 0.8 * a * a])) for a in s]))
    return G.make_psf(torch.arange(n), 'cpu').double()


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('psf_kind', [None, 'gdsynth'])
def test_reference_is_linear_in_the_noise(psf_kind):
    x = G.make_batch(0, 4, 100.0)['obs'].reshape(-1, 48, 48).double()
    psf = _psfs(psf_kind, 4)
    n = fixnoise_field(7, 4, 3, SIGMA).double()
    zero, plain = reference(x, psf, noise=torch.zeros_like(x)), metacal_oracle(x, psf)
    assert torch.equal(zero['images'], plain['images']) and torch.equal(zero['status'], plain['status'])
    both = reference(x, psf, noise=n)['images']
    parts = metacal_images(x, psf) + reference(torch.zeros_like(x), psf, noise=n)['images']
    assert float((both - parts).abs().max() / both.abs().max()) <= 1e-12


def folded(n, psf, delta, rs):
    """the fix-noise term of csrc/metacal_core.cuh in float64: FT = exp(i (kx + qy)) n~(A_j' k) F_j(R^-1 k), q = A_j R^-1 k"""
    u, v = _grid(n.device, n.dtype)
    w = 2 * math.pi / STAMP
    gam = torch.exp(-0.5 * rs ** 2 * w * w * (u * u + v * v))
    nyq = (u == -STAMP // 2) | (v == -STAMP // 2)
    sign = 1 - 2 * ((u + v).remainder(2))
    col = torch.arange(STAMP).view(1, STAMP).expand(STAMP, STAMP)
    row = torch.arange(STAMP).view(STAMP, 1).expand(STAMP, STAMP)
    outs = []
    for s in SHEARS:
        g1, g2 = delta * s[0], delta * s[1]
        F = gam.expand(n.shape[0], STAMP, STAMP).to(torch.complex128)
        if psf is not None:
            P = dtft(psf, (g1, g2)) / psf.sum((1, 2)).reshape(-1, 1, 1)
            bad = P.real ** 2 + P.imag ** 2 < PSF_FLOOR
            F = torch.where(bad, torch.zeros((), dtype=F.dtype), F / torch.where(bad, torch.ones((), dtype=P.dtype), P))
        F = torch.where(nyq, torch.zeros((), dtype=F.dtype), F)
        F_rot = F[:, (-col) % STAMP, row]                             # F_j(R^-1 k), R^-1 (u, v) = (v, -u)
        qy = w * (g2 * v - (1 - g1) * u) / math.sqrt(1 - g1 * g1 - g2 * g2)
        M = torch.exp(1j * (w * u + qy)) * dtft(n, (-g1, -g2)) * F_rot
        outs.append(torch.fft.ifft2(torch.where(nyq, torch.zeros((), dtype=M.dtype), M) * sign).real)
    return torch.stack(outs, 1)


@pytest.mark.parametrize('delta', [0.01, 0.1])
@pytest.mark.parametrize('psf_kind', [None, 'gaussian', 'gdsynth'])
def test_folded_formula_is_the_literal_rotation(psf_kind, delta):
    n = fixnoise_field(0, 4, 11, 1.0).double()
    psf = _psfs(psf_kind, 4)
    want = reference(torch.zeros_like(n), psf, delta, 1.5, noise=n)['images']
    got = folded(n, psf, delta, 1.5)
    err = float((got - want).abs().max() / want.abs().max())
    print(f'\npsf={psf_kind} delta={delta}: {err:.2e}')
    assert err <= 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# CPU: host-compiled core
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def host_core(tmp_path_factory):
    if not os.path.exists(NVCC):
        pytest.skip('nvcc not found')
    d = tmp_path_factory.mktemp('metacal_fixnoise_core')
    exe = str(d / 'test_metacal_fixnoise_core')
    r = subprocess.run([NVCC, '-O2', '-std=c++17', '-Wno-deprecated-gpu-targets', '-I', CSRC,
                        os.path.join(ROOT, 'tests', 'cpu', 'test_metacal_fixnoise_core.cpp'), '-o', exe], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return exe, d


def run_host(host_core, stamps, psf=None, sigma=None, noise=None, start=0, seed=0, delta=0.01, reconv_sigma=2.5):
    exe, d = host_core
    d = d / f'run{len(os.listdir(d))}'
    d.mkdir()
    stamps.detach().cpu().float().contiguous().numpy().tofile(d / 'stamps.f32')
    if psf is not None:
        psf.detach().cpu().float().contiguous().numpy().tofile(d / 'psf.f32')
    if noise is not None:
        noise.detach().cpu().float().contiguous().numpy().tofile(d / 'noise.f32')
    else:
        torch.as_tensor(sigma, dtype=torch.float32).reshape(-1).numpy().tofile(d / 'sigma.f32')
    r = subprocess.run([exe, str(d), repr(float(delta)), repr(float(reconv_sigma)), str(start), str(seed)], capture_output=True, text=True,
                       timeout=1200)
    assert r.returncode == 0 and r.stdout.strip().endswith('OK'), r.stdout[-2000:] + r.stderr[-2000:]
    ld = lambda name, *shape: torch.from_numpy(np.fromfile(d / name, dtype=np.float32).reshape(*shape))
    return ld('images.f32', -1, 5, 48, 48), ld('field.f32', -1, 48, 48), ld('uniform.f32', -1, 2, 64)


@pytest.fixture(scope='module')
def synth_stamps():
    b = {snr: G.make_batch(0, 24, snr) for snr in (20.0, 100.0, 300.0)}
    return dict(gt=b[100.0]['gt'], **{f'obs{int(s)}': b[s]['obs'] for s in b}, psf_of=b[100.0]['psf'])


@pytest.mark.parametrize('kind,with_psf', [('gaussians', False), ('gaussians', True), ('gt', False), ('gt', True), ('obs20', False),
                                           ('obs20', True), ('obs100', False), ('obs100', True), ('obs300', False), ('obs300', True)])
def test_host_core_matches_reference(host_core, synth_stamps, kind, with_psf):
    x = (gaussians(24) if kind == 'gaussians' else synth_stamps[kind]).reshape(-1, 48, 48)
    psf = synth_stamps['psf_of'][:x.shape[0]] if with_psf else None
    start, seed = 2 ** 31 + 5, 17
    got, field, uni = run_host(host_core, x, psf, sigma=SIGMA, start=start, seed=seed)
    want_field = fixnoise_field(start, x.shape[0], seed, SIGMA)
    assert float(rel_l2(field[:, None], want_field[:, None]).max()) <= 2e-6
    key = (torch.arange(start, start + x.shape[0], dtype=torch.int64)[:, None] * 4099 + torch.arange(64)).reshape(-1)
    for st in range(2):
        assert torch.equal(uni[:, st].reshape(-1).view(torch.int32), G.hashed_uniform(key, 60 + st, seed).view(torch.int32))
    want = reference(x.double(), None if psf is None else psf.double(), noise=field.double())['images']
    err = rel_l2(got, want)
    print(f'\n{kind} psf={with_psf}: rel-L2 max {float(err.max()):.3e} median {float(err.median()):.3e}')
    assert float(err.max()) <= 2e-6


def test_host_core_caller_noise_and_sigma_forms(host_core, synth_stamps):
    x, psf = synth_stamps['obs100'][:6].reshape(-1, 48, 48), synth_stamps['psf_of'][2:3]
    n = fixnoise_field(40, 6, 1, SIGMA)
    got, field, _ = run_host(host_core, x, psf, noise=n, delta=0.05, reconv_sigma=3.0)
    assert torch.equal(field, n)
    assert float(rel_l2(got, reference(x.double(), psf.double(), 0.05, 3.0, noise=n.double())['images']).max()) <= 2e-6
    a, _, _ = run_host(host_core, x, psf, sigma=SIGMA, start=40, seed=1)
    b, _, _ = run_host(host_core, x, psf.expand(6, -1, -1, -1), sigma=[SIGMA] * 6, start=40, seed=1)
    assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: validation and build
# ---------------------------------------------------------------------------------------------------------------------
def test_fixnoise_validates_without_a_device():
    from gdeconv import _lib
    lib = _lib.lib
    buf = (C.c_float * 16)()
    p = C.cast(buf, C.c_void_p)
    nan, inf = float('nan'), float('inf')
    ok = (p, None, 0, 2, 0.01, 2.5, 3.0, None, p, 1, 0, 0, p, p, p)

    def case(**kw):
        names = ('img', 'psf', 'psf_batch', 'batch', 'delta', 'rs', 'gs', 'noise', 'sigma', 'sigma_batch', 'start', 'seed', 'images',
                 'shape', 'info')
        return tuple(kw.get(k, v) for k, v in zip(names, ok))

    cases = [case(batch=-1), case(img=None), case(shape=None), case(info=None), case(psf_batch=1), case(psf=p),
             case(psf=p, psf_batch=3), case(psf=p, psf_batch=-1),
             case(noise=p), case(sigma=None), case(noise=p, sigma=None, sigma_batch=1), case(sigma_batch=0), case(sigma_batch=3),
             case(sigma_batch=-1), case(start=-1), case(start=2 ** 63 - 1)] \
        + [case(delta=d) for d in (0.0, -0.01, 0.1001, nan, inf)] + [case(rs=s) for s in (0.0, 24.5, nan)] \
        + [case(gs=s) for s in (0.0, 24.5, inf)]
    for c in cases:
        rc = lib.gd_metacal_fixnoise(*c, None)
        assert rc == -1, (c, rc)                          # GD_EBADSHAPE
        assert b'gd_metacal_fixnoise' in lib.gd_last_error(), 'gd_last_error() must explain the rejection'
    assert lib.gd_metacal_fixnoise(*case(batch=0, img=None), None) == 0
    assert lib.gd_metacal_fixnoise(*case(batch=0, img=None, noise=p, sigma=None, sigma_batch=0, start=2 ** 63 - 1), None) == 0
    assert lib.gd_metacal_fixnoise(*case(batch=0, img=None, psf=p, psf_batch=1), None) == 0


def test_metacal_rejects_bad_noise_arguments_on_the_host():
    from gdeconv import metacal
    x = torch.rand(2, 1, 48, 48)
    with pytest.raises(ValueError, match='not both'):
        metacal(x, noise=torch.zeros(2, 1, 48, 48), noise_sigma=1.0)
    with pytest.raises(RuntimeError, match='no CPU path'):
        metacal(x, noise_sigma=1.0)


def test_fixnoise_kernels_compile_without_spills(tmp_path):
    if not os.path.exists(NVCC):
        pytest.skip('nvcc not found')
    r = subprocess.run([NVCC, '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-std=c++17', '--expt-relaxed-constexpr', '-Xptxas', '-v',
                        '-c', os.path.join(CSRC, 'metacal_fixnoise.cu'), '-o', str(tmp_path / 'metacal_fixnoise.o')], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    log = r.stdout + r.stderr
    found = re.findall(r"Compiling entry function '(\w*k_metacal_fixnoise\w*)'.*?(\d+) bytes spill stores, (\d+) bytes spill loads\s*"
                       r"ptxas info\s*: Used (\d+) registers", log, re.S)
    assert len(found) == 3, log[-3000:]                   # no PSF, one PSF, a PSF per stamp
    for name, st, ld, regs in found:
        assert (st, ld) == ('0', '0') and int(regs) <= 128, (name, st, ld, regs)
    # shared memory with a PSF: 5 planes of 24 x 50 float2, the stamp and the PSF / noise slot, the [5][1105] factor table;
    # two CTAs of it fit in an SM's 228 KB less 1 KB reserved per CTA
    assert 5 * 24 * 50 * 8 + 2 * NPIX * 4 + 5 * 1105 * 8 <= (228 * 1024 - 2 * 1024) // 2


def test_library_contains_the_fixnoise_kernels():
    from gdeconv import _lib
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    sass = subprocess.run([cuobjdump, '-sass', _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert len(set(re.findall(r'Function : (\w*k_metacal_fixnoise\w*)', sass))) == 3 and 'sm_100a' in sass


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _bits(r, i=slice(None)):
    return torch.cat([r['e'][i].reshape(-1).view(torch.int32), r['status'][i].reshape(-1), r['n_iter'][i].reshape(-1),
                      r['images'][i].reshape(-1).view(torch.int32)])


def _kind(kind, snr, n=2048, start=30000):
    """(stamps [n,1,48,48], PSF or None, fix-noise keyword arguments, the reference's noise [n,48,48])"""
    from gdeconv import make_batch_device
    from models.Wiener import Wiener
    b = make_batch_device(start, n, snr, device='cuda:0')
    if kind == 'wiener':
        nz = Wiener()(SIGMA * torch.randn(n, 1, 48, 48, device='cuda:0', generator=torch.Generator('cuda:0').manual_seed(3)),
                      b['psf'], b['alpha'])
        return Wiener()(b['obs'], b['psf'], b['alpha']), None, dict(noise=nz), nz.reshape(-1, 48, 48)
    if kind == 'gaussians':
        x, psf, sigma = gaussians(n).reshape(-1, 1, 48, 48).cuda(), None, 1.0
    else:
        x, psf, sigma = b[kind], b['psf'], SIGMA
    return x, psf, dict(noise_sigma=sigma, start=start, seed=5), fixnoise_field(start, n, 5, sigma)


@pytest.mark.gpu
@pytest.mark.parametrize('kind,snr,with_psf', [('gaussians', 100.0, False), ('gt', 100.0, False), ('obs', 20.0, True), ('obs', 100.0, True),
                                               ('obs', 300.0, True), ('wiener', 100.0, False)])
def test_kernel_matches_reference(kind, snr, with_psf):
    from gdeconv import metacal
    x, psf, kw, n = _kind(kind, snr)
    psf = psf if with_psf else None
    got = metacal(x, psf, images=True, **kw)
    want = reference(x.double().reshape(-1, 48, 48), None if psf is None else psf.double(), noise=n.cuda().double())
    want = {k: v.cpu() for k, v in want.items()}
    print(f'\n{kind} snr={snr} psf={with_psf} {sorted(kw)}:', check_against_reference(got, want, psf))


@pytest.mark.gpu
def test_zero_sigma_is_gd_metacal():
    from gdeconv import metacal, make_batch_device
    b = make_batch_device(0, 600, 'mixed', device='cuda:0')
    for p in (None, b['psf'][:1], b['psf']):
        a, z = metacal(b['obs'], p, images=True), metacal(b['obs'], p, images=True, noise_sigma=0.0)
        assert torch.equal(a['e'].view(torch.int32), z['e'].view(torch.int32)) and torch.equal(a['status'], z['status'])
        assert torch.equal(a['n_iter'], z['n_iter']) and torch.equal(a['images'], z['images'])


@pytest.mark.gpu
def test_generated_noise_is_the_reference_field():
    from gdeconv import metacal, make_batch_device
    b = make_batch_device(100, 1000, 50.0, device='cuda:0')
    s, sd = 2 ** 31 + 11, 123
    n = fixnoise_field(s, 1000, sd, SIGMA).reshape(-1, 1, 48, 48).cuda()
    for p in (None, b['psf']):
        gen = metacal(b['obs'], p, images=True, noise_sigma=SIGMA, start=s, seed=sd)
        cal = metacal(b['obs'], p, images=True, noise=n)
        assert float(rel_l2(gen['images'].reshape(-1, 5, NPIX).cpu(), cal['images'].reshape(-1, 5, NPIX).cpu()).max()) <= 1e-6
        assert torch.equal(gen['status'], cal['status'])
        neg = metacal(b['obs'], p, images=True, noise_sigma=-SIGMA, start=s, seed=sd)
        cal = metacal(b['obs'], p, images=True, noise=-n)
        assert float(rel_l2(neg['images'].reshape(-1, 5, NPIX).cpu(), cal['images'].reshape(-1, 5, NPIX).cpu()).max()) <= 1e-6
        assert torch.equal(neg['status'], cal['status'])


@pytest.mark.gpu
def test_a_stamp_does_not_depend_on_its_batch_offset_or_argument_forms():
    from gdeconv import metacal, make_batch_device
    b = make_batch_device(0, 1200, 'mixed', device='cuda:0')
    x, psf = b['obs'], b['psf']
    sig = SIGMA * (0.5 + torch.rand(1200, device='cuda:0'))
    for s0 in (0, 2 ** 31 - 500, 2 ** 40):
        for p in (None, psf):
            full = metacal(x, p, images=True, noise_sigma=sig, start=s0, seed=9)
            for i in (0, 600, 1000):
                one = metacal(x[i:i + 1], None if p is None else p[i:i + 1], images=True, noise_sigma=sig[i:i + 1], start=s0 + i, seed=9)
                assert torch.equal(_bits(one, 0), _bits(full, i)), (s0, i)
    p1 = psf[7:8]
    a = metacal(x[:300], p1, images=True, noise_sigma=SIGMA, start=5, seed=2)
    assert torch.equal(_bits(a), _bits(metacal(x[:300], p1.expand(300, -1, -1, -1).contiguous(), images=True, noise_sigma=SIGMA, start=5, seed=2)))
    assert torch.equal(_bits(a), _bits(metacal(x[:300], p1, images=True, noise_sigma=torch.full((300,), SIGMA, device='cuda:0'), start=5, seed=2)))
    assert torch.equal(_bits(a), _bits(metacal(x[:300], p1, images=True, noise_sigma=torch.full((1,), SIGMA, device='cuda:0'), start=5, seed=2)))
    n = torch.randn(300, 1, 48, 48, device='cuda:0')
    a = metacal(x[:300], psf[:300], images=True, noise=n)
    assert torch.equal(_bits(a, 200), _bits(metacal(x[200:201], psf[200:201], images=True, noise=n[200:201]), 0))
    for bad in (dict(noise=n[:2]), dict(noise=n.double()), dict(noise=n.cpu()), dict(noise_sigma=sig[:2]), dict(noise_sigma=sig.double()),
                dict(noise_sigma=sig.cpu()), dict(noise_sigma=sig[:300, None])):
        with pytest.raises((ValueError, TypeError, RuntimeError)):
            metacal(x[:300], noise_sigma=bad.get('noise_sigma'), noise=bad.get('noise'))
    with pytest.raises(RuntimeError, match='out of range'):
        metacal(x[:3], noise_sigma=1.0, start=-1)


@pytest.mark.gpu
def test_empty_batch_nan_stamp_nan_sigma_and_stream():
    from gdeconv import launch_count, metacal, make_batch_device
    n0 = launch_count()
    for kw in (dict(noise_sigma=1.0), dict(noise=torch.empty(0, 1, 48, 48, device='cuda:0'))):
        got = metacal(torch.empty(0, 1, 48, 48, device='cuda:0'), None, images=True, **kw)
        assert tuple(got['images'].shape) == (0, 5, 1, 48, 48) and tuple(got['g'].shape) == (0, 2)
    assert launch_count() == n0
    b = make_batch_device(0, 40, 100.0, device='cuda:0')
    sig = torch.full((40,), SIGMA, device='cuda:0')
    for p in (None, b['psf']):
        want = metacal(b['obs'], p, images=True, noise_sigma=sig, seed=4)
        keep = torch.arange(40, device='cuda:0') != 17
        x = b['obs'].clone()
        x[17, 0, 5, 9] = float('nan')
        got = metacal(x, p, images=True, noise_sigma=sig, seed=4)
        assert (got['status'][17] == 2).all() and got['g'][17].isnan().all()          # GD_SHAPE_FLUX
        assert torch.equal(_bits(got, keep), _bits(want, keep))
        for bad in (float('nan'), float('inf')):
            s = sig.clone()
            s[17] = bad
            got = metacal(b['obs'], p, images=True, noise_sigma=s, seed=4)
            assert (got['status'][17] == 2).all() and got['images'][17].isnan().all()
            assert torch.equal(_bits(got, keep), _bits(want, keep))
    big = make_batch_device(0, 2048, 100.0, device='cuda:0')
    want = metacal(big['obs'], big['psf'], images=True, noise_sigma=SIGMA)
    buf = torch.zeros_like(big['obs'])
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device='cuda:0')
    with torch.cuda.stream(s):
        torch.cuda._sleep(20_000_000)
        buf.copy_(big['obs'])
        got = metacal(buf, big['psf'], images=True, noise_sigma=SIGMA)
    s.synchronize()
    assert torch.equal(_bits(got), _bits(want))


# ---------------------------------------------------------------------------------------------------------------------
# GPU: noise bias on rings
# ---------------------------------------------------------------------------------------------------------------------
def noisy_ring_sums(g, n_rings, snr=50.0, chunk=4096, seed=0):
    """Per ring group (4 orientations x obs noise +-n x fix-noise +-n'), the sums of e(noshear) [G,2] and R [G,2,2] with and
    without fix-noise, and whether every image of the group is OK: dict(fix=(e, R, ok), nofix=(e, R, ok)).  The rings are those
    of test_metacal_device.ring (elliptical Gaussians of size 2-4 px, |e| <= 0.5, sheared by g, convolved with gdsynth PSFs),
    scaled to the SNR of gdsynth (sqrt(sum gal^2) = SNR sigma before the PSF), built on the device in chunks."""
    from gdeconv import metacal
    dev = torch.device('cuda:0')
    gen = torch.Generator(device=dev).manual_seed(seed)
    out = {k: ([], [], []) for k in ('fix', 'nofix')}
    rot = torch.arange(4, dtype=torch.float64, device=dev) * (math.pi / 4)
    y, x = torch.meshgrid(torch.arange(48, dtype=torch.float64, device=dev), torch.arange(48, dtype=torch.float64, device=dev), indexing='ij')
    A = torch.tensor([[1 + g[0], g[1]], [g[1], 1 - g[0]]], dtype=torch.float64, device=dev)
    for c0 in range(0, n_rings, chunk):
        m = min(chunk, n_rings - c0)
        u = lambda: torch.rand(m, generator=gen, device=dev, dtype=torch.float64)
        sig, e, th = 2 + 2 * u(), 0.5 * u(), math.pi * u()
        a2, b2 = sig ** 2 * ((1 + e) / (1 - e)).sqrt(), sig ** 2 * ((1 - e) / (1 + e)).sqrt()
        t = (th[:, None] + rot).flatten()
        a2, b2 = a2.repeat_interleave(4), b2.repeat_interleave(4)
        ct, st = t.cos(), t.sin()
        S = torch.stack([torch.stack([a2 * ct ** 2 + b2 * st ** 2, (a2 - b2) * ct * st], -1),
                         torch.stack([(a2 - b2) * ct * st, a2 * st ** 2 + b2 * ct ** 2], -1)], -2)
        S = A @ S @ A.T
        Si = torch.linalg.inv(S)
        dx, dy = x - 24, y - 24
        q = Si[:, 0, 0, None, None] * dx * dx + 2 * Si[:, 0, 1, None, None] * dx * dy + Si[:, 1, 1, None, None] * dy * dy
        gal = torch.exp(-0.5 * q)
        gal = gal * (snr * SIGMA / gal.flatten(1).norm(dim=1))[:, None, None]
        idx = 4 * (c0 + torch.arange(m, device=dev)).repeat_interleave(4) + torch.arange(4, device=dev).repeat(m)
        psf = G.make_psf(idx.cpu(), 'cpu').to(dev).double()
        psf = psf / psf.sum((1, 2), keepdim=True)
        stamp = torch.fft.ifft2(torch.fft.fft2(gal) * torch.fft.fft2(torch.roll(psf, (-24, -24), (-2, -1)))).real
        n = SIGMA * torch.randn(4 * m, 48, 48, generator=gen, device=dev, dtype=torch.float64)
        p32 = psf.float().reshape(-1, 1, 48, 48)
        for key, calls in (('nofix', [(1, None)]), ('fix', [(1, SIGMA), (1, -SIGMA)])):
            es, Rs, oks = [], [], []
            for sn in (1, -1):
                obs = (stamp + sn * n).float().reshape(-1, 1, 48, 48)
                for _, s in calls:
                    kw = {} if s is None else dict(noise_sigma=s, start=4 * c0, seed=seed + 1)
                    r = metacal(obs, p32, **kw)
                    es.append(r['e'][:, 0].double())
                    Rs.append(r['R'].double())
                    oks.append((r['status'] == OK).all(1))
            ok = torch.stack(oks).all(0).reshape(m, 4).all(1)
            e_sum = torch.stack(es).nan_to_num().sum(0).reshape(m, 4, 2).sum(1)
            R_sum = torch.stack(Rs).nan_to_num().sum(0).reshape(m, 4, 2, 2).sum(1)
            out[key][0].append(e_sum)
            out[key][1].append(R_sum)
            out[key][2].append(ok)
    return {k: tuple(torch.cat(v) for v in vals) for k, vals in out.items()}


def jackknife_shear(e, R, ok):
    """ensemble shear <R>^-1 <e> over the kept groups and its delete-one-group estimates -> (g [2], g_i [G,2])"""
    e, R = e[ok], R[ok]
    E, Rt = e.sum(0), R.sum(0)
    g = torch.linalg.solve(Rt, E)
    gi = torch.linalg.solve(Rt[None] - R, (E[None] - e)[..., None])[..., 0]
    return g, gi


def jackknife_sigma(vals):
    G_ = vals.shape[0]
    return ((G_ - 1) / G_ * (vals - vals.mean(0)).pow(2).sum(0)).sqrt()


def noise_bias(n_rings, g_true=(0.02, -0.01), seed=0):
    """m (projected on g_true) and c with their jackknife errors, with and without fix-noise"""
    gt = torch.tensor(g_true, dtype=torch.float64, device='cuda:0')
    sheared, null = noisy_ring_sums(g_true, n_rings, seed=seed), noisy_ring_sums((0.0, 0.0), n_rings, seed=seed + 100)
    res = {}
    for k in ('fix', 'nofix'):
        g, gi = jackknife_shear(*sheared[k])
        m, mi = (g @ gt) / (gt @ gt) - 1, (gi @ gt) / (gt @ gt) - 1
        c, ci = jackknife_shear(*null[k])
        res[k] = dict(m=float(m), sigma_m=float(jackknife_sigma(mi)), c=c.tolist(), sigma_c=jackknife_sigma(ci).tolist(),
                      groups=int(sheared[k][2].sum()), groups_null=int(null[k][2].sum()), n_rings=n_rings)
    return res


@pytest.mark.gpu
def test_fixnoise_removes_the_noise_bias_on_rings():
    res = noise_bias(20000)
    print(f"\nSNR 50 rings: fix-noise m = {res['fix']['m']:+.2e} +- {res['fix']['sigma_m']:.1e}, c = {res['fix']['c']}; "
          f"without: m = {res['nofix']['m']:+.2e} +- {res['nofix']['sigma_m']:.1e}, c = {res['nofix']['c']}  {res}")
    f = res['fix']
    assert f['groups'] >= 0.9 * f['n_rings'] and f['groups_null'] >= 0.9 * f['n_rings'], res
    assert abs(f['m']) <= 3 * f['sigma_m'] + 1e-3, res
    assert all(abs(c) <= 3 * s for c, s in zip(f['c'], f['sigma_c'])), res
