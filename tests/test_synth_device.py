"""The on-device stamp generator (gd_synth_batch / gdeconv.make_batch_device, csrc/synth.cu) against gdsynth.make_batch.

CPU: the scalar core (csrc/synth_core.cuh) compiled for the host (tests/cpu/test_synth_core.cpp) must reproduce gdsynth's
hash bit for bit, its per-stamp draws exactly and its stamps to fp32 rounding; the C ABI validates without a device.
GPU: parity of every output with gdsynth on the CPU (the fp32 reference), per-index determinism, partial outputs."""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_l2

import gdsynth as G

SEEDS = (0, 31415, 2 ** 31 + 5, -7)
STREAMS = (0, 10, 11, 12, 13, 20, 21, 22, 23, 24, 25, 26, 30, 40, 41, 50, 51)
STAMP_TOL = 2e-6


# ---------------------------------------------------------------------------------------------------------------------
# CPU: host-compiled core
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def host_core(tmp_path_factory):
    nvcc = shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    if not os.path.exists(nvcc):
        pytest.skip('nvcc not found')
    d = tmp_path_factory.mktemp('synth_core')
    exe = str(d / 'test_synth_core')
    # -ffp-contract=off: one rounding per operation, as torch evaluates gdsynth's expressions (the device code uses __fmul_rn & co.)
    r = subprocess.run([nvcc, '-O1', '-std=c++17', '-Wno-deprecated-gpu-targets', '-Xcompiler', '-ffp-contract=off',
                        '-I', os.path.join(ROOT, 'galaxy-deconv_b200', 'csrc'), os.path.join(ROOT, 'tests', 'cpu', 'test_synth_core.cpp'),
                        '-o', exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return exe, d


def _idx_sample():
    g = torch.Generator().manual_seed(5)
    return torch.cat([torch.arange(0, 16), torch.arange(2 ** 31 - 4, 2 ** 31 + 4), torch.arange(2 ** 40 - 4, 2 ** 40 + 4),
                      torch.randint(0, 2 ** 62, (32,), generator=g)]).to(torch.int64)


def _run_core(host_core, seed, snr, fwhm_err, shear_err, index):
    exe, d = host_core
    d = d / f'run_{seed}_{snr}_{fwhm_err}_{shear_err}'
    d.mkdir()
    idx = _idx_sample()
    triples = torch.stack([torch.stack([idx, torch.full_like(idx, s), torch.full_like(idx, sd)], 1) for s in STREAMS for sd in SEEDS]).reshape(-1, 3)
    triples.numpy().tofile(d / 'triples.i64')
    index.numpy().astype(np.int64).tofile(d / 'index.i64')
    r = subprocess.run([exe, str(d), str(seed), str(-1.0 if snr == 'mixed' else snr), repr(fwhm_err), repr(shear_err)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith('OK'), r.stdout[-2000:] + r.stderr[-2000:]
    ld = lambda name, *shape: torch.from_numpy(np.fromfile(d / name, dtype=np.float32).reshape(*shape))
    M = index.numel()
    return dict(triples=triples, uniform=ld('uniform.f32', -1), gal_params=ld('gal_params.f32', M, 9), psf_params=ld('psf_params.f32', M, 13),
                galaxy=ld('galaxy.f32', M, 48, 48), psf=ld('psf.f32', M, 48, 48), model_psf=ld('model_psf.f32', M, 48, 48),
                gt=ld('gt.f32', M, 48, 48), obs=ld('obs.f32', M, 48, 48), alpha=ld('alpha.f32', M))


def test_hashed_uniform_is_bit_identical(host_core):
    out = _run_core(host_core, G.REF_SEED, 100.0, 0.0, 0.0, torch.arange(0, 1))
    t, got = out['triples'], out['uniform']
    assert t.shape[0] >= 4000
    want = torch.empty_like(got)
    n = _idx_sample().numel()
    k = 0
    for s in STREAMS:
        for sd in SEEDS:
            want[k:k + n] = G.hashed_uniform(t[k:k + n, 0], s, sd)
            k += n
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))


# 16 stamps near 1000 and 16 past 2^31, mixed SNR, both PSF errors: every draw and every stage of the pipeline
CORE_RANGES = ((1000, 16), (2 ** 31 + 3, 16))
FWHM_ERR, SHEAR_ERR = 0.05, 0.03


@pytest.fixture(scope='module')
def core_run(host_core):
    index = torch.cat([torch.arange(a, a + n) for a, n in CORE_RANGES])
    return index, _run_core(host_core, 31415, 'mixed', FWHM_ERR, SHEAR_ERR, index)


def test_per_stamp_parameters_match_gdsynth(core_run):
    idx, out = core_run
    seed = 31415
    u = lambda s: G.hashed_uniform(idx, s, seed)
    gp, pp = out['gal_params'], out['psf_params']
    # galaxy draws (streams 20-26) and the arithmetic on them: exact
    is_gauss = u(20) < 0.5
    n = torch.where(is_gauss, torch.full_like(u(20), 0.5), 0.5 + 3.5 * u(21))
    e = 0.6 * u(23)
    want = [n, 1.5 + 4.5 * u(22), e, math.pi * u(24), 2.0 * u(25) - 1.0, 2.0 * u(26) - 1.0, is_gauss.float(), (1 - e) / (1 + e),
            2.0 * n - 1.0 / 3.0 + 4.0 / (405.0 * n)]
    for j, w in enumerate(want):
        assert torch.equal(gp[:, j], w), f'galaxy parameter {j}'
    assert 0 < int(is_gauss.sum()) < idx.numel()
    # PSF draws (streams 10-13), mismatch signs (50 / 51) and the model FWHM: exact
    sg = torch.where(u(50) < 0.5, -1.0, 1.0)
    sg2 = torch.where(u(51) < 0.5, -1.0, 1.0)
    fwhm = 2.25 + 2.5 * u(11)
    for j, w in ((0, 2.5 + 2.0 * u(10)), (1, fwhm), (2, 0.01 + 0.02 * u(12)), (3, math.pi * u(13)), (7, fwhm + sg * FWHM_ERR / 0.2),
                 (8, sg), (9, sg2)):
        assert torch.equal(pp[:, j], w), f'psf parameter {j}'
    assert 0 < int((sg > 0).sum()) < idx.numel() and 0 < int((sg2 > 0).sum()) < idx.numel()
    # through transcendentals (cos, sin, atan2, pow, exp): ulp-level
    beta, th0, e0 = pp[:, 0], pp[:, 3], pp[:, 2]
    for j, (sh1, sh2) in ((4, (0.0, 0.0)), (10, (sg * SHEAR_ERR, sg2 * SHEAR_ERR))):
        e1, e2 = e0 * torch.cos(2 * th0) + sh1, e0 * torch.sin(2 * th0) + sh2
        torch.testing.assert_close(pp[:, j], torch.sqrt(e1 * e1 + e2 * e2).clamp(1e-6, 0.9), rtol=1e-6, atol=0)
        torch.testing.assert_close(pp[:, j + 1], 0.5 * torch.atan2(e2, e1), rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(pp[:, 6], fwhm / (2.0 * torch.sqrt(torch.pow(2.0, 1.0 / beta) - 1.0)), rtol=2e-6, atol=0)
    snr = torch.exp(math.log(20.0) + (math.log(300.0) - math.log(20.0)) * u(30))
    torch.testing.assert_close(pp[:, 12], snr, rtol=1e-6, atol=0)


def _reference(ranges, snr, **kw):
    parts = [G.make_batch(a, n, snr, **kw) for a, n in ranges]
    return {k: torch.cat([p[k] for p in parts]) for k in parts[0]}


def test_rendered_stamps_match_gdsynth(core_run):
    idx, out = core_run
    seed = 31415
    assert float(rel_l2(out['galaxy'], G.make_galaxy(idx, 'cpu', seed)).max()) <= STAMP_TOL
    assert float(rel_l2(out['psf'], G.make_psf(idx, 'cpu', seed)).max()) <= STAMP_TOL
    sg = torch.where(G.hashed_uniform(idx, 50, seed) < 0.5, -1.0, 1.0).view(-1, 1, 1)
    sg2 = torch.where(G.hashed_uniform(idx, 51, seed) < 0.5, -1.0, 1.0).view(-1, 1, 1)
    model = G.make_psf(idx, 'cpu', seed, fwhm_delta=sg * FWHM_ERR, shear=(sg * SHEAR_ERR, sg2 * SHEAR_ERR))
    assert float(rel_l2(out['model_psf'], model).max()) <= STAMP_TOL
    # the whole per-stamp pipeline (flux scale, 96x96 transforms with the PSF-centre shift, noise, alpha) on the host
    ref = _reference(CORE_RANGES, 'mixed', seed=seed, psf_fwhm_err=FWHM_ERR, psf_shear_err=SHEAR_ERR)
    assert float(rel_l2(out['gt'], ref['gt'][:, 0]).max()) <= STAMP_TOL
    assert float(rel_l2(out['obs'], ref['obs'][:, 0]).max()) <= STAMP_TOL
    a_ref = ref['alpha'].flatten()
    rms = ref['obs'].flatten(1).pow(2).mean(1).sqrt()
    assert bool(((out['alpha'] - a_ref).abs() <= 2e-6 * torch.maximum(a_ref.abs(), rms)).all())


def test_synth_batch_validates_without_a_device():
    from gdeconv import _lib
    lib = _lib.lib
    buf = (C.c_float * 4)()
    p = C.cast(buf, C.c_void_p)
    cases = [  # (start, count, snr_mode, snr, outputs)
        (0, -1, 0, 100.0, (p, p, p, p)),
        (0, 0, 0, 100.0, (None, None, None, None)),
        (0, 0, 7, 100.0, (p, None, None, None)),
        (0, 0, 0, 0.0, (None, p, None, None)),
        (0, 0, 0, -3.0, (None, None, p, None)),
        (-1, 0, 1, 0.0, (None, None, None, p)),
    ]
    for start, count, mode, snr, outs in cases:
        lib.gd_last_error()
        rc = lib.gd_synth_batch(start, count, 31415, mode, snr, 0.0, 0.0, *outs, None)
        assert rc == -1, (start, count, mode, snr, rc)             # GD_EBADSHAPE
        assert lib.gd_last_error(), 'gd_last_error() must explain the rejection'


def test_make_batch_device_rejects_cpu_and_bad_arguments():
    from gdeconv import make_batch_device
    with pytest.raises(RuntimeError, match='CUDA'):
        make_batch_device(0, 4, device='cpu')
    with pytest.raises(ValueError):
        make_batch_device(0, 4, keys=('obs', 'noise'), device='cpu')
    with pytest.raises(TypeError):
        make_batch_device(0, 4, keys='psf', device='cpu')


def test_library_contains_the_native_generator():
    """k_synth is compiled into the shipped .so for sm_100a."""
    from gdeconv import _lib
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not available')
    sass = subprocess.run([cuobjdump, '-sass', _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert 'k_synth' in sass and 'sm_100a' in sass


def test_gdsynth_stays_free_of_gdeconv():
    """bench.py's reference arm imports gdsynth without mapping libgdeconv.so."""
    import sys
    code = 'import sys, gdsynth; assert not [m for m in sys.modules if m.startswith("gdeconv")]'
    r = subprocess.run([sys.executable, '-c', code], cwd=os.path.join(ROOT, 'galaxy-deconv_b200'), capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
PARITY_CASES = [(100.0, 0.0, 0.0), (20.0, 0.0, 0.0), (300.0, 0.0, 0.0), ('mixed', 0.0, 0.0), (100.0, 0.05, 0.0), (100.0, 0.0, 0.03)]


@pytest.mark.gpu
@pytest.mark.parametrize('snr,fwhm_err,shear_err', PARITY_CASES)
def test_parity_with_gdsynth(snr, fwhm_err, shear_err):
    from gdeconv import make_batch_device, moments_e
    start, B = 7000, 256
    ref = G.make_batch(start, B, snr, psf_fwhm_err=fwhm_err, psf_shear_err=shear_err)
    got = make_batch_device(start, B, snr, device='cuda:0', psf_fwhm_err=fwhm_err, psf_shear_err=shear_err)
    for k in ('obs', 'psf', 'gt', 'alpha'):
        assert got[k].shape == ref[k].shape and got[k].dtype == torch.float32 and got[k].is_cuda, k
    got = {k: v.cpu() for k, v in got.items()}
    for k in ('obs', 'psf', 'gt'):
        err = float(rel_l2(got[k], ref[k]).max())
        assert err <= STAMP_TOL, (k, err)
    a_ref, a = ref['alpha'].flatten(), got['alpha'].flatten()
    rms = ref['obs'].flatten(1).pow(2).mean(1).sqrt()
    bound = 2e-6 * torch.maximum(a_ref.abs(), rms)
    assert bool(((a - a_ref).abs() <= bound).all()), float(((a - a_ref).abs() / bound).max())
    e_got = moments_e(got['gt'].cuda()).cpu()
    e_ref = moments_e(ref['gt'].cuda()).cpu()
    assert float((e_got - e_ref).abs().max()) <= 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize('base', [0, 2 ** 31 - 100, 3 * 2 ** 40])
def test_stamps_depend_only_on_their_index(base):
    from gdeconv import make_batch_device
    full = make_batch_device(base, 1000, 'mixed', device='cuda:0')
    part = make_batch_device(base + 300, 400, 'mixed', device='cuda:0')
    for k in ('obs', 'psf', 'alpha', 'gt'):
        assert torch.equal(full[k][300:700], part[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize('fwhm_err,shear_err', [(0.0, 0.0), (0.0, 0.03)])
def test_partial_outputs_are_the_same_bits(fwhm_err, shear_err):
    from gdeconv import make_batch_device
    kw = dict(device='cuda:0', psf_fwhm_err=fwhm_err, psf_shear_err=shear_err)
    full = make_batch_device(40, 300, 20.0, **kw)
    only_psf = make_batch_device(40, 300, 20.0, keys=('psf',), **kw)
    assert set(only_psf) == {'psf'} and torch.equal(only_psf['psf'], full['psf'])
    oa = make_batch_device(40, 300, 20.0, keys=('obs', 'alpha'), **kw)
    assert set(oa) == {'obs', 'alpha'} and torch.equal(oa['obs'], full['obs']) and torch.equal(oa['alpha'], full['alpha'])
    gt = make_batch_device(40, 300, 20.0, keys=('gt',), **kw)
    assert torch.equal(gt['gt'], full['gt'])
    one = make_batch_device(139, 1, 20.0, **kw)
    for k in ('obs', 'psf', 'alpha', 'gt'):
        assert torch.equal(one[k], full[k][99:100]), k


@pytest.mark.gpu
def test_empty_batch_and_current_stream():
    from gdeconv import launch_count, make_batch_device
    n0 = launch_count()
    empty = make_batch_device(5, 0, device='cuda:0')
    assert launch_count() == n0
    assert empty['obs'].shape == (0, 1, 48, 48) and empty['alpha'].shape == (0, 1, 1, 1) and empty['psf'].is_cuda
    ref = make_batch_device(5, 64, device='cuda:0')
    s = torch.cuda.Stream(device='cuda:0')
    with torch.cuda.stream(s):
        got = make_batch_device(5, 64, device='cuda:0')
    s.synchronize()
    assert launch_count() == n0 + 2
    for k in ref:
        assert torch.equal(got[k], ref[k]), k
