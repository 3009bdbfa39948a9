"""The oracle (oracle/ref_models.py) against the golden vectors produced by the real reference
(tests/golden/make_golden.py).  Bit-exactness oracle==reference is asserted at generation time and
re-checked here whenever GDECONV_REFERENCE names a checkout of the upstream project; elsewhere (other CPU,
other BLAS kernels) the oracle must reproduce the committed vectors to 1e-5."""
import os
import subprocess
import sys

import pytest
import torch

import oracle.ref_models as O
from conftest import ROOT, rel_l2

TOL = 2e-5
REF = os.environ.get('GDECONV_REFERENCE', '')       # a checkout of the upstream Galaxy-Deconv project, if one is at hand


def _inputs(g, n=4):
    i = g['inputs']
    return i['y'][:n].contiguous(), i['psf'][:n].contiguous(), i['alpha'][:n].contiguous()


def test_generation_time_pin(golden):
    assert all(golden['meta']['oracle_bitexact'].values())


@pytest.mark.parametrize('tag,n', [('G4', 4), ('G8', 8)])
def test_path_g(golden, tag, n):
    torch.set_num_threads(1)
    m = O.UnrolledADMMGaussian(n).eval()
    m.load_state_dict(O.seeded_state_dict(lambda: O.UnrolledADMMGaussian(n), golden['seeds'][tag]))
    with torch.no_grad():
        out = m(*_inputs(golden))
    assert rel_l2(out, golden['out'][tag]).max() < TOL


def test_path_g_analysis(golden):
    m = O.UnrolledADMMGaussian(2, analysis=True).eval()
    m.load_state_dict(O.seeded_state_dict(lambda: O.UnrolledADMMGaussian(2), 11))
    with torch.no_grad():
        xs, zs, us, rhos = m(*_inputs(golden))
    flat = xs + zs + us + rhos
    for a, b in zip(flat, golden['out']['G2_analysis']):
        assert rel_l2(a, b).max() < TOL


@pytest.mark.parametrize('tag,llh', [('U2_gauss', 'Gaussian'), ('U2_poisson', 'Poisson')])
def test_path_u(golden, tag, llh):
    m = O.Unrolled_ADMM(2, llh=llh).eval()
    m.load_state_dict(O.seeded_state_dict(lambda: O.Unrolled_ADMM(2, llh=llh), golden['seeds'][tag]))
    with torch.no_grad():
        out = m(*_inputs(golden))
    assert rel_l2(out, golden['out'][tag]).max() < TOL


def test_fft_solvers(golden):
    y, k, a = _inputs(golden)
    for n in (10, 50):
        assert rel_l2(O.Richard_Lucy(n)(y, k), golden['out'][f'RL{n}']).max() < 1e-4
    assert rel_l2(O.Wiener()(y, k, a), golden['out']['Wiener']).max() < TOL
    yc, lam = y.clamp_min(0), torch.tensor(1.)
    for f in ('Identity', 'Laplacian'):
        assert rel_l2(O.Tikhonov(f)(yc, k, a, lam), golden['out'][f'Tikhonov_{f}']).max() < TOL


def test_laplacian_quirk():
    """SURVEY.md section 0.6: psf_to_otf on the 3x3 Laplacian yields 7 non-zeros summing to 2."""
    p, _ = O.psf_to_otf(O.laplacian_kernel(), (1, 1, 48, 48))
    nz = {(int(r), int(c)): float(p[0, 0, r, c]) for r, c in p[0, 0].nonzero()}
    assert nz == {(0, 47): 1, (1, 47): 1, (46, 47): 1, (47, 0): 1, (47, 1): 1, (47, 46): 1, (47, 47): -4}


def test_moments(golden):
    assert torch.allclose(O.moments_e(golden['inputs']['gt']), golden['out']['e_gt'], atol=1e-5)
    assert torch.allclose(O.moments_e(golden['out']['G8']), golden['out']['e_G8'], atol=1e-5)


def test_survey_known_answers():
    """SURVEY.md section 8c smoke values on tutorials/obs.pth (stamp 0 of the golden inputs)."""
    g = torch.load(os.path.join(ROOT, 'tests', 'golden', 'golden_v1.pt'))
    y, k, a = (t[:1] for t in _inputs(g))
    w = O.Wiener()(y, k, a)
    assert abs(float(w.sum()) - 202.298) < 0.05 and abs(float(w.max()) - 1.2263) < 1e-3
    rl = O.Richard_Lucy(10)(y, k)
    assert abs(float(rl.sum()) / 1020936.9 - 1) < 1e-4
    torch.manual_seed(0)
    m = O.UnrolledADMMGaussian(8).eval()
    with torch.no_grad():
        out = m(y, k, a)
    assert abs(float(out.sum()) - 55.3592) < 0.02 and abs(float(out.abs().mean()) - 0.121897) < 1e-4


def test_admmnet_and_old_without_subnet(tmp_path):
    """oracle ADMMNet (models/ADMMNet.py:78-129) and Unrolled_ADMM_Old(SubNet=False) (:385-386) vs the outputs of the REAL reference
    (tests/golden/make_golden_admmnet.py, bit-exact at generation time)"""
    g = torch.load(os.path.join(ROOT, 'tests', 'golden', 'golden_v1.pt'))
    ga = torch.load(os.path.join(ROOT, 'tests', 'golden', 'admmnet_v1.pt'))
    y, k, a = (t[:2] for t in _inputs(g))
    torch.manual_seed(ga['seeds']['net'])
    f = str(tmp_path / 'resunet.pth')
    torch.save(O.ResUNet().state_dict(), f)
    for llh in ('Gaussian', 'Poisson'):
        with torch.no_grad():
            out = O.ADMMNet(2, llh=llh, model_file=f).eval()(y, k, a)
        assert rel_l2(out, ga['out'][f'ADMMNet2_{llh}']).max() < TOL
    with pytest.raises(ValueError):
        O.ADMMNet(2, model_file=str(tmp_path / 'missing.pth'))
    m = O.Unrolled_ADMM_Old(2, llh='Gaussian', SubNet=False).eval()
    m.load_state_dict(O.seeded_state_dict(lambda: O.Unrolled_ADMM_Old(2, llh='Gaussian', SubNet=False), ga['seeds']['old']))
    with torch.no_grad():
        lists = m(y, k, a)
    for got, want in zip([t[-1] for t in lists[:5]], ga['out']['UOld2_norho']):
        assert rel_l2(got, want).max() < TOL


def test_xdenseunet_as_admm_denoiser(tmp_path):
    """oracle ADMM classes with denoiser='XDenseUNet' (models/Unrolled_ADMM.py:142-151,163; models/ADMMNet.py:65-74,87) vs the outputs of
    the REAL reference with its trained XDenseUNet as the Z-update (tests/golden/make_golden_xdense_admm.py, bit-exact at generation)"""
    g = torch.load(os.path.join(ROOT, 'tests', 'golden', 'golden_v1.pt'))
    gx = torch.load(os.path.join(ROOT, 'tests', 'golden', 'xdense_admm_v1.pt'))
    tik = torch.load(os.path.join(ROOT, 'tests', 'golden', 'tikhonet_v1.pt'))['state']['Laplacian']
    xsd = {k[len('denoiser.'):]: v for k, v in tik.items() if k.startswith('denoiser.')}
    y, k, a = (t[:2] for t in _inputs(g))
    m = O.Unrolled_ADMM(2, llh='Gaussian', denoiser='XDenseUNet').eval()
    sd = dict(gx['state']['U2_gauss_xd']); sd.update({'Z.net.' + kk: v for kk, v in xsd.items()})
    m.load_state_dict(sd)
    with torch.no_grad():
        assert rel_l2(m(y, k, a), gx['out']['U2_gauss_xd']).max() < TOL
    f = str(tmp_path / 'xdense.pth')
    torch.save(xsd, f)
    with torch.no_grad():
        out = O.ADMMNet(2, llh='Poisson', denoiser='XDenseUNet', model_file=f).eval()(y, k, a)
    assert rel_l2(out, gx['out']['ADMMNet2_Poisson_xd']).max() < TOL


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, 'models')), reason='GDECONV_REFERENCE names no upstream checkout')
def test_xdense_admm_golden_vs_live_reference():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'golden', 'make_golden_xdense_admm.py'), '--check'],
                       capture_output=True, text=True, timeout=900, env=dict(os.environ, PYTHONDONTWRITEBYTECODE='1'))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, 'models')), reason='GDECONV_REFERENCE names no upstream checkout')
def test_admmnet_golden_vs_live_reference():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'golden', 'make_golden_admmnet.py'), '--check'],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, PYTHONDONTWRITEBYTECODE='1'))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, 'models')), reason='GDECONV_REFERENCE names no upstream checkout')
def test_oracle_bitexact_vs_live_reference():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'golden', 'make_golden.py'), '--check'],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
