"""The drop-in boundary drops in (SURVEY.md section 8b, INTEGRATION.md section A): with galaxy-deconv_b200/ AHEAD of the
reference checkout on sys.path, the modules of the hot path resolve to this package and every other reference module
(utils.utils_data, utils.utils_test, utils.utils_deblur, ...) still resolves to the reference's own file, because ``models`` and
``utils`` are namespace packages here exactly as they are in the reference.

CPU part: import resolution (in a subprocess with a clean sys.path; fpfs is stubbed because it is not installable here) and
the reference-signature FFT helpers' input contract.  GPU part: the model-construction / load / forward sequence of
test.py:32-54,85 executed as written there, and psf_to_otf / conv_fft_batch / conv_fft against the oracle."""
import os
import subprocess
import sys

import pytest
import torch

import oracle.ref_models as O
from conftest import ROOT, rel_l2

PKG = os.path.join(ROOT, 'galaxy-deconv_b200')
REF = os.environ.get('GDECONV_REFERENCE', '')       # a checkout of the upstream Galaxy-Deconv project, if one is at hand


def test_models_and_utils_are_namespace_packages():
    import models
    import utils
    for pkg in (models, utils):
        assert getattr(pkg, '__file__', None) is None, f'{pkg.__name__} must not have an __init__.py (it would shadow the reference)'
        assert any(os.path.samefile(p, os.path.join(PKG, pkg.__name__)) for p in pkg.__path__)
    assert not os.path.exists(os.path.join(PKG, 'models', '__init__.py'))
    assert not os.path.exists(os.path.join(PKG, 'utils', '__init__.py'))


def test_reference_signature_helpers_exist():
    import inspect
    import utils.utils_torch as u
    assert list(inspect.signature(u.psf_to_otf).parameters) == ['ker', 'size']           # utils/utils_torch.py:79
    assert list(inspect.signature(u.conv_fft_batch).parameters) == ['H', 'x']            # :46
    assert list(inspect.signature(u.conv_fft).parameters) == ['H', 'x']                  # :35
    for name in ('pad_double', 'crop_half', 'laplacian_kernel'):
        assert callable(getattr(u, name))
    # no CPU path: CPU tensors raise instead of computing
    with pytest.raises(RuntimeError):
        u.psf_to_otf(torch.zeros(1, 1, 48, 48), (1, 1, 48, 48))
    with pytest.raises(ValueError):
        u.psf_to_otf(torch.zeros(1, 1, 48, 48), (1, 1, 32, 32))


CHILD = r'''
import sys, types, os
pkg, ref = sys.argv[1], sys.argv[2]
sys.path[:0] = [pkg, ref]
sys.modules.setdefault('fpfs', types.ModuleType('fpfs'))          # utils/utils_test.py:3 imports it at module top; not installable here
# the import block of test.py:9-15 / test_psf.py:9-14, verbatim
from models.Richard_Lucy import Richard_Lucy
from models.Tikhonet import Tikhonet
from models.Unrolled_ADMM import Unrolled_ADMM
from models.Wiener import Wiener
from utils.utils_data import get_dataloader
from utils.utils_test import delta_2D, estimate_shear
# train.py:13 and the ablation model's import line (models/ADMMNet.py:8)
from models.unrolled_admm_gaussian import UnrolledADMMGaussian
from utils.utils_torch import conv_fft, conv_fft_batch, psf_to_otf
import models.ADMMNet
import utils.utils_data, utils.utils_test, utils.utils_torch
mine = lambda m: os.path.realpath(m.__file__).startswith(os.path.realpath(pkg))
theirs = lambda m: os.path.realpath(m.__file__).startswith(os.path.realpath(ref))
import utils.utils_deblur                                           # a reference-only helper module (scipy): must stay importable
assert all(mine(sys.modules[n]) for n in ('models.Richard_Lucy', 'models.Tikhonet', 'models.Unrolled_ADMM', 'models.Wiener', 'models.ADMMNet',
                                          'models.unrolled_admm_gaussian', 'utils.utils_torch')), 'hot-path modules must come from this package'
assert all(theirs(sys.modules[n]) for n in ('utils.utils_data', 'utils.utils_test', 'utils.utils_deblur')), 'other modules must stay the reference files'
print('DROPIN-OK')
'''


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, 'models')), reason='GDECONV_REFERENCE names no upstream checkout')
def test_reference_drivers_import_unchanged_on_top_of_this_package(tmp_path):
    env = {k: v for k, v in os.environ.items() if k != 'PYTHONPATH'}
    r = subprocess.run([sys.executable, '-c', CHILD, PKG, REF], capture_output=True, text=True, timeout=300, env=env, cwd=tmp_path)
    assert r.returncode == 0 and 'DROPIN-OK' in r.stdout, r.stderr[-3000:]


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    return torch.device('cuda:0')


@pytest.mark.gpu
def test_psf_to_otf_and_conv_fft_batch_match_reference(golden, dev):
    """same-size PSF (pure ifftshift), the 3x3 Laplacian (7-non-zero broadcast artefact) and an even 4x4 kernel"""
    from utils.utils_torch import conv_fft, conv_fft_batch, laplacian_kernel, psf_to_otf
    psf = golden['inputs']['psf'][:4]
    g = torch.Generator().manual_seed(3)
    x = torch.randn(4, 1, 48, 48, generator=g)
    for ker in (psf, laplacian_kernel(), torch.randn(1, 1, 4, 4, generator=g), torch.randn(4, 1, 2, 2, generator=g)):
        p_ref, H_ref = O.psf_to_otf(ker, x.size())
        p, H = psf_to_otf(ker.to(dev), x.size())
        assert p.shape == p_ref.shape and H.shape == H_ref.shape and H.dtype == torch.complex64
        assert torch.equal(p.cpu(), p_ref)                                   # index shuffle: bit-exact
        assert (H.cpu() - H_ref).abs().max() <= 2e-5 * H_ref.abs().max()
        for Hh in (H, torch.conj(H)):                                        # models/Unrolled_ADMM.py:172,207 use both
            want = O.conv_fft_batch(Hh.cpu().resolve_conj(), x)
            assert rel_l2(conv_fft_batch(Hh, x.to(dev)).cpu(), want).max() < 2e-5
    # a batch-1 OTF broadcast over the batch (conv_fft's H.repeat, utils/utils_torch.py:38) and the 3-D form (:40-43)
    _, H1 = psf_to_otf(psf[:1].to(dev), (1, 1, 48, 48))
    want = O.conv_fft_batch(H1.cpu().expand(4, 1, 48, 48), x)
    assert rel_l2(conv_fft(H1, x.to(dev)).cpu(), want).max() < 2e-5
    got3 = conv_fft(H1.view(1, 48, 48), x[:, 0].to(dev))
    assert got3.shape == (4, 48, 48) and rel_l2(got3.cpu().unsqueeze(1), want).max() < 2e-5
    # a non-Hermitian H: .real must still be exact (the kernel multiplies by the Hermitian part of H)
    Hn = torch.complex(torch.randn(4, 1, 48, 48, generator=g), torch.randn(4, 1, 48, 48, generator=g))
    assert rel_l2(conv_fft_batch(Hn.to(dev), x.to(dev)).cpu(), O.conv_fft_batch(Hn, x)).max() < 2e-5


@pytest.mark.gpu
@pytest.mark.parametrize('method,n_iters', [('Wiener', 0), ('Richard-Lucy(10)', 10), ('Tikhonet_Laplacian', 0),
                                            ('Unrolled_ADMM_Gaussian(2)', 2), ('Unrolled_ADMM(2)', 2)])
def test_test_py_model_sequence_verbatim(golden, dev, tmp_path, method, n_iters):
    """test.py:32-54 (model selection by method name, .to(device), load_state_dict(torch.load(file, map_location)), .eval())
    and :85 (model(obs, psf, alpha) under no_grad), statement by statement, against the oracle with the same weights."""
    from models.Richard_Lucy import Richard_Lucy
    from models.Tikhonet import Tikhonet
    from models.Unrolled_ADMM import Unrolled_ADMM
    from models.Wiener import Wiener
    device = dev
    model_file = str(tmp_path / 'weights.pth')
    ref = None
    if method == 'Wiener':
        ref = O.Wiener()
    elif 'Richard-Lucy' in method:
        ref = O.Richard_Lucy(n_iters)
    elif 'Laplacian' in method:
        torch.manual_seed(21)
        ref = O.Tikhonet(filter='Laplacian')
    elif 'Gaussian' in method:
        torch.manual_seed(22)
        ref = O.Unrolled_ADMM(n_iters, llh='Gaussian', PnP=True)
    else:
        torch.manual_seed(23)
        ref = O.Unrolled_ADMM(n_iters, llh='Poisson', PnP=True)
    ref.eval()
    torch.save(ref.state_dict(), model_file)

    # ---- test.py:32-54 ----
    model = None
    if method == 'Wiener':
        model = Wiener()
    elif 'Richard-Lucy' in method:
        model = Richard_Lucy(n_iters=n_iters)
    elif method == 'Tikhonet':
        model = Tikhonet(filter='Identity')
    elif method == 'ShapeNet' or 'Laplacian' in method:
        model = Tikhonet(filter='Laplacian')
    elif 'Gaussian' in method:
        model = Unrolled_ADMM(n_iters=n_iters, llh='Gaussian', PnP=True)
    else:
        model = Unrolled_ADMM(n_iters=n_iters, llh='Poisson', PnP=True)
    if model is not None:
        model.to(device)
        if 'Tikhonet' in method or 'ShapeNet' in method or 'ADMM' in method:
            model.load_state_dict(torch.load(model_file, map_location=torch.device(device)))
        model.eval()

    # ---- test.py:80-85 (one galaxy at a time, batch 1) ----
    i = golden['inputs']
    with torch.no_grad():
        for n in range(2):
            obs, psf, alpha = i['y'][n:n + 1], i['psf'][n:n + 1], i['alpha'][n:n + 1]
            want = ref(obs, psf) if 'Richard-Lucy' in method else ref(obs, psf, alpha)
            obs, psf, alpha = obs.to(device), psf.to(device), alpha.to(device)
            rec = model(obs, psf) if 'Richard-Lucy' in method else model(obs, psf, alpha)
            rec = rec.cpu().squeeze(dim=0).squeeze(dim=0).detach().numpy()          # test.py:86
            err = rel_l2(torch.from_numpy(rec)[None, None], want)
            assert err.max() < (1e-3 if 'ADMM' in method else 2e-4), (method, err)
