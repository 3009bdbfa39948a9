"""Tikhonet / XDenseUNet (SURVEY.md section 8f #1) with the reference's TRAINED weights (tests/golden/tikhonet_v1.pt, made by
tests/golden/make_golden_tikhonet.py from saved_models/Tikhonet_Laplacian_50epochs.pth): oracle vs golden on CPU, CUDA path
vs golden on the GPU.  fp32 end to end -> internal gate 2e-5 (stamps) on top of the BASELINE tolerances."""
import os
import subprocess
import sys

import pytest
import torch

import oracle.ref_models as O
from conftest import ROOT, rel_l2

REF = os.environ.get('GDECONV_REFERENCE', '')       # a checkout of the upstream Galaxy-Deconv project, if one is at hand


@pytest.fixture(scope='module')
def tik():
    return torch.load(os.path.join(ROOT, 'tests', 'golden', 'tikhonet_v1.pt'))


def _inp(golden):
    i = golden['inputs']
    return i['y'], i['psf'], i['alpha']


def test_oracle_tikhonet_trained_weights(golden, tik):
    assert all(tik['exact'].values())                       # bit-exact vs the real reference at generation time
    m = O.Tikhonet('Laplacian').eval()
    m.load_state_dict(tik['state']['Laplacian'])
    with torch.no_grad():
        out = m(*_inp(golden))
        den = m.denoiser(tik['x_in'])
    assert rel_l2(out, tik['out']['Tikhonet_Laplacian']).max() < 2e-5
    assert rel_l2(den, tik['out']['XDenseUNet']).max() < 2e-5


def test_state_dict_layout_matches_reference_file(tik):
    from models.Tikhonet import Tikhonet
    m = Tikhonet('Laplacian')
    missing, unexpected = m.load_state_dict(tik['state']['Laplacian'])
    assert not missing and not unexpected
    torch.manual_seed(31)
    a = Tikhonet('Identity').state_dict()
    torch.manual_seed(31)
    b = O.Tikhonet('Identity').state_dict()
    assert list(a.keys()) == list(b.keys()) and all(torch.equal(a[k], b[k]) for k in a)


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, 'saved_models')), reason='GDECONV_REFERENCE names no upstream checkout')
def test_golden_regenerates_from_live_reference():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'tests', 'golden', 'make_golden_tikhonet.py'), '--check'],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]


@pytest.mark.gpu
def test_tikhonet_trained_weights_on_gpu(golden, tik):
    from gdeconv import moments_e
    from models.Tikhonet import Tikhonet
    dev = torch.device('cuda:0')
    m = Tikhonet('Laplacian').eval()
    m.load_state_dict(tik['state']['Laplacian'])
    m = m.to(dev)
    y, k, a = (t.to(dev) for t in _inp(golden))
    out = m(y, k, a)
    want = tik['out']['Tikhonet_Laplacian']
    err = rel_l2(out.cpu(), want)
    assert err.max() < 2e-5, err
    assert (moments_e(out).cpu() - O.moments_e(want)).abs().max() < 1e-4
    den = m.denoiser(tik['x_in'].to(dev)).cpu()
    assert rel_l2(den, tik['out']['XDenseUNet']).max() < 2e-5


@pytest.mark.gpu
def test_tikhonet_identity_seeded_and_ragged_batches(golden, tik):
    from models.Tikhonet import Tikhonet
    dev = torch.device('cuda:0')
    torch.manual_seed(31)
    m = Tikhonet('Identity').eval().to(dev)
    y, k, a = (t.to(dev) for t in _inp(golden))
    out = m(y, k, a)
    assert rel_l2(out.cpu(), tik['out']['Tikhonet_Identity_seed31']).max() < 2e-5
    one = m(y[2:3], k[2:3], a[2:3])
    assert torch.equal(one[0], out[2])
    # a batch that is not a power of two and larger than one chunk
    from gdeconv.synth import make_batch
    b = make_batch(0, 2500, 100.0, device=dev)
    big = m(b['obs'], b['psf'], b['alpha'])
    ref = O.Tikhonet('Identity').eval()
    ref.load_state_dict({kk: v.cpu() for kk, v in m.state_dict().items()})
    idx = torch.tensor([0, 2047, 2048, 2499])
    with torch.no_grad():
        want = ref(b['obs'][idx].cpu(), b['psf'][idx].cpu(), b['alpha'][idx].cpu())
    assert rel_l2(big[idx].cpu(), want).max() < 2e-5


@pytest.mark.gpu
def test_tikhonet_is_the_first_call_of_a_process():
    """The Tikhonov step of Tikhonet runs in k_wiener48, whose shared-memory size needs a per-device opt-in: it must be in place even when
    gd_pack_xdense / gd_tikhonet_forward are the first library calls of the process (no ADMM model, no solver call before them)."""
    import subprocess
    import sys
    child = (
        "import os, sys, torch\n"
        "ROOT = sys.argv[1]\n"
        "sys.path[:0] = [os.path.join(ROOT, 'galaxy-deconv_b200'), ROOT]\n"
        "from models.Tikhonet import Tikhonet\n"
        "torch.manual_seed(1)\n"
        "m = Tikhonet('Laplacian').eval().to('cuda:0')\n"
        "g = torch.load(os.path.join(ROOT, 'tests', 'golden', 'golden_v1.pt'))['inputs']\n"
        "out = m(g['y'][:3].to('cuda:0'), g['psf'][:3].to('cuda:0'), g['alpha'][:3].to('cuda:0'))\n"
        "torch.cuda.synchronize()\n"
        "print('FIRST-CALL-OK', bool(torch.isfinite(out).all()))\n")
    r = subprocess.run([sys.executable, '-c', child, ROOT], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and 'FIRST-CALL-OK True' in r.stdout, r.stderr[-2000:]
