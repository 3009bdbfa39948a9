"""Every tuning switch of the tcgen05 conv kernel stays a valid implementation: the product configuration and each
alternative (cluster multicast of 1 or 2 CTAs instead of 4, epilogue prefetch placement) reproduce the golden
UnrolledADMMGaussian(4) output of the real reference within the BASELINE tolerance, and so do both classical-solver
kernels.  The switches move weights (cluster size, prefetch placement, ring depth), not sums, so each variant's ResUNet
output is bit-identical to the default's on both layer graphs.  The switches are read once per process, so each variant
runs in a subprocess."""
import functools
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r'''
import json, os, sys
ROOT = sys.argv[1]
sys.path[:0] = [os.path.join(ROOT, 'galaxy-deconv_b200'), ROOT, os.path.join(ROOT, 'tests')]
import torch
import oracle.ref_models as O
from conftest import rel_l2
from gdeconv.synth import make_batch
from models.unrolled_admm_gaussian import UnrolledADMMGaussian
dev = torch.device('cuda:0')
g = torch.load(os.path.join(ROOT, 'tests', 'golden', 'golden_v1.pt'))
i = g['inputs']
sd = O.seeded_state_dict(lambda: O.UnrolledADMMGaussian(4), g['seeds']['G4'])
m = UnrolledADMMGaussian(4).eval()
m.load_state_dict(sd)
m = m.to(dev)
out = m(i['y'].to(dev), i['psf'].to(dev), i['alpha'].to(dev)).cpu()
err_golden = float(rel_l2(out, g['out']['G4']).max())
# a larger ragged batch (several work items per CTA, partial last item, cluster dummies) against the oracle on a sample
b = make_batch(7, 301, 100.0, device=dev)
big = m(b['obs'], b['psf'], b['alpha'])
idx = torch.tensor([0, 150, 299, 300])
ref = O.UnrolledADMMGaussian(4).eval(); ref.load_state_dict(sd)
with torch.no_grad():
    want = ref(b['obs'][idx].cpu(), b['psf'][idx].cpu(), b['alpha'][idx].cpu())
err_big = float(rel_l2(big[idx].cpu(), want).max())
# one fixed ResUNet output per layer graph (chain: nc 32..256, fused: nc 64..512), hashed bit for bit
import hashlib
from models.ResUNet import ResUNet
hashes = {}
for name, nc in (('chain', [32, 64, 128, 256]), ('fused', [64, 128, 256, 512])):
    r = ResUNet(nc=nc).eval()
    r.load_state_dict(O.seeded_state_dict(lambda: O.ResUNet(nc=nc), 29))
    z = r.to(dev)(b['obs']).cpu().contiguous()
    hashes[name] = hashlib.sha256(z.numpy().tobytes()).hexdigest()
print(json.dumps({'golden': err_golden, 'big': err_big, 'finite': bool(torch.isfinite(big).all()), 'hashes': hashes}))
'''

VARIANTS = [
    {},
    {'GDECONV_CLUSTER': '1'},
    {'GDECONV_CLUSTER': '2'},
    {'GDECONV_LATEPF': '0'},
    {'GDECONV_LATEPF': '1'},
    {'GDECONV_BSTAGES': '3'},
]


@functools.lru_cache(maxsize=None)
def _run_child(env_items):
    r = subprocess.run([sys.executable, '-c', CHILD, ROOT], env=dict(os.environ, **dict(env_items)), capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize('env', VARIANTS, ids=lambda e: ','.join(f'{k[8:]}={v}' for k, v in e.items()) or 'default')
def test_switch_variant_matches_reference(env):
    res = _run_child(tuple(sorted(env.items())))
    assert res['hashes'] == _run_child(())['hashes'], res      # bit-identical ResUNet outputs on both graphs
    assert res['finite']
    assert res['golden'] < 1e-3, res          # BASELINE tolerance: relative L2 per stamp
    assert res['big'] < 1e-3, res


SOLVER_CHILD = r'''
import json, os, sys
ROOT = sys.argv[1]
sys.path[:0] = [os.path.join(ROOT, 'galaxy-deconv_b200'), ROOT, os.path.join(ROOT, 'tests')]
import torch
import oracle.ref_models as O
from conftest import rel_l2
from gdsynth import make_batch
from models.Richard_Lucy import Richard_Lucy
from models.Tikhonet import Tikhonov
from models.Wiener import Wiener
dev = torch.device('cuda:0')
res = {}
for B in (1, 4, 5, 6, 1483):                      # below, at and above one CTA pass of 5 stamps; many passes per CTA
    b = make_batch(11, B, 'mixed', device=dev)
    idx = torch.arange(B) if B < 8 else torch.tensor([0, 4, 5, 741, 1479, 1480, 1482])
    args = [b[k][idx].cpu() for k in ('obs', 'psf', 'alpha')]
    for n_it in ((0, 1, 3, 10) if B in (4, 6) else (10,)):
        got = Richard_Lucy(n_it)(b['obs'], b['psf'])
        res['rl'] = max(res.get('rl', 0.0), float(rel_l2(got[idx].cpu(), O.Richard_Lucy(n_it)(args[0], args[1])).max()))
        res['finite'] = res.get('finite', True) and bool(torch.isfinite(got).all())
    for name, mine, ref in (('wiener', lambda: Wiener()(b['obs'], b['psf'], b['alpha']), lambda: O.Wiener()(*args)),
                            ('tik_id', lambda: Tikhonov('Identity')(b['obs'], b['psf'], b['alpha'], 0.7), lambda: O.Tikhonov('Identity')(*args, 0.7)),
                            ('tik_lap', lambda: Tikhonov('Laplacian')(b['obs'], b['psf'], b['alpha'], 1.3), lambda: O.Tikhonov('Laplacian')(*args, 1.3))):
        got = mine()
        res[name] = max(res.get(name, 0.0), float(rel_l2(got[idx].cpu(), ref()).max()))
        res['finite'] = res.get('finite', True) and bool(torch.isfinite(got).all())
print(json.dumps(res))
'''


@pytest.mark.parametrize('env', [{}, {'GDECONV_SOLVER48': '0'}], ids=['register-fft', 'phase-fft'])
def test_wiener_tikhonov_kernels_match_reference(env):
    """k_wiener48 / k_rl48 (every 48-point transform in one thread's registers, five stamps per CTA pass) and the phase-structured
    k_solver they replace, on ragged batches, against the oracle (models/Wiener.py:10-20, models/Tikhonet.py:15-31,
    models/Richard_Lucy.py:10-24); internal fp32 gates 2e-5 / 2e-4"""
    r = subprocess.run([sys.executable, '-c', SOLVER_CHILD, ROOT], env=dict(os.environ, **env), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res['finite']
    for k in ('wiener', 'tik_id', 'tik_lap'):
        assert res[k] < 2e-5, res
    assert res['rl'] < 2e-4, res                  # Richardson-Lucy accumulates over its iterations: the internal gate of test_gpu_parity
