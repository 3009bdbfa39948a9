"""The tcgen05 ResUNet (GDECONV_PRECISION=fp16_umma) against a reference that rounds where its kernels round.

The other ResUNet tests compare with the fp32 oracle at the 1e-3 BASELINE tolerance, i.e. above the fp16 operand noise of
the product path (2.4e-4 .. 7.8e-4, DESIGN section 4): a dropped lo half, a wrong halo at the stamp's frame, one wrong
k_tail_gather class or a seam slip between the half-stamp items of k_l1_chain hides in that noise.  Here the reference is
oracle/resunet_fp16.py, which stores fp16 / fp32 exactly where the chain graph (nc 32..256) and the fused graph
(nc 64..512) store them, so the noise cancels:

  * routing weights: every output of every 3x3 and k2s2 conv has ONE nonzero weight +-2^k (all taps, every K chunk and all
    four sub-pixels drawn), so each tensor-core sum is one exact product and only fp32 epilogue adds remain;
  * dense weights: the default init; what remains is the fp32 accumulation order flipping an fp16 rounding now and then.

Inputs: 301 stamps (ragged: several work items per CTA, a partial last wave), nine families interleaved so that neighbours
differ: noise-free galaxies (fp16-subnormal wings after scaling), observations at SNR 20 and 300, Wiener deconvolutions,
white noise, a border frame only, the seam band of the half-stamp items only, single impulses at the corners and on rows
23/24, and negated galaxies.

Metrics, per compared stamp: rel-L2 (max and RMS over stamps) and the region error, the RMS difference over the border
frame and over each 4-row band divided by the RMS of the whole reference stamp (a localised defect is not averaged away).

Measured on one NVIDIA B200 (power limit 1000 W, max SM clock 1965 MHz) at the gates' introduction; the outputs are
deterministic (test_chunking_and_determinism), so a rerun measures the same values:
    routing, both graphs:  bit-identical to the emulator (rel-L2 0, region 0)      -> gates 1e-6 (rel max / RMS / region)
    dense, chain:          rel-L2 max 7.1e-5, RMS 5.7e-5, region 2.1e-4            -> gates 2e-4 / 1.5e-4 / 4.5e-4
    dense, fused:          rel-L2 max 1.9e-4, RMS 1.1e-4, region 5.1e-4            -> gates 4e-4 / 2.5e-4 / 1.1e-3
(the fp32-oracle gate these replace is 1e-3).  The routing result pins every rounding point of the emulator, fp16 subnormal
operands included (the tensor cores do not flush them).  The dense residue is the tensor cores' fp32 accumulation order, not
a missed rounding point: perturbing the emulator's own accumulators by +-1 fp32 ulp moves it by as much (7.9e-5 chain,
1.6e-4 fused), because every flipped fp16 rounding propagates through the 34 layers.  For the same reason the dense set with
every second ResBlock conv x4 is not gated here: kernel and emulator differ by 1.0e-3 there, and so does the perturbed
emulator (0.98e-3) -- it measures that chaos, which the fp32-oracle tests already bound.

Besides, exact properties the design guarantees are asserted bit for bit: zero in / zero out, power-of-two homogeneity,
neighbour and position independence (NaN neighbours included), chunking and determinism.  The CPU self-check shows
each gate fails a deliberately wrong emulator by >= 3x.
"""
import pytest
import torch

import oracle.ref_models as O
from conftest import rel_l2
from oracle.resunet_fp16 import resunet_fp16

# ---- gates (measured values in the module docstring): (rel-L2 max over stamps, RMS over stamps of the rel-L2, region) ----
ROUTING_GATES = (1e-6, 1e-6, 1e-6)
DENSE_CHAIN_GATES = (2e-4, 1.5e-4, 4.5e-4)
DENSE_FUSED_GATES = (4e-4, 2.5e-4, 1.1e-3)
GATES = {('routing', 'chain'): ROUTING_GATES, ('routing', 'fused'): ROUTING_GATES,
         ('dense', 'chain'): DENSE_CHAIN_GATES, ('dense', 'fused'): DENSE_FUSED_GATES}
METRICS = ('rel_max', 'rel_rms', 'region')

NC = {'chain': [32, 64, 128, 256], 'fused': [64, 128, 256, 512]}
BATCH = 301
N_FAMILIES = 9
IMPULSES = ((0, 0), (0, 47), (47, 0), (47, 47), (23, 17), (24, 30))
# compared stamps: every family several times, the impulse positions, CTA-wave neighbours, the batch's end
COMPARE = {
    'chain': sorted(set(range(27)) | {34, 43, 52} | {72, 73, 74, 75, 146, 147, 148, 149, 150} | set(range(292, BATCH))),
    'fused': sorted(set(range(9)) | {16, 25, 34, 43, 52} | {73, 74, 147, 148, 149} | set(range(296, BATCH))),
}
REGIMES = ('routing', 'dense')


# ---------------------------------------------------------------------------------------------------
# inputs and weights (CPU, seeded)
# ---------------------------------------------------------------------------------------------------
def input_batch(n=BATCH, seed=23):
    """[n,1,48,48] fp32: family i % 9 for stamp i (see the module docstring)."""
    from gdsynth import make_batch
    g = torch.Generator().manual_seed(seed)
    b20, b300 = make_batch(0, n, 20.0), make_batch(0, n, 300.0)
    wiener = O.Wiener()(b20['obs'], b20['psf'], b20['alpha']).float()
    x = torch.zeros(n, 1, 48, 48)
    for i in range(n):
        f = i % N_FAMILIES
        if f == 0:
            x[i] = b300['gt'][i]
        elif f == 1:
            x[i] = b20['obs'][i]
        elif f == 2:
            x[i] = wiener[i]
        elif f == 3:
            x[i, 0] = torch.randn(48, 48, generator=g)
        elif f == 4:
            x[i] = b300['obs'][i]
        elif f == 5:                      # border frame only: rows and columns 0, 1, 46, 47
            v = torch.randn(48, 48, generator=g)
            m = torch.zeros(48, 48, dtype=torch.bool)
            m[[0, 1, 46, 47], :] = True
            m[:, [0, 1, 46, 47]] = True
            x[i, 0] = torch.where(m, v, torch.zeros(()))
        elif f == 6:                      # the seam band of k_l1_chain's half-stamp items only: rows 20..27
            x[i, 0, 20:28] = torch.randn(8, 48, generator=g)
        elif f == 7:                      # one impulse: the four corners, rows 23 / 24
            y, xx = IMPULSES[(i // N_FAMILIES) % len(IMPULSES)]
            x[i, 0, y, xx] = 1.0 if (i // N_FAMILIES) % 2 else -3.0
        else:
            x[i] = -b300['gt'][i]
    return x


def _pow2(shape, kmin, kmax, g):
    k = torch.randint(kmin, kmax + 1, shape, generator=g).double()
    s = torch.where(torch.rand(shape, generator=g) < 0.5, -1.0, 1.0).double()
    return (s * torch.pow(2.0, k)).float()


def routing_state_dict(nc, seed=7):
    """One nonzero weight +-2^k per output channel of every 3x3 conv (tap and input channel drawn: all 9 taps, every input
    channel once) and per (output channel, sub-pixel) of every k2s2 conv; m_tail dense +-2^k.  Magnitudes: first convs of
    a ResBlock 2^-1..2^1, second convs 2^-4..2^-2, k2s2 2^-1..2^0, head 2^-1..2^0, tail 2^-5..2^-3."""
    g = torch.Generator().manual_seed(seed)
    sd = O.ResUNet(nc=nc).state_dict()
    out = {}
    for key, w in sd.items():
        w = torch.zeros_like(w)
        if key == 'm_head.weight':                        # [C, 1, 3, 3]
            C = w.shape[0]
            taps = torch.randperm(C, generator=g) % 9
            w.view(C, 9)[torch.arange(C), taps] = _pow2((C,), -1, 0, g)
        elif key == 'm_tail.weight':
            w = _pow2(tuple(w.shape), -5, -3, g)
        elif w.shape[-1] == 3:                            # ResBlock conv [C, C, 3, 3]
            C = w.shape[0]
            taps = torch.randperm(C, generator=g) % 9
            ci = torch.randperm(C, generator=g)
            lo, hi = (-1, 1) if key.endswith('res.0.weight') else (-4, -2)
            w.view(C, C, 9)[torch.arange(C), ci, taps] = _pow2((C,), lo, hi, g)
        elif '.0.weight' in key and key.startswith('m_up'):   # transposed [2C, C, 2, 2]: one input per (co, sub-pixel)
            Ci, Co = w.shape[:2]
            ci = torch.cat([torch.randperm(Ci, generator=g), torch.randperm(Ci, generator=g)])[torch.randperm(2 * Ci, generator=g)]
            co = torch.arange(Co).repeat_interleave(4)
            sp = torch.arange(4).repeat(Co)
            w.view(Ci, Co, 4)[ci, co, sp] = _pow2((4 * Co,), -1, 0, g)
        else:                                             # strided [2C, C, 2, 2]: K = sub-pixel * C + ci, every K pair drawn
            Co, Ci = w.shape[:2]
            k = 2 * torch.randperm(Co, generator=g) + torch.randint(0, 2, (Co,), generator=g)
            w.view(Co, Ci, 4)[torch.arange(Co), k % Ci, k // Ci] = _pow2((Co,), -1, 0, g)
        out[key] = w
    return out


def state_dict_for(regime, graph):
    nc = NC[graph]
    if regime == 'routing':
        return routing_state_dict(nc)
    return O.seeded_state_dict(lambda: O.ResUNet(nc=nc), 41)


# ---------------------------------------------------------------------------------------------------
# metrics
# ---------------------------------------------------------------------------------------------------
def region_masks():
    m = [torch.zeros(48, 48, dtype=torch.bool) for _ in range(13)]
    m[0][[0, 1, 46, 47], :] = True
    m[0][:, [0, 1, 46, 47]] = True
    for b in range(12):
        m[1 + b][4 * b:4 * b + 4] = True
    return m


def region_error(got, ref):
    """[n]: max over the border frame and the twelve 4-row bands of RMS(got - ref) over that region / RMS(ref) over the stamp."""
    d = (got.double() - ref.double())[:, 0]
    den = ref.double()[:, 0].pow(2).mean((1, 2)).sqrt().clamp_min(1e-300)
    per = torch.stack([d[:, m].pow(2).mean(1).sqrt() for m in region_masks()], 1)
    return (per / den[:, None]).max(1).values


def metrics(got, ref):
    rel = rel_l2(got, ref).double()
    return {'rel_max': float(rel.max()), 'rel_rms': float(rel.pow(2).mean().sqrt()), 'region': float(region_error(got, ref).max())}


def check_gates(m, regime, graph):
    return all(m[k] < g for k, g in zip(METRICS, GATES[(regime, graph)]))


# ---------------------------------------------------------------------------------------------------
# CPU self-check: the emulator is the network, and the gates would fail a subtly wrong kernel
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('graph', ['chain', 'fused'])
def test_unrounded_emulator_is_the_oracle(graph):
    sd = O.seeded_state_dict(lambda: O.ResUNet(nc=NC[graph]), 5)
    ref = O.ResUNet(nc=NC[graph]).double().eval()
    ref.load_state_dict(sd)
    x = input_batch(18)
    with torch.no_grad():
        want = ref(x.double())
    got = resunet_fp16(sd, x, graph, round=False)
    assert float(rel_l2(got, want).max()) < 1e-12


def test_routing_weights_cover_every_tap_chunk_and_subpixel():
    for graph in ('chain', 'fused'):
        sd = routing_state_dict(NC[graph])
        for key, w in sd.items():
            if key == 'm_tail.weight':
                assert bool((w != 0).all())
                continue
            nz = w != 0
            if w.shape[-1] == 3 and key != 'm_head.weight':
                assert bool((nz.flatten(1).sum(1) == 1).all()), key                   # one product per output channel
                assert set(nz.sum((0, 1)).flatten().nonzero().flatten().tolist()) == set(range(9)), key
                assert bool(nz.any(0).any(-1).any(-1).all()), key                      # every input channel (every K chunk)
            elif key.startswith('m_up'):
                assert bool((nz.sum(0) == 1).all()), key                               # one input per (co, sub-pixel)
            elif key != 'm_head.weight':
                assert bool((nz.flatten(1).sum(1) == 1).all()), key
                assert bool(nz.sum((0, 1)).flatten().gt(0).all()), key                 # all four sub-pixels
                Ci = w.shape[1]
                kk = (nz.permute(0, 2, 3, 1).reshape(w.shape[0], 4 * Ci).float().argmax(1)) // 64
                assert set(kk.tolist()) == set(range(4 * Ci // 64)), key               # every 64-wide K slab of the GEMM
            vals = w[nz].double().abs()
            assert bool((torch.frexp(vals).mantissa == 0.5).all()), key               # powers of two: fp16-exact
        # the emulator asserts that no fp16 store overflows
        resunet_fp16(sd, input_batch(18), graph)


# mutant -> (graph, regime, metric)
MUTATIONS = [
    ('lo_l2', 'chain', 'routing', 'rel_max'),
    ('up_dx', 'chain', 'routing', 'rel_max'),
    ('tail_lastcol', 'chain', 'routing', 'region'),
    ('tail_lastcol', 'fused', 'dense', 'region'),
    ('seam', 'chain', 'dense', 'region'),
    ('kslab', 'fused', 'dense', 'rel_max'),
]


@pytest.fixture(scope='module')
def module_inputs():
    return input_batch()


def test_mutants_exceed_their_gates(module_inputs):
    """Each deliberate defect is >= 3x over the gate of its regime and metric on this module's own inputs and weights."""
    idx = {g: torch.tensor(COMPARE[g]) for g in COMPARE}
    base, report = {}, []
    for mutant, graph, regime, metric in MUTATIONS:
        sd = state_dict_for(regime, graph)
        x = module_inputs[idx[graph]]
        if (graph, regime) not in base:
            base[(graph, regime)] = resunet_fp16(sd, x, graph)
        m = metrics(resunet_fp16(sd, x, graph, mutant=mutant), base[(graph, regime)])
        gate = GATES[(regime, graph)][METRICS.index(metric)]
        report.append((mutant, graph, regime, metric, m[metric], gate))
    bad = [r for r in report if not r[4] >= 3 * r[5]]
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------
# GPU: kernel against the emulator
# ---------------------------------------------------------------------------------------------------
def _gpu_resunet(sd, graph, x):
    from models.ResUNet import ResUNet
    m = ResUNet(nc=NC[graph]).eval()
    m.load_state_dict(sd)
    m = m.cuda()
    with torch.no_grad():
        out = m(x.cuda())
    torch.cuda.synchronize()
    return out.cpu()


@pytest.fixture
def product_precision(monkeypatch):
    monkeypatch.setenv('GDECONV_PRECISION', 'fp16_umma')
    monkeypatch.delenv('GDECONV_CHUNK', raising=False)


@pytest.mark.gpu
@pytest.mark.parametrize('regime', REGIMES)
@pytest.mark.parametrize('graph', ['chain', 'fused'])
def test_kernel_matches_rounding_emulator(graph, regime, module_inputs, product_precision):
    sd = state_dict_for(regime, graph)
    got = _gpu_resunet(sd, graph, module_inputs)
    assert bool(torch.isfinite(got).all())
    idx = torch.tensor(COMPARE[graph])
    want = resunet_fp16(sd, module_inputs[idx], graph)
    m = metrics(got[idx], want)
    assert check_gates(m, regime, graph), (graph, regime, m, GATES[(regime, graph)])


# ---------------------------------------------------------------------------------------------------
# GPU: exact properties (bit equality where the design guarantees it)
# ---------------------------------------------------------------------------------------------------
def _bits_equal(a, b):
    return a.shape == b.shape and bool((a.view(torch.int32) == b.view(torch.int32)).all())


@pytest.mark.gpu
@pytest.mark.parametrize('graph', ['chain', 'fused'])
def test_zero_in_zero_out(graph, module_inputs, product_precision):
    sd = state_dict_for('dense', graph)
    x = module_inputs[:9].clone()
    x[4] = 0                                                   # a zero stamp between busy neighbours
    got = _gpu_resunet(sd, graph, x)
    assert bool((got[4] == 0).all())
    assert bool((_gpu_resunet(sd, graph, torch.zeros(3, 1, 48, 48)) == 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize('graph', ['chain', 'fused'])
def test_power_of_two_homogeneity(graph, module_inputs, product_precision):
    """The per-stamp power-of-two input scale makes f(2^k x) = 2^k f(x) exactly (no fp32 subnormals on either side)."""
    sd = state_dict_for('dense', graph)
    x = module_inputs[:54]
    base = _gpu_resunet(sd, graph, x)

    def smallest(v):
        a = v.abs().flatten(1)
        return torch.where(a > 0, a, torch.full_like(a, float('inf'))).min(1).values

    # stamps whose inputs and outputs stay normal fp32 numbers at every k (2^-126 < |.| * 2^k, no overflow)
    keep = (torch.minimum(smallest(x), smallest(base)) > 2.0 ** -80) & (torch.maximum(x.abs().flatten(1).max(1).values,
                                                                                      base.abs().flatten(1).max(1).values) < 2.0 ** 90)
    assert int(keep.sum()) >= 30
    x, base = x[keep], base[keep]
    base = _gpu_resunet(sd, graph, x)
    for k in (-40, -8, 3, 24):
        got = _gpu_resunet(sd, graph, x * 2.0 ** k)
        assert _bits_equal(got, base * 2.0 ** k), k


@pytest.mark.gpu
@pytest.mark.parametrize('graph', ['chain', 'fused'])
def test_neighbour_and_position_independence(graph, module_inputs, product_precision):
    """A probe stamp's output is bit-identical alone and anywhere in batches of 2 .. 301 among zero, border-heavy or NaN
    neighbours; finite stamps next to a NaN stamp are untouched by it."""
    sd = state_dict_for('dense', graph)
    probe = module_inputs[10:11]
    alone = _gpu_resunet(sd, graph, probe)
    g = torch.Generator().manual_seed(3)
    border = torch.randn(BATCH, 1, 48, 48, generator=g) * 4
    border[:, :, 3:45, 3:45] = 0
    nan = module_inputs.clone()
    nan[:, 0, 30, 11] = float('nan')
    for B in (2, 3, 75, 148, 149, 301):
        for kind, fill in (('zeros', torch.zeros(B, 1, 48, 48)), ('border', border[:B].clone()), ('nan', nan[:B].clone())):
            for pos in sorted({0, min(73, B - 1), min(74, B - 1), min(147, B - 1), min(148, B - 1), B - 1}):
                x = fill.clone()
                x[pos] = probe[0]
                got = _gpu_resunet(sd, graph, x)
                assert _bits_equal(got[pos:pos + 1], alone), (B, kind, pos)
                if kind == 'nan':
                    # containment: the finite probe next to NaN stamps is what it is alone (above); the NaN stamps may be NaN
                    assert bool(torch.isfinite(got[pos]).all())
    # finite neighbours of a NaN stamp
    x = module_inputs.clone()
    ref = _gpu_resunet(sd, graph, x)
    x[[1, 74, 148, 300], 0, 5, 40] = float('nan')
    got = _gpu_resunet(sd, graph, x)
    keep = torch.ones(BATCH, dtype=torch.bool)
    keep[[1, 74, 148, 300]] = False
    assert _bits_equal(got[keep], ref[keep])


@pytest.mark.gpu
@pytest.mark.parametrize('graph', ['chain', 'fused'])
def test_chunking_and_determinism(graph, module_inputs, monkeypatch):
    monkeypatch.setenv('GDECONV_PRECISION', 'fp16_umma')
    sd = state_dict_for('dense', graph)
    monkeypatch.delenv('GDECONV_CHUNK', raising=False)
    base = _gpu_resunet(sd, graph, module_inputs)
    assert _bits_equal(_gpu_resunet(sd, graph, module_inputs), base)               # two calls, same bits
    for chunk in ('1', '5', '148'):
        monkeypatch.setenv('GDECONV_CHUNK', chunk)
        assert _bits_equal(_gpu_resunet(sd, graph, module_inputs), base), chunk
