"""Rounding-faithful emulator of the tcgen05 ResUNet (precision mode fp16_umma), in float64 on the CPU.

``oracle.ref_models.ResUNet`` is the mathematics; this module is the same network evaluated with the roundings of the
product graph of ``resunet_chunk`` (galaxy-deconv_b200/csrc/api.cu): every value the kernels store is rounded where they
store it, everything else stays float64.  Against it the fp16 operand noise of the product path cancels, so a kernel
can be held to a gate far below the fp32-oracle tolerance (tests/test_resunet_rounding.py).

Rounding points (the kernels hold fp32 before every cvt.rn.f16, so fp16 values are made through fp32):
  * rn16(v) = v.float().half(): fp16 operand copies, ReLU(conv1) planes, space-to-depth copies;
  * hi/lo stream (conv_epilogue.cuh split8_hilo): hi = rn16(v), lo = rn16(fp32(v - hi)); read back as fp32(hi + lo)
    (hilo_pair);
  * every epilogue add is an fp32 add in the kernel's order: (acc + residual) + skip (k_conv_umma, conv_l2chain.cu);
  * tensor-core accumulators are fp32; here the sum is exact in float64 and rounded once to fp32.  With one nonzero
    product per output (routing weights) this is exactly what the tensor core returns;
  * m_head, the head recomputation of EPI_HT, the m_tail partial sums and k_tail_gather's stencil are fp32 fma chains
    in the kernels' order (conv_simt.cu k_head / k_tail_gather, conv_umma.cu ht_head / ht_tail, conv_l1chain.cu).

The two graphs:
  * 'chain' (nc 32..256, path G): level 0 in k_l1_chain (fp32 stream in tensor memory), level 1 in k_l2_chain (hi/lo
    stream; block 1 adds hi + lo of x2), levels 2-3 in k_conv_umma, m_tail as per-tap partial sums + k_tail_gather;
  * 'fused' (nc 64..512, path U): k_head writes rn16(x1); level 0 block 1 recomputes x1 in its epilogue (EPI_HT); every
    level uses the hi/lo stream; two 32-channel tail units.

``round=False`` drops every rounding and equals ``oracle.ref_models.ResUNet`` run in float64.  ``mutant`` injects one
deliberate defect (see MUTANTS); the test suite uses them to show its gates would catch a subtly wrong kernel.
"""
import torch
import torch.nn.functional as F

STAMP = 48
FP16_MAX = 65504.0

MUTANTS = (
    'lo_l2',          # the lo half dropped after the first ResBlock of level 2 (m_down3)
    'up_dx',          # dx sub-pixels swapped for channels 16..31 of m_up3's transposed conv
    'tail_lastcol',   # k_tail_gather uses the interior stencil class on the last column
    'seam',           # chain, level 0 DOWN: the top item's window is one row short (rows 0..26 instead of 0..27)
    'kslab',          # fused: input channels 448..511 (one 64-channel K slab) of m_body.0.res.2 are missing
)


def _r32(v):
    return v.float().double()


def _r16(v):
    h = v.float().half()
    if not torch.isfinite(h).all() and torch.isfinite(v).all():
        raise OverflowError(f'an fp16 store overflows: max |v| = {float(v.abs().max()):.4g} > {FP16_MAX}')
    return h.double()


class _Emu:
    def __init__(self, sd, rnd, mutant):
        if mutant is not None and mutant not in MUTANTS:
            raise ValueError(f'unknown mutant {mutant!r}; expected one of {MUTANTS}')
        self.sd = {k: v.detach().double().cpu() for k, v in sd.items()}
        self.rnd, self.mutant = rnd, mutant
        if mutant == 'kslab':
            w = self.sd['m_body.0.res.2.weight'].clone()
            if w.shape[1] != 512:
                raise ValueError("mutant 'kslab' needs the 64..512 configuration")
            w[:, 448:512] = 0
            self.sd['m_body.0.res.2.weight'] = w

    # ---- rounding points ----
    def f32(self, v):
        return _r32(v) if self.rnd else v

    def f16(self, v):
        return _r16(v) if self.rnd else v

    def hilo(self, v):
        if not self.rnd:
            return v, torch.zeros_like(v)
        hi = _r16(v)
        return hi, _r16(_r32(v - hi))

    def hilo_sum(self, hi, lo):
        return self.f32(hi + lo)

    # ---- layers (tensor-core GEMMs: fp16 operands and weights, fp32 accumulator) ----
    def w16(self, key):
        return self.f16(self.sd[key])

    def conv(self, a, key, rows=None):
        out = self.f32(F.conv2d(a, self.w16(key), padding=1))
        return out if rows is None else out * rows

    def down(self, a, key):
        return self.f32(F.conv2d(a, self.w16(key), stride=2))

    def up(self, a, key):
        u = self.f32(F.conv_transpose2d(a, self.w16(key), stride=2))
        if self.mutant == 'up_dx' and key == 'm_up3.0.weight':
            u = u.clone()
            even, odd = u[:, 16:32, :, 0::2].clone(), u[:, 16:32, :, 1::2].clone()
            u[:, 16:32, :, 0::2], u[:, 16:32, :, 1::2] = odd, even
        return u

    def relu16(self, v, rows=None):
        out = self.f16(torch.relu(v))
        return out if rows is None else out * rows

    # ---- fp32 fma chains ----
    def head_fma(self, t, acc=None):
        """acc + m_head(t): per channel an fma chain over the taps 0..8 (k_head, k_l1_chain head_row, ht_head)."""
        w = self.sd['m_head.weight']                                  # [C, 1, 3, 3]
        tp = F.pad(t, (1, 1, 1, 1))
        v = torch.zeros(t.shape[0], w.shape[0], STAMP, STAMP, dtype=torch.float64) if acc is None else acc
        for tap in range(9):
            ky, kx = divmod(tap, 3)
            v = self.f32(v + tp[:, :, ky:ky + STAMP, kx:kx + STAMP] * w[:, 0, ky, kx].view(1, -1, 1, 1))
        return v

    def tail_partials(self, v):
        """P[b, unit, tap] = sum over the unit's 32 channels of w_tail[tap][c] * v[c]: four fma chains over c = k mod 4,
        then (s0 + s1) + (s2 + s3) (lc_tail, ht_tail)."""
        w = self.sd['m_tail.weight'][0].reshape(-1, 9)                 # [C, tap]
        B, C = v.shape[:2]
        units = []
        for u in range(C // 32):
            s = []
            for j in range(4):
                acc = torch.zeros(B, 9, STAMP, STAMP, dtype=torch.float64)
                for k in range(j, 32, 4):
                    c = 32 * u + k
                    acc = self.f32(acc + v[:, c:c + 1] * w[c].view(1, 9, 1, 1))
                s.append(acc)
            units.append(self.f32(self.f32(s[0] + s[1]) + self.f32(s[2] + s[3])))
        return torch.stack(units, 1)                                   # [B, units, 9, 48, 48]

    def tail_gather(self, P, t, scale):
        """k_tail_gather: z = (sum_u sum_tap P[u][tap] shifted by the tap) + the class stencil of t, times the stamp's scale."""
        B, units = P.shape[:2]
        Pp = F.pad(P, (1, 1, 1, 1))
        s = torch.zeros(B, STAMP, STAMP, dtype=torch.float64)
        for u in range(units):
            for tap in range(9):
                ky, kx = divmod(tap, 3)
                s = self.f32(s + Pp[:, u, tap, ky:ky + STAMP, kx:kx + STAMP])
        c5 = self.stencils()                                            # [9 classes, 25]
        cls_y = torch.ones(STAMP, dtype=torch.long)
        cls_y[0], cls_y[-1] = 0, 2
        cls_x = cls_y.clone()
        if self.mutant == 'tail_lastcol':
            cls_x[-1] = 1
        cls = cls_y.view(-1, 1) * 3 + cls_x.view(1, -1)                 # [48, 48]
        tp = F.pad(t[:, 0], (2, 2, 2, 2))
        a = torch.zeros(B, STAMP, STAMP, dtype=torch.float64)
        for i in range(25):
            dy, dx = divmod(i, 5)
            a = self.f32(a + c5[cls, i] * tp[:, dy:dy + STAMP, dx:dx + STAMP])
        s = self.f32(s + a)
        return self.f32(s * scale.view(-1, 1, 1)).unsqueeze(1)

    def stencils(self):
        """m_tail(m_head(t)) as nine 5x5 stencils (launch_tail_gather): G[t2][t1] = sum_c tail[t2][c] head[t1][c] in float64
        stored fp32 (gd_pack_weights), collapsed per class in float64 and stored fp32."""
        h = self.sd['m_head.weight'][:, 0].reshape(-1, 9)               # [C, t1]
        tl = self.sd['m_tail.weight'][0].reshape(-1, 9)                 # [C, t2]
        G = self.f32(tl.t() @ h)                                        # [t2, t1]
        c5 = torch.zeros(9, 25, dtype=torch.float64)
        for cy in range(3):
            for cx in range(3):
                for t2 in range(9):
                    ty, tx = divmod(t2, 3)
                    if (cy == 0 and ty == 0) or (cy == 2 and ty == 2) or (cx == 0 and tx == 0) or (cx == 2 and tx == 2):
                        continue
                    for t1 in range(9):
                        c5[cy * 3 + cx, (ty + t1 // 3) * 5 + tx + t1 % 3] += G[t2, t1]
        return self.f32(c5)

    # ---- levels ----
    def block_pair_fp32_stream(self, X, S, blocks, rows=None):
        """Level 0 in k_l1_chain: two ResBlocks on the fp32 stream S (tensor memory) with first operand X, then rn16(stream).
        `rows` masks the image rows an item's window holds (mutant 'seam')."""
        T = self.relu16(self.conv(X, f'{blocks[0]}.res.0.weight', rows), rows)
        S = self.f32(self.conv(T, f'{blocks[0]}.res.2.weight', rows) + S)
        T = self.relu16(self.conv(self.f16(S), f'{blocks[1]}.res.0.weight', rows), rows)
        return self.f32(self.conv(T, f'{blocks[1]}.res.2.weight', rows) + S)

    def down_level(self, hi, res, pre):
        """Two ResBlocks on the hi/lo stream, block 1's residual `res` (fp32), then the strided conv: (x fp32, rn16(x))."""
        T = self.relu16(self.conv(hi, f'{pre}.0.res.0.weight'))
        hi, lo = self.hilo(self.f32(self.conv(T, f'{pre}.0.res.2.weight') + res))
        if self.mutant == 'lo_l2' and pre == 'm_down3':
            lo = torch.zeros_like(lo)
        T = self.relu16(self.conv(hi, f'{pre}.1.res.0.weight'))
        v = self.f32(self.conv(T, f'{pre}.1.res.2.weight') + self.hilo_sum(hi, lo))
        x = self.down(self.f16(v), f'{pre}.2.weight')
        return x, self.f16(x)

    def up_level(self, a, skip, pre):
        """Transposed conv (hi/lo out), two ResBlocks on the hi/lo stream, + U-Net skip (fp32) -> rn16."""
        hi, lo = self.hilo(self.up(a, f'{pre}.0.weight'))
        T = self.relu16(self.conv(hi, f'{pre}.1.res.0.weight'))
        hi, lo = self.hilo(self.f32(self.conv(T, f'{pre}.1.res.2.weight') + self.hilo_sum(hi, lo)))
        T = self.relu16(self.conv(hi, f'{pre}.2.res.0.weight'))
        v = self.f32(self.f32(self.conv(T, f'{pre}.2.res.2.weight') + self.hilo_sum(hi, lo)) + skip)
        return self.f16(v)

    def forward(self, x, graph):
        x = x.detach().double().cpu()
        if tuple(x.shape[1:]) != (1, STAMP, STAMP):
            raise ValueError(f'expected [B,1,48,48] stamps, got {tuple(x.shape)}')
        C0 = self.sd['m_head.weight'].shape[0]
        if graph not in ('chain', 'fused') or (graph == 'chain') != (C0 == 32):
            raise ValueError(f"graph {graph!r} does not fit nc[0] = {C0} ('chain' runs 32..256, 'fused' 64..512)")
        # k_scale_in / pow2_scale: t = in * 2^-e with e from frexpf(max |in|), output times 2^e
        amax = x.abs().flatten(1).max(1).values.float()
        e = torch.frexp(amax).exponent
        ok = (amax > 0) & torch.isfinite(amax)
        scale = torch.where(ok, torch.ldexp(torch.ones_like(amax), e), torch.ones_like(amax)).double()
        t = self.f32(x / scale.view(-1, 1, 1, 1))

        x1 = self.head_fma(t)
        if graph == 'chain':
            # k_l1_chain DOWN: stream = x1 (fp32), operand rn16(stream); the strided conv's x2 -> fp32 skip + hi/lo
            S = self.block_pair_fp32_stream(self.f16(x1), x1, ('m_down1.0', 'm_down1.1'))
            if self.mutant == 'seam':
                rows = torch.zeros(1, 1, STAMP, 1, dtype=torch.float64)
                rows[..., :27, :] = 1
                S_top = self.block_pair_fp32_stream(self.f16(x1) * rows, x1 * rows, ('m_down1.0', 'm_down1.1'), rows)
                S = torch.cat([S_top[:, :, :24], S[:, :, 24:]], 2)
            x2 = self.down(self.f16(S), 'm_down1.2.weight')
            hi2, lo2 = self.hilo(x2)
            # k_l2_chain DOWN: block 1's residual is hi + lo of x2
            x3, a3 = self.down_level(hi2, self.hilo_sum(hi2, lo2), 'm_down2')
        else:
            # k_head -> rn16(x1); level 0 block 1 recomputes x1 in the epilogue (EPI_HT): fma chain onto the accumulator
            T = self.relu16(self.conv(self.f16(x1), 'm_down1.0.res.0.weight'))
            hi, lo = self.hilo(self.head_fma(t, self.conv(T, 'm_down1.0.res.2.weight')))
            T = self.relu16(self.conv(hi, 'm_down1.1.res.0.weight'))
            v = self.f32(self.conv(T, 'm_down1.1.res.2.weight') + self.hilo_sum(hi, lo))
            x2 = self.down(self.f16(v), 'm_down1.2.weight')
            x3, a3 = self.down_level(self.f16(x2), x2, 'm_down2')
        x4, a4 = self.down_level(a3, x3, 'm_down3')
        # m_body and the skip x + x4
        T = self.relu16(self.conv(a4, 'm_body.0.res.0.weight'))
        hi, lo = self.hilo(self.f32(self.conv(T, 'm_body.0.res.2.weight') + x4))
        T = self.relu16(self.conv(hi, 'm_body.1.res.0.weight'))
        a = self.f16(self.f32(self.f32(self.conv(T, 'm_body.1.res.2.weight') + self.hilo_sum(hi, lo)) + x4))
        a = self.up_level(a, x3, 'm_up3')
        a = self.up_level(a, x2, 'm_up2')
        hi, lo = self.hilo(self.up(a, 'm_up1.0.weight'))
        if graph == 'chain':
            # k_l1_chain UP: stream = fp32(hi + lo) in tensor memory, operand rn16(stream)
            v = self.block_pair_fp32_stream(hi, self.hilo_sum(hi, lo), ('m_up1.1', 'm_up1.2'))
        else:
            T = self.relu16(self.conv(hi, 'm_up1.1.res.0.weight'))
            hi, lo = self.hilo(self.f32(self.conv(T, 'm_up1.1.res.2.weight') + self.hilo_sum(hi, lo)))
            T = self.relu16(self.conv(hi, 'm_up1.2.res.0.weight'))
            v = self.f32(self.conv(T, 'm_up1.2.res.2.weight') + self.hilo_sum(hi, lo))
        # m_tail(v + x1) = per-tap partial sums of v + the stencil of t
        return self.tail_gather(self.tail_partials(v), t, scale)


@torch.no_grad()
def resunet_fp16(state_dict, x, graph='chain', round=True, mutant=None):
    """ResUNet forward of the fp16_umma product graph on [B,1,48,48] stamps -> float64 [B,1,48,48] (CPU).

    state_dict: a ResUNet state_dict (models/ResUNet.py keys).  graph: 'chain' for nc 32..256, 'fused' for 64..512.
    round=False: no rounding at all (equals oracle.ref_models.ResUNet in float64).  mutant: one of MUTANTS or None."""
    return _Emu(state_dict, round, mutant).forward(x, graph)
