"""Host runtime between the reference-shaped nn.Modules (models/*.py) and the C ABI of libgdeconv.

torch is used for device memory, streams and the nn.Module protocol only; every computation on stamps is a call
into libgdeconv.so on the current CUDA stream.  There is no CPU path: CPU tensors raise.
"""
from __future__ import annotations

import copy
import ctypes as C
import os
import threading

import torch

from . import _lib
from ._lib import check, lib

STAMP = 48
NPIX = STAMP * STAMP
_DEFAULT_CHUNK = 8192      # stamps per pass through the layer graph: long kernels beat L2 residency (profiles/ablation_r01.md)


def default_precision() -> str:
    """Arithmetic of the inner ResUNet convolutions: env GDECONV_PRECISION in {fp16_umma, fp32_simt, fp16_simt}."""
    p = os.environ.get('GDECONV_PRECISION', 'fp16_umma')
    if p not in _lib.PRECISIONS:
        raise ValueError(f'GDECONV_PRECISION={p!r}; expected one of {sorted(_lib.PRECISIONS)}')
    return p


def max_chunk(arch=_lib.ARCH_G) -> int:
    """Upper bound on the stamps per pass through the layer graph (env GDECONV_CHUNK).  Long kernels beat L2 residency on
    this path (profiles/ablation_r01.md), so the default is large: 8192 stamps = 22 GB of workspace for path G,
    4096 = 22 GB for the twice-as-wide path U."""
    env = os.environ.get('GDECONV_CHUNK')
    c = int(env) if env else (_DEFAULT_CHUNK if arch == _lib.ARCH_G else _DEFAULT_CHUNK // 2)
    # the row decode of the kernels is exact below 2^26 GEMM rows (~27.9 k stamps): larger requests are clamped here and
    # rejected by gd_workspace_bytes / gd_workspace_init, never mis-decoded
    return max(1, min(c, int(lib.gd_max_chunk())))


def launch_count() -> int:
    return int(lib.gd_launch_count())


def _stream(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t) -> C.c_void_p:
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def require_cuda_stamps(name, t, batch=None):
    """The boundary's input contract (SURVEY.md section 8b): fp32 CUDA [B,1,48,48]; returns it contiguous."""
    if not torch.is_tensor(t):
        raise TypeError(f'{name} must be a torch.Tensor')
    if not t.is_cuda:
        raise RuntimeError(f'{name} is on {t.device}: gdeconv has no CPU path (CUDA sm_100a only)')
    if t.dtype != torch.float32:
        raise TypeError(f'{name} must be float32, got {t.dtype}')
    if t.dim() != 4 or t.shape[1] != 1 or t.shape[2] != STAMP or t.shape[3] != STAMP:
        raise ValueError(f'{name} must have shape [B,1,{STAMP},{STAMP}], got {tuple(t.shape)}')
    if batch is not None and t.shape[0] != batch:
        raise ValueError(f'{name} has batch {t.shape[0]}, expected {batch}')
    return t.detach().contiguous()


def _alpha_vector(alpha, batch, device):
    """alpha as the reference passes it ([B,1,1,1], [1,1,1,1] or a scalar) -> contiguous [B] fp32 on device."""
    if not torch.is_tensor(alpha):
        alpha = torch.tensor(float(alpha))
    a = alpha.detach().to(device=device, dtype=torch.float32).reshape(-1)
    if a.numel() == 1 and batch != 1:
        a = a.expand(batch)
    if a.numel() != batch:
        raise ValueError(f'alpha has {a.numel()} elements for a batch of {batch}')
    return a.contiguous()


# ---------------------------------------------------------------------------------------------------
# workspaces: caller-owned device memory, cached per (device, arch, precision, chunk)
# ---------------------------------------------------------------------------------------------------
_ws_lock = threading.Lock()
_ws_cache = {}


def _chunk_for(batch, arch=_lib.ARCH_G):
    """Workspace capacity for a batch: the batch is cut into the fewest chunks that respect the cap, of (nearly) equal
    size -- a short ragged last chunk would waste whole waves of the persistent kernels."""
    cap = max(1, max_chunk(arch))
    n = max(1, -(-batch // cap))
    per = -(-max(batch, 1) // n)
    if per <= 256:                      # small batches: powers of two keep the number of distinct workspaces low
        c = 1
        while c < per:
            c *= 2
        return min(c, cap)
    return min(-(-per // 256) * 256, max(cap, 256))


class _WsRelease:
    """Rides on a workspace tensor: unregisters the workspace from the library when the tensor object dies, i.e. before its
    memory can go back to the allocator and be handed to an unrelated buffer at the same address."""

    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        try:
            lib.gd_workspace_release(C.c_void_p(self.ptr))
        except Exception:
            pass


def _workspace(device, arch, prec, chunk, slot=0):
    """Scratch memory for `chunk` stamps.  Keyed by the CURRENT STREAM as well: kernels of one stream are ordered, two streams (or two
    host threads driving different streams) must not share activations, and nothing else orders them."""
    key = (device.index, arch, prec, chunk, slot, torch.cuda.current_stream(device).cuda_stream)
    with _ws_lock:
        hit = _ws_cache.get(key)
        if hit is not None:
            return hit
        nbytes = int(lib.gd_workspace_bytes(arch, prec, chunk))
        if nbytes == 0:
            raise RuntimeError('gd_workspace_bytes rejected the configuration')
        # at most two chunk sizes per (device, arch, precision) (each with its stream slots): drop the oldest before a third
        sizes = []
        for k in _ws_cache:
            if k[:3] == key[:3] and k[3] != chunk and k[3] not in sizes:
                sizes.append(k[3])
        for old in sizes[:-1] if len(sizes) >= 2 else []:
            for k in [k for k in _ws_cache if k[:3] == key[:3] and k[3] == old]:
                del _ws_cache[k]
        buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        check(lib.gd_workspace_init(_ptr(buf), nbytes, arch, prec, chunk, _stream(device)))
        buf._gd_release = _WsRelease(buf.data_ptr())
        _ws_cache[key] = (buf, nbytes)
        return buf, nbytes


def drop_workspaces():
    with _ws_lock:
        _ws_cache.clear()


# Chunks of a large batch alternate between the caller's stream and one side stream per device (each with its own
# workspace): every kernel of the path is a persistent one-CTA-per-SM kernel, so while one chunk's kernel drains its last
# work items the other chunk's next kernel already fills the freed SMs instead of leaving them idle until the dependent
# launch starts (GDECONV_STREAMS=1: one stream, chunks back to back inside gd_admm_forward).
_side_streams = {}


def n_streams() -> int:
    try:
        return 2 if int(os.environ.get('GDECONV_STREAMS', '2')) >= 2 else 1
    except ValueError:
        return 2


def _side_stream(device):
    s = _side_streams.get(device.index)
    if s is None:
        s = _side_streams[device.index] = torch.cuda.Stream(device=device)
    return s


# ---------------------------------------------------------------------------------------------------
# packed weights
# ---------------------------------------------------------------------------------------------------
class _Packed:
    def __init__(self, handle, device):
        self.handle, self.device = handle, device

    def __del__(self):
        try:
            if self.handle:
                lib.gd_free_weights(self.handle)
        except Exception:
            pass


def pack_state_dict(state_dict, arch, n_iters, precision, device) -> _Packed:
    """state_dict (the reference's key layout) -> GdWeights on `device` (gd_pack_weights)."""
    names, arrays = [], []
    for k, v in state_dict.items():
        if not torch.is_tensor(v) or not v.dtype.is_floating_point or v.dim() > 4:
            continue                      # num_batches_tracked (int64) is not part of the arithmetic
        names.append(k.encode())
        arrays.append(v.detach().to('cpu', torch.float32).contiguous())
    descs = (_lib.GdTensorDesc * len(names))()
    for i, (n, a) in enumerate(zip(names, arrays)):
        descs[i].name = n
        descs[i].data = a.data_ptr()
        descs[i].ndim = a.dim()
        for d in range(a.dim()):
            descs[i].shape[d] = a.shape[d]
    out = C.c_void_p()
    check(lib.gd_pack_weights(arch, n_iters, descs, len(names), _lib.PRECISIONS[precision], device.index, C.byref(out)))
    return _Packed(out, device)


def graph_max_batch() -> int:
    """Batches up to this size run as ONE replayed CUDA graph (env GDECONV_GRAPH_MAX, 0 disables): a forward pass is ~300 kernel
    launches, which dominate the latency of a single galaxy (BASELINE config 1, tutorials/deconv_cpu.ipynb cell 7)."""
    try:
        return max(0, int(os.environ.get('GDECONV_GRAPH_MAX', '64')))
    except ValueError:
        return 64


class AdmmEngine:
    """Per-module cache of packed weights + the forward calls.  The module's parameters stay the source of truth:
    the pack is redone whenever a parameter/buffer is replaced (load_state_dict, .to(device)) or modified in place
    (``_version`` bump).  Updates that bypass autograd's version counter (``param.data.copy_()``) need ``invalidate()``."""

    def __init__(self, module, arch, n_iters):
        self._module = module
        self.arch, self.n_iters = arch, n_iters
        self._packed = {}        # (device index, precision) -> (signature, _Packed)
        self._tensors = None     # cached list of the module's parameter / buffer tensors (the signature walks it, not state_dict())
        self._graphs = {}        # (device index, precision, llh, v0, B) -> captured forward

    # engines hold ctypes handles and CUDA graphs: copies / pickles of the owning module start with an empty cache
    def __deepcopy__(self, memo):
        # bind the copy to the COPY of the owning module (already in `memo` while copy.deepcopy(model) walks its attributes)
        return AdmmEngine(copy.deepcopy(self._module, memo), self.arch, self.n_iters)

    def __getstate__(self):
        return dict(_module=self._module, arch=self.arch, n_iters=self.n_iters)

    def __setstate__(self, st):
        self.__init__(st['_module'], st['arch'], st['n_iters'])

    def invalidate(self):
        """Drop packed weights and captured graphs (call after in-place updates through ``.data``, which do not bump ``_version``)."""
        self._packed.clear()
        self._graphs.clear()
        self._tensors = None

    def _signature(self):
        # (data_ptr, _version) of every parameter / buffer.  The tensor list is cached: nn.Module replaces the tensor OBJECTS on
        # load_state_dict(assign=True) / .to(device) of parameters only through _parameters / _buffers, whose identity we check.
        m = self._module
        ts = self._tensors
        if ts is None or not hasattr(m, 'parameters'):
            sd = m.state_dict(keep_vars=True)
            if not hasattr(m, 'parameters'):
                return tuple((k, v.data_ptr(), v._version) for k, v in sd.items())
            ts = self._tensors = list(sd.values())
        sig = tuple((v.data_ptr(), v._version) for v in ts)
        return sig

    def weights(self, device, precision):
        key = (device.index, precision)
        sig = self._signature()
        hit = self._packed.get(key)
        if hit is None or hit[0] != sig:
            # the cached tensor list may be stale (parameters replaced): rebuild it and compare once more before repacking
            self._tensors = None
            sig = self._signature()
            if hit is None or hit[0] != sig:
                hit = (sig, pack_state_dict(self._module.state_dict(), self.arch, self.n_iters, precision, device))
                self._packed[key] = hit
                self._graphs.clear()
        return hit[1]

    def _graphed(self, w, y, psf, a, llh, v0, precision, ws, nbytes):
        """Small batches: the whole forward (SubNet, prologue, n x [x-update, ~35 conv launches, tail]) is captured ONCE per
        (weights, batch size) into a CUDA graph over static buffers and replayed -- three small device copies + one graph launch
        instead of ~300 kernel launches."""
        B, dev = y.shape[0], y.device
        key = (dev.index, precision, llh, int(v0), B, nbytes)
        g = self._graphs.get(key)
        cur = torch.cuda.current_stream(dev)
        if g is None:
            st = dict(y=torch.empty_like(y), psf=torch.empty_like(psf), a=torch.empty_like(a), out=torch.empty_like(y), ws=ws, w=w)   # ws / w: kept alive

            def run(stream):
                check(lib.gd_admm_forward(w.handle, llh, int(v0), _ptr(st['y']), _ptr(st['psf']), _ptr(st['a']), _ptr(st['out']),
                                          None, None, B, _ptr(ws), nbytes, C.c_void_p(stream.cuda_stream)))
            st['y'].copy_(y); st['psf'].copy_(psf); st['a'].copy_(a)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                run(side)                                   # warm-up outside capture (lazy per-kernel attributes, occupancy queries)
            cur.wait_stream(side)
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                run(torch.cuda.current_stream(dev))
            st['graph'], st['launches'] = graph, None
            if len(self._graphs) >= 8:
                self._graphs.pop(next(iter(self._graphs)))
            g = self._graphs[key] = st
        g['y'].copy_(y, non_blocking=True); g['psf'].copy_(psf, non_blocking=True); g['a'].copy_(a, non_blocking=True)
        g['graph'].replay()
        return g['out'].clone()

    def admm(self, y, psf, alpha, llh=_lib.LLH_GAUSSIAN, v0_over_alpha=False, want_rho=False, want_analysis=False,
             precision=None, times_alpha=False, xdense=None):
        """xdense: an XDenseEngine -> the Z-update is that XDenseUNet (gd_admm_forward_xdense, arch U only) instead of the ResUNet."""
        v0_over_alpha = int(bool(v0_over_alpha)) | (2 if times_alpha else 0)          # flag word of gd_admm_forward
        y = require_cuda_stamps('y', y)
        B, dev = y.shape[0], y.device
        psf = require_cuda_stamps('psf', psf, B)
        a = _alpha_vector(alpha, B, dev)
        precision = precision or default_precision()
        n_rho = self.n_iters if self.arch == _lib.ARCH_G else 2 * self.n_iters
        with torch.cuda.device(dev):
            w = self.weights(dev, precision)
            ws, nbytes = _workspace(dev, self.arch, _lib.PRECISIONS[precision], _chunk_for(B, self.arch))
            out = torch.empty_like(y)
            rho = torch.empty(B, n_rho, device=dev) if want_rho else None
            ana = None
            if want_analysis:
                shape = (self.n_iters, 3, B, 1, STAMP, STAMP) if self.arch == _lib.ARCH_G else (self.n_iters + 1, 5, B, 1, STAMP, STAMP)
                ana = torch.empty(shape, device=dev)
            chunk = _chunk_for(B, self.arch)
            if xdense is not None:
                xw = xdense._weights(dev)
                xchunk = xdense._chunk(min(B, chunk))
                xws, xbytes = _xd_workspace(dev, xchunk)
                check(lib.gd_admm_forward_xdense(w.handle, xw.handle, llh, int(v0_over_alpha), _ptr(y), _ptr(psf), _ptr(a), _ptr(out), _ptr(rho),
                                                 _ptr(ana), B, _ptr(ws), nbytes, _ptr(xws), xbytes, xchunk, _stream(dev)))
                return out, rho, ana
            if ana is None and rho is None and 0 < B <= graph_max_batch() and not torch.cuda.is_current_stream_capturing():
                return self._graphed(w, y, psf, a, llh, v0_over_alpha, precision, ws, nbytes), None, None
            if ana is None and B > chunk and n_streams() == 2:
                # two chunks in flight: even chunks on the caller's stream, odd chunks on the side stream
                ws2, _ = _workspace(dev, self.arch, _lib.PRECISIONS[precision], chunk, slot=1)
                cur, side = torch.cuda.current_stream(dev), _side_stream(dev)
                side.wait_stream(cur)
                for t in (y, psf, a, out, rho):
                    if t is not None:
                        t.record_stream(side)
                for i, c0 in enumerate(range(0, B, chunk)):
                    nb = min(chunk, B - c0)
                    st, wsi = (cur, ws) if i % 2 == 0 else (side, ws2)
                    check(lib.gd_admm_forward(w.handle, llh, int(v0_over_alpha), _ptr(y[c0:c0 + nb]), _ptr(psf[c0:c0 + nb]),
                                              _ptr(a[c0:c0 + nb]), _ptr(out[c0:c0 + nb]), _ptr(rho[c0:c0 + nb]) if rho is not None else None,
                                              None, nb, _ptr(wsi), nbytes, C.c_void_p(st.cuda_stream)))
                cur.wait_stream(side)
            else:
                check(lib.gd_admm_forward(w.handle, llh, int(v0_over_alpha), _ptr(y), _ptr(psf), _ptr(a), _ptr(out),
                                          _ptr(rho), _ptr(ana), B, _ptr(ws), nbytes, _stream(dev)))
        return out, rho, ana

    # ---- host-resident batches: chunk-pipelined H2D / compute / D2H ----------------------------------------------------
    def _host_state(self, dev, prec, cap):
        key = (dev.index, prec, cap)
        st = self.__dict__.setdefault('_host', {}).get(key)
        if st is None:
            mk = lambda *shape: [torch.empty(*shape, device=dev) for _ in range(2)]
            st = dict(y=mk(cap, 1, STAMP, STAMP), psf=mk(cap, 1, STAMP, STAMP), a=mk(cap), out=mk(cap, 1, STAMP, STAMP),
                      h2d=torch.cuda.Stream(device=dev), d2h=torch.cuda.Stream(device=dev),
                      ev_h2d=[torch.cuda.Event() for _ in range(2)], ev_comp=[torch.cuda.Event() for _ in range(2)],
                      ev_d2h=[torch.cuda.Event() for _ in range(2)])
            self._host.clear()                      # one staging set per engine
            self._host[key] = st
        return st

    @staticmethod
    def _host_plan(B, cap):
        """Chunk sizes for a host-resident batch: the fewest balanced chunks that fit the workspace (long persistent kernels).  In
        a loop of calls the first chunk's H2D and the last chunk's D2H overlap the neighbouring calls' compute (copy streams)."""
        parts = max(1, -(-B // cap))
        per = -(-B // parts)
        return [min(per, B - i * per) for i in range(parts) if B - i * per > 0]

    def admm_host(self, y, psf, alpha, out=None, want_e=True, device=None, precision=None):
        """model(y, psf, alpha) for a batch that lives in (pinned) HOST memory: the batch is cut into chunks and chunk k+1's
        host->device copies and chunk k-1's device->host copy run on two copy streams while chunk k computes (one
        cudaMemcpyAsync per tensor and chunk, double-buffered device staging).  Returns (out_host, e12) with out_host the
        deconvolved stamps in host memory (``out`` if given) and e12 [B,2] the moment ellipticities on the device (or None).
        Stream-ordered on the current stream: synchronize it before reading out_host."""
        for name, t in (('y', y), ('psf', psf)):
            if not torch.is_tensor(t) or t.is_cuda or t.dtype != torch.float32 or t.dim() != 4 or tuple(t.shape[1:]) != (1, STAMP, STAMP):
                raise ValueError(f'admm_host: {name} must be a float32 host tensor [B,1,{STAMP},{STAMP}]')
        B = y.shape[0]
        if psf.shape[0] != B:
            raise ValueError('admm_host: y and psf differ in batch size')
        y, psf = y.contiguous(), psf.contiguous()
        a = alpha.detach().to(torch.float32).reshape(-1)
        a = (a.expand(B) if a.numel() == 1 and B != 1 else a).contiguous()
        if a.numel() != B:
            raise ValueError(f'alpha has {a.numel()} elements for a batch of {B}')
        dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        precision = precision or default_precision()
        prec = _lib.PRECISIONS[precision]
        if out is None:
            out = torch.empty(B, 1, STAMP, STAMP).pin_memory()
        with torch.cuda.device(dev):
            w = self.weights(dev, precision)
            cap = _chunk_for(B, self.arch)
            sizes = self._host_plan(B, cap)
            st = self._host_state(dev, prec, cap)
            wss = [_workspace(dev, self.arch, prec, cap, slot=s) for s in range(2)]
            cur = torch.cuda.current_stream(dev)
            side = _side_stream(dev) if len(sizes) > 1 and n_streams() == 2 else cur
            if side is not cur:
                side.wait_stream(cur)
            e12 = torch.empty(B, 2, device=dev) if want_e else None
            if e12 is not None and side is not cur:
                e12.record_stream(side)
            c0 = 0
            for i, nb in enumerate(sizes):
                s = i & 1
                comp = cur if s == 0 else side
                with torch.cuda.stream(st['h2d']):
                    st['h2d'].wait_event(st['ev_comp'][s])           # the slot's previous chunk no longer reads its inputs
                    st['y'][s][:nb].copy_(y[c0:c0 + nb], non_blocking=True)
                    st['psf'][s][:nb].copy_(psf[c0:c0 + nb], non_blocking=True)
                    st['a'][s][:nb].copy_(a[c0:c0 + nb], non_blocking=True)
                    st['ev_h2d'][s].record(st['h2d'])
                comp.wait_event(st['ev_h2d'][s])
                comp.wait_event(st['ev_d2h'][s])                     # the slot's previous result has left the device
                check(lib.gd_admm_forward(w.handle, _lib.LLH_GAUSSIAN, 0, _ptr(st['y'][s]), _ptr(st['psf'][s]), _ptr(st['a'][s]),
                                          _ptr(st['out'][s]), None, None, nb, _ptr(wss[s][0]), wss[s][1], C.c_void_p(comp.cuda_stream)))
                if e12 is not None:
                    check(lib.gd_moments_e(_ptr(st['out'][s]), _ptr(e12[c0:c0 + nb]), nb, C.c_void_p(comp.cuda_stream)))
                st['ev_comp'][s].record(comp)
                with torch.cuda.stream(st['d2h']):
                    st['d2h'].wait_event(st['ev_comp'][s])
                    out[c0:c0 + nb].copy_(st['out'][s][:nb], non_blocking=True)
                    st['ev_d2h'][s].record(st['d2h'])
                c0 += nb
            if side is not cur:
                cur.wait_stream(side)
            cur.wait_stream(st['d2h'])
        return out, e12

    def resunet(self, x, precision=None):
        x = require_cuda_stamps('x', x)
        dev = x.device
        precision = precision or default_precision()
        with torch.cuda.device(dev):
            w = self.weights(dev, precision)
            ws, nbytes = _workspace(dev, self.arch, _lib.PRECISIONS[precision], _chunk_for(x.shape[0], self.arch))
            out = torch.empty_like(x)
            check(lib.gd_resunet_forward(w.handle, _ptr(x), _ptr(out), x.shape[0], _ptr(ws), nbytes, _stream(dev)))
        return out

    def subnet(self, psf, alpha):
        psf = require_cuda_stamps('kernel', psf)
        B, dev = psf.shape[0], psf.device
        a = _alpha_vector(alpha, B, dev)
        n_rho = self.n_iters if self.arch == _lib.ARCH_G else 2 * self.n_iters
        with torch.cuda.device(dev):
            w = self.weights(dev, default_precision())
            rho = torch.empty(B, n_rho, device=dev)
            check(lib.gd_subnet_forward(w.handle, _ptr(psf), _ptr(a), _ptr(rho), B, _stream(dev)))
        return rho


def resunet_forward(engine: AdmmEngine, x, precision=None):
    return engine.resunet(x, precision)


# ---------------------------------------------------------------------------------------------------
# weight-free entry points
# ---------------------------------------------------------------------------------------------------
def fft_solver(kind, y, psf, alpha=None, n_iters=0, lam=1.0):
    y = require_cuda_stamps('y', y)
    B, dev = y.shape[0], y.device
    psf = require_cuda_stamps('psf', psf, B)
    a = _alpha_vector(alpha, B, dev) if alpha is not None else None
    out = torch.empty_like(y)
    with torch.cuda.device(dev):
        check(lib.gd_fft_solver(kind, int(n_iters), float(lam), _ptr(y), _ptr(psf), _ptr(a), _ptr(out), B, _stream(dev)))
    return out


def conv_fft_batch(x, psf, adjoint=False):
    x = require_cuda_stamps('x', x)
    psf = require_cuda_stamps('psf', psf, x.shape[0])
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        check(lib.gd_conv_fft(_ptr(x), _ptr(psf), _ptr(out), int(bool(adjoint)), x.shape[0], _stream(x.device)))
    return out


def psf_to_otf(ker, size):
    """psf_to_otf(ker, size) of utils/utils_torch.py:79-92 on the device: (psf, otf) with psf fp32 and otf complex64, both
    of shape ``size`` = (B,1,48,48); ``ker`` is [1 or B,1,kh,kw] fp32 CUDA."""
    size = tuple(int(v) for v in size)
    if len(size) != 4 or size[1] != 1 or size[2] != STAMP or size[3] != STAMP:
        raise ValueError(f'psf_to_otf: size must be (B,1,{STAMP},{STAMP}), got {size}')
    if not torch.is_tensor(ker) or not ker.is_cuda:
        raise RuntimeError('psf_to_otf: the kernel must be a CUDA tensor (gdeconv has no CPU path)')
    if ker.dtype != torch.float32 or ker.dim() != 4 or ker.shape[1] != 1 or ker.shape[0] not in (1, size[0]):
        raise ValueError(f'psf_to_otf: kernel must be float32 [1 or {size[0]},1,kh,kw], got {ker.dtype} {tuple(ker.shape)}')
    ker = ker.detach().contiguous()
    dev, B = ker.device, size[0]
    psf = torch.empty(size, device=dev)
    otf = torch.empty(size + (2,), device=dev)
    with torch.cuda.device(dev):
        check(lib.gd_psf_to_otf(_ptr(ker), ker.shape[0], ker.shape[2], ker.shape[3], _ptr(psf), _ptr(otf), B, _stream(dev)))
    return psf, torch.view_as_complex(otf)


def conv_otf(H, x):
    """conv_fft_batch(H, x) of utils/utils_torch.py:46-50: ifft2(fft2(x) * H).real with a full complex spectrum H [1 or B,1,48,48]."""
    x = require_cuda_stamps('x', x)
    B, dev = x.shape[0], x.device
    if not torch.is_tensor(H) or not H.is_cuda or H.dtype != torch.complex64:
        raise TypeError('conv_fft_batch: H must be a complex64 CUDA tensor')
    if H.dim() != 4 or H.shape[1] != 1 or H.shape[2] != STAMP or H.shape[3] != STAMP or H.shape[0] not in (1, B):
        raise ValueError(f'conv_fft_batch: H must have shape [1 or {B},1,{STAMP},{STAMP}], got {tuple(H.shape)}')
    Hr = torch.view_as_real(H.detach().resolve_conj().contiguous())
    out = torch.empty_like(x)
    with torch.cuda.device(dev):
        check(lib.gd_conv_otf(_ptr(Hr), H.shape[0], _ptr(x), _ptr(out), B, _stream(dev)))
    return out


def moments_e(img):
    img = require_cuda_stamps('img', img)
    e = torch.empty(img.shape[0], 2, device=img.device)
    with torch.cuda.device(img.device):
        check(lib.gd_moments_e(_ptr(img), _ptr(e), img.shape[0], _stream(img.device)))
    return e


def adaptive_moments(img, guess_sigma=3.0):
    """Adaptive second moments of every stamp (gd_adaptive_moments, csrc/shape.cu): an elliptical Gaussian weight, started at
    pixel (24, 24) with sigma = ``guess_sigma`` px, iterated until it matches the stamp's own weighted centroid and second moments.
    ``img`` is fp32 CUDA [B,1,48,48]; the work runs on the current stream of its device.  Returns a dict:
    flux [B], centroid [B,2] (x, y; x = column), M [B,3] (Mxx, Mxy, Myy, px^2), e [B,2] (distortion, as moments_e),
    sigma [B] = det(M)^(1/4), status [B] int32 (_lib.SHAPE_*: OK, MAXITER, FLUX, MOMENTS, CENTROID) and n_iter [B] int32 passes.
    The floats are NaN wherever status is not OK."""
    img = require_cuda_stamps('img', img)
    B, dev = img.shape[0], img.device
    shape = torch.empty(B, 8, device=dev)
    info = torch.empty(B, 2, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib.gd_adaptive_moments(_ptr(img), B, float(guess_sigma), _ptr(shape), _ptr(info), _stream(dev)))
        M = shape[:, 3:6]
        sigma = (M[:, 0] * M[:, 2] - M[:, 1] * M[:, 1]).pow(0.25)
    return dict(flux=shape[:, 0], centroid=shape[:, 1:3], M=M, e=shape[:, 6:8], sigma=sigma, status=info[:, 0], n_iter=info[:, 1])


def fpfs(img, psf=None, sigma=3.5, const=0.0):
    """FPFS shear estimation of every stamp (gd_fpfs, csrc/fpfs.cu; the estimator behind the reference's `estimate_shear`,
    built from Li, Li & Mandelbaum 2018 without bit parity with the fpfs package): the power spectrum of ``img``, divided by the
    normalised PSF power of ``psf`` (None: a delta PSF), projected on shapelet modes of scale ``sigma`` px.  ``img`` is fp32
    CUDA [B,1,48,48], ``psf`` None, [1,1,48,48] or [B,1,48,48] on the same device (its normalisation and centring do not
    matter); ``const`` >= 0 is added to M00 in the denominators.  The work runs on the current stream of img's device.
    Returns a dict: modes [B,6] (M00, M22c, M22s, M40, M42c, M42s), e [B,2], R [B] (the shear response) and g [B,2] = e / R,
    the per-galaxy shear; the ensemble shear is e.sum(0) / R.sum()."""
    img = require_cuda_stamps('img', img)
    B, dev = img.shape[0], img.device
    if psf is not None:
        if torch.is_tensor(psf) and psf.is_cuda and psf.device != dev:
            raise ValueError(f'psf is on {psf.device}, img on {dev}')
        psf = require_cuda_stamps('psf', psf)
        if psf.shape[0] not in (1, B):
            raise ValueError(f'psf must have batch 1 or {B}, got {psf.shape[0]}')
        if B == 0:
            psf = None
    modes = torch.empty(B, 6, device=dev)
    ell = torch.empty(B, 3, device=dev)
    with torch.cuda.device(dev):
        check(lib.gd_fpfs(_ptr(img), _ptr(psf), 0 if psf is None else psf.shape[0], B, float(sigma), float(const), _ptr(modes),
                          _ptr(ell), _stream(dev)))
        e, R = ell[:, :2], ell[:, 2]
        g = e / R[:, None]
    return dict(modes=modes, e=e, R=R, g=g)


def metacal(img, psf=None, delta=0.01, reconv_sigma=2.5, guess_sigma=3.0, images=False, noise_sigma=None, noise=None, seed=0, start=0):
    """Metacalibration of every stamp (gd_metacal, csrc/metacal.cu): ``img`` deconvolved by ``psf`` (None: no deconvolution, for
    stamps that are already deconvolved), sheared by (0,0), (+delta,0), (-delta,0), (0,+delta), (0,-delta), reconvolved with a
    round Gaussian of sigma ``reconv_sigma`` px (one for the whole call) and measured with adaptive moments started at
    ``guess_sigma`` px.  ``img`` is fp32 CUDA [B,1,48,48], ``psf`` None, [1,1,48,48] or [B,1,48,48] on the same device (its
    normalisation does not matter; it is centred on pixel (24, 24)).  The work runs on the current stream of img's device.

    Fix-noise (gd_metacal_fixnoise, Sheldon & Huff 2017): with ``noise_sigma`` or ``noise`` (not both), image j becomes
    T_j(img) + rot90^-1(T_j(rot90(n))) for a noise field n of each stamp, which cancels the response of the sheared noise; the
    images then carry twice the stamp's noise variance.  ``noise_sigma`` (a float, or fp32 CUDA [1] or [B]) generates
    n = sigma N(start + i, p) from the counter hash of gdsynth on streams 60 / 61 and ``seed`` (a negative sigma negates the field, a
    non-finite one fails the stamp); ``noise`` is the caller's unrotated field, fp32 CUDA [B,1,48,48] (for a Wiener output pass the
    Wiener filter of sigma N).  With neither, the call is gd_metacal.

    Returns a dict: e [B,5,2] and status, n_iter [B,5] int32 (_lib.SHAPE_*) of the five images in that order, the response
    R [B,2,2] with R[:, i, j] = (e_i(+delta_j) - e_i(-delta_j)) / (2 delta), the per-galaxy shear g [B,2] = R^-1 e(noshear) (NaN
    unless all five statuses are OK) and, with ``images=True``, the five images [B,5,1,48,48].  The shear of an ensemble is
    mean(R)^-1 mean(e(noshear)) over the stamps whose five statuses are OK."""
    if noise is not None and noise_sigma is not None:
        raise ValueError('metacal: pass noise or noise_sigma, not both')
    fix = noise is not None or noise_sigma is not None
    img = require_cuda_stamps('img', img)
    B, dev = img.shape[0], img.device
    if psf is not None:
        if torch.is_tensor(psf) and psf.is_cuda and psf.device != dev:
            raise ValueError(f'psf is on {psf.device}, img on {dev}')
        psf = require_cuda_stamps('psf', psf)
        if psf.shape[0] not in (1, B):
            raise ValueError(f'psf must have batch 1 or {B}, got {psf.shape[0]}')
        if B == 0:
            psf = None
    if noise is not None:
        if torch.is_tensor(noise) and noise.is_cuda and noise.device != dev:
            raise ValueError(f'noise is on {noise.device}, img on {dev}')
        noise = require_cuda_stamps('noise', noise, B)
    if noise_sigma is not None:
        if torch.is_tensor(noise_sigma):
            if not noise_sigma.is_cuda or noise_sigma.device != dev or noise_sigma.dtype != torch.float32:
                raise ValueError(f'noise_sigma must be a float or an fp32 tensor on {dev}, got {noise_sigma.dtype} on {noise_sigma.device}')
            if noise_sigma.dim() != 1 or noise_sigma.shape[0] not in (1, B):
                raise ValueError(f'noise_sigma must have shape [1] or [{B}], got {tuple(noise_sigma.shape)}')
            noise_sigma = noise_sigma.detach().contiguous()
        else:
            noise_sigma = torch.full((1,), float(noise_sigma), device=dev)
    ims = torch.empty(B, 5, 1, STAMP, STAMP, device=dev) if images else None
    shape = torch.empty(B, 5, 8, device=dev)
    info = torch.empty(B, 5, 2, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        if B and fix:
            check(lib.gd_metacal_fixnoise(_ptr(img), _ptr(psf), 0 if psf is None else psf.shape[0], B, float(delta), float(reconv_sigma),
                                          float(guess_sigma), _ptr(noise), _ptr(noise_sigma), 0 if noise_sigma is None else noise_sigma.shape[0],
                                          int(start), int(seed), _ptr(ims), _ptr(shape), _ptr(info), _stream(dev)))
        elif B:
            check(lib.gd_metacal(_ptr(img), _ptr(psf), 0 if psf is None else psf.shape[0], B, float(delta), float(reconv_sigma),
                                 float(guess_sigma), _ptr(ims), _ptr(shape), _ptr(info), _stream(dev)))
        e, status = shape[:, :, 6:8], info[:, :, 0]
        R = torch.stack([e[:, 1] - e[:, 2], e[:, 3] - e[:, 4]], 2) / (2 * float(delta))
        det = R[:, 0, 0] * R[:, 1, 1] - R[:, 0, 1] * R[:, 1, 0]
        e0 = e[:, 0]
        g = torch.stack([R[:, 1, 1] * e0[:, 0] - R[:, 0, 1] * e0[:, 1], R[:, 0, 0] * e0[:, 1] - R[:, 1, 0] * e0[:, 0]], 1) / det[:, None]
        g = torch.where((status == _lib.SHAPE_OK).all(1)[:, None], g, torch.full_like(g, float('nan')))
    out = dict(e=e, status=status, n_iter=info[:, :, 1], R=R, g=g)
    if images:
        out['images'] = ims
    return out


def synth_batch(device, start, count, seed, snr_mode, snr, psf_fwhm_err, psf_shear_err, obs=None, psf=None, alpha=None, gt=None):
    """gd_synth_batch on `device`'s current stream into preallocated contiguous fp32 CUDA tensors (any may be None, not all)."""
    with torch.cuda.device(device):
        check(lib.gd_synth_batch(int(start), int(count), int(seed), int(snr_mode), float(snr), float(psf_fwhm_err), float(psf_shear_err),
                                 _ptr(obs), _ptr(psf), _ptr(alpha), _ptr(gt), _stream(device)))


# ---------------------------------------------------------------------------------------------------
# XDenseUNet / Tikhonet (csrc/xdense.cu)
# ---------------------------------------------------------------------------------------------------
class _PackedX:
    def __init__(self, handle):
        self.handle = handle

    def __del__(self):
        try:
            if self.handle:
                lib.gd_free_xdense(self.handle)
        except Exception:
            pass


_XD_CHUNK = 2048
_xd_ws = {}


def _xd_workspace(device, chunk):
    key = (device.index, chunk)
    hit = _xd_ws.get(key)
    if hit is None:
        for k in [k for k in _xd_ws if k[0] == device.index]:
            del _xd_ws[k]
        nbytes = int(lib.gd_xdense_workspace_bytes(chunk))
        hit = (torch.empty(nbytes, dtype=torch.uint8, device=device), nbytes)
        _xd_ws[key] = hit
    return hit


class XDenseEngine:
    """Packed XDenseUNet weights of a module (XDenseUNet itself: prefix '', Tikhonet: prefix 'denoiser.')."""

    def __init__(self, module, prefix):
        self._module, self._prefix, self._packed = module, prefix, {}

    # ctypes handles cannot be copied or pickled: copies of the owning module start with an empty cache, bound to the copy
    def __deepcopy__(self, memo):
        return XDenseEngine(copy.deepcopy(self._module, memo), self._prefix)

    def __getstate__(self):
        return dict(_module=self._module, _prefix=self._prefix)

    def __setstate__(self, st):
        self.__init__(st['_module'], st['_prefix'])

    def invalidate(self):
        """Drop the packed weights (call after in-place updates through ``.data``, which do not bump ``_version``)."""
        self._packed.clear()

    def _weights(self, device):
        sd = self._module.state_dict(keep_vars=True)
        sig = tuple((k, v.data_ptr(), v._version) for k, v in sd.items())
        hit = self._packed.get(device.index)
        if hit is None or hit[0] != sig:
            names, arrays = [], []
            for k, v in self._module.state_dict().items():
                if torch.is_tensor(v) and v.dtype.is_floating_point and v.dim() <= 4:
                    names.append(k.encode()); arrays.append(v.detach().to('cpu', torch.float32).contiguous())
            descs = (_lib.GdTensorDesc * len(names))()
            for i, (n, a) in enumerate(zip(names, arrays)):
                descs[i].name, descs[i].data, descs[i].ndim = n, a.data_ptr(), a.dim()
                for d in range(a.dim()):
                    descs[i].shape[d] = a.shape[d]
            out = C.c_void_p()
            check(lib.gd_pack_xdense(descs, len(names), self._prefix.encode(), device.index, C.byref(out)))
            hit = (sig, _PackedX(out))
            self._packed[device.index] = hit
        return hit[1]

    @staticmethod
    def _chunk(batch):
        c = 1
        while c < min(batch, _XD_CHUNK):
            c *= 2
        return c

    def denoise(self, x):
        x = require_cuda_stamps('x', x)
        dev, B = x.device, x.shape[0]
        with torch.cuda.device(dev):
            w = self._weights(dev)
            chunk = self._chunk(B)
            ws, nbytes = _xd_workspace(dev, chunk)
            out = torch.empty_like(x)
            check(lib.gd_xdense_forward(w.handle, _ptr(x), _ptr(out), B, _ptr(ws), nbytes, chunk, _stream(dev)))
        return out

    def tikhonet(self, kind, lam, y, psf, alpha):
        y = require_cuda_stamps('y', y)
        dev, B = y.device, y.shape[0]
        psf = require_cuda_stamps('psf', psf, B)
        a = _alpha_vector(alpha, B, dev)
        with torch.cuda.device(dev):
            w = self._weights(dev)
            chunk = self._chunk(B)
            ws, nbytes = _xd_workspace(dev, chunk)
            out = torch.empty_like(y)
            check(lib.gd_tikhonet_forward(w.handle, kind, float(lam), _ptr(y), _ptr(psf), _ptr(a), _ptr(out), B, _ptr(ws), nbytes, chunk,
                                          _stream(dev)))
        return out
