"""Python wrappers (pointer plumbing only) around the C-ABI kernels."""
import ctypes
import math
import weakref

import torch

from .. import _lib
from .._lib import ConvGemmDesc, check, lib, ptr, require_cuda, stream_ptr


# kernel launches issued through this module (bench.py reports it as `gpu_launches`)
LAUNCHES = [0]


def _launch_conv_gemm(d):
    """single choke point of the tcgen05 kernel (bench.py wraps it with CUDA events for the roofline)"""
    if _CHAIN_MODE[0] == "record":
        _CHAIN_REC[0].append(_copy_desc(d))
        return
    if _CHAIN_MODE[0] == "skip":
        return

    def run():
        check(lib.mega_conv_gemm(ctypes.byref(d), stream_ptr()), "mega_conv_gemm")
    _run_timed(run, _desc_flops(d), _desc_info(d))
    LAUNCHES[0] += 1


# bench.py installs a hook here to bracket every tensor-core kernel launch with CUDA events: hook(run, flops, info)
TIMING_HOOK = [None]


def _run_timed(run, flops, info):
    h = TIMING_HOOK[0]
    if h is None:
        run()
    else:
        h(run, flops, info)


def _desc_flops(d):
    return 2.0 * d.n_img * d.out_h * d.out_w * d.batch * d.cout * d.k_per_tap * d.taps_r * d.taps_s


def _desc_info(d):
    return {"m": d.n_img * d.out_h * d.out_w, "batch": d.batch, "cout": d.cout, "k": d.k_per_tap,
            "taps": d.taps_r * d.taps_s, "bn": d.block_n, "sk": d.stream_k, "res": bool(d.residual), "out16": d.out_f16}


# ---------------------------------------------------------------------------------------------------------------------
# Layer chains: a fixed sequence of dependent conv_gemm calls executed by ONE persistent kernel (csrc/conv_chain.cu).
#     with ops.chain(cache, key) as ch:      # first time: the conv_gemm calls inside are RECORDED (not launched) and
#         ... ops.conv_gemm(...) ...         # compiled into a device-side layer table; afterwards they are skipped
#     # on exit the whole chain is launched (one kernel)
# Only conv_gemm calls may appear inside (anything else would run before the chain); all tensors must be persistent.
_CHAIN_MODE = [None]
_CHAIN_REC = [None]
CHAINS_ENABLED = [True]
MAX_BN = [256]          # widest N tile conv_gemm may pick (128 while recording a chain)


def _copy_desc(d):
    c = ConvGemmDesc()
    ctypes.memmove(ctypes.byref(c), ctypes.byref(d), ctypes.sizeof(ConvGemmDesc))
    return c


class ConvChain(object):
    def __init__(self, descs, device, max_ctas=0, depth=1):
        n = len(descs)
        self.n, self.depth = n, depth
        arr = (ConvGemmDesc * n)(*descs)
        nbytes = int(lib.mega_conv_chain_plan_bytes(n))
        host = torch.zeros(nbytes + 128, dtype=torch.uint8)
        off = (-host.data_ptr()) % 128
        grid = ctypes.c_int(0)
        check(lib.mega_conv_chain_encode2(arr, n, ctypes.c_void_p(host.data_ptr() + off), nbytes, ctypes.byref(grid), depth),
              "mega_conv_chain_encode2")
        if max_ctas > 0 and grid.value > max_ctas:
            raise _lib.MegaError("conv chain: a layer wants %d CTAs, more than max_ctas=%d (pass max_ctas to every "
                                 "conv_gemm of the chain)" % (grid.value, max_ctas))
        self.grid = grid.value
        dev_buf = torch.zeros(nbytes + 128, dtype=torch.uint8, device=device)
        doff = (-dev_buf.data_ptr()) % 128
        self.plan = dev_buf[doff:doff + nbytes]
        self.plan.copy_(host[off:off + nbytes])
        self._keep = dev_buf
        self.sync = torch.zeros(4, dtype=torch.int32, device=device)
        self.flops = sum(_desc_flops(d) for d in descs)
        self.info = {"chain_layers": n, "grid": self.grid, "depth": depth, "layers": [_desc_info(d) for d in descs]}
        torch.cuda.current_stream(device).synchronize()

    def launch(self):
        def run():
            check(lib.mega_conv_chain_launch2(ptr(self.plan), self.n, self.grid, ptr(self.sync), stream_ptr(),
                                              1 if PDL[0] else 0, self.depth), "mega_conv_chain_launch2")
        _run_timed(run, self.flops, self.info)
        LAUNCHES[0] += 1


class chain(object):
    """context manager: record-once / replay a chain of conv_gemm calls (see above). `cache` is a dict owned by the
    caller, `key` identifies the call sequence (shapes); disabled (plain per-layer launches) when the tensors are not
    fp16, when chains are switched off, or while autotuning a shape for the first time.

    interleave=True: the body issues the SAME layer sequence twice, on two independent halves of its batch (disjoint
    buffers), calling `next_lane()` between them; the two recordings are interleaved A0 B0 A1 B1 ... and run with barrier
    depth 2 (csrc/conv_chain.cu): a CTA streams lane B's layer while lane A's layer drains its epilogue / stores / grid
    barrier. Results are those of the two sequences run one after the other."""

    def __init__(self, cache, key, device, enabled=True, max_ctas=0, interleave=False, depth=1):
        if SM_LIMIT[0] > 0 or WS_LANE[0] != 0:   # a chain recorded under an SM limit / on another workspace lane is a different chain
            key = tuple(key) + ("sm", SM_LIMIT[0], WS_LANE[0])
        if SM_LIMIT[0] > 0:
            max_ctas = min(max_ctas, SM_LIMIT[0]) if max_ctas > 0 else SM_LIMIT[0]
        self.cache, self.key, self.device, self.max_ctas = cache, key, device, max_ctas
        self.enabled = enabled and CHAINS_ENABLED[0] and _CHAIN_MODE[0] is None
        self.interleave = interleave and self.enabled
        self.depth = depth          # 2: the caller guarantees that no layer reads what the layer directly before it wrote
        self.split = None

    def next_lane(self):
        if self.enabled and _CHAIN_MODE[0] == "record":
            assert self.interleave and self.split is None
            self.split = len(_CHAIN_REC[0])

    def __enter__(self):
        if not self.enabled:
            return self
        self.saved_bn = MAX_BN[0]
        MAX_BN[0] = 128
        if self.key in self.cache:
            _CHAIN_MODE[0] = "skip"
        else:
            _CHAIN_MODE[0] = "record"
            _CHAIN_REC[0] = []
        return self

    def __exit__(self, et, ev, tb):
        if not self.enabled:
            return False
        mode = _CHAIN_MODE[0]
        _CHAIN_MODE[0] = None
        MAX_BN[0] = self.saved_bn
        if et is not None:
            _CHAIN_REC[0] = None
            return False
        if mode == "record":
            descs = _CHAIN_REC[0]
            _CHAIN_REC[0] = None
            depth = self.depth
            if self.interleave:
                assert self.split is not None and 2 * self.split == len(descs), \
                    "interleaved chain: the two lanes must record the same number of layers (%s / %d)" % (self.split, len(descs))
                descs = [d for pair in zip(descs[:self.split], descs[self.split:]) for d in pair]
                depth = 2
            self.cache[self.key] = ConvChain(descs, self.device, self.max_ctas, depth)
        self.cache[self.key].launch()
        return False


# interleaved (depth-2) chains for the per-frame branch when the image batch splits into two halves
import os as _os
# Measured on a B200 (backbone chain, fp16, 600x1000; ms for 2 / 4 / 8 images): one chain 1.61 / 2.49 / 4.06, two
# interleaved lanes 1.87 / 2.33 / 3.75 -- lanes of a single image leave too few tiles per layer, so the engine interleaves
# from 4 images on (DUAL_MIN_IMAGES); MEGA_B200_DUAL_CHAIN=0 switches it off
DUAL_CHAIN = [_os.environ.get("MEGA_B200_DUAL_CHAIN", "1") != "0"]
DUAL_MIN_IMAGES = 4

# programmatic dependent launch of the GEMM kernels (prologue overlapped with the previous kernel's tail)
PDL = [True]

_gemm_ws = {}
WS_LANE = [0]   # launches that may overlap on different streams must use different lanes
SM_LIMIT = [0]  # > 0: persistent kernels (conv_gemm / chains) launched inside `with sm_limit(n)` take at most n CTAs, so that two
                # launch sequences on two streams share the GPU by SMs (MegaEngine.stepn_pipelined)


class sm_limit(object):
    """context manager: cap the persistent grids at `n` CTAs and select stream-K workspace lane `lane`"""

    def __init__(self, n, lane=None):
        self.n, self.lane = int(n), lane

    def __enter__(self):
        self.saved = (SM_LIMIT[0], WS_LANE[0])
        SM_LIMIT[0] = self.n
        if self.lane is not None:
            WS_LANE[0] = self.lane
        return self

    def __exit__(self, *a):
        SM_LIMIT[0], WS_LANE[0] = self.saved
        return False


def gemm_workspace(device):
    """zero-initialised stream-K workspace, one per (device, lane): kernels on one stream are
    ordered; kernels issued on concurrent streams must select distinct lanes (WS_LANE) so they do
    not share tile counters"""
    key = (device, WS_LANE[0])
    ws = _gemm_ws.get(key)
    if ws is None:
        ws = torch.zeros(int(lib.mega_conv_gemm_workspace_bytes()), dtype=torch.uint8, device=device)
        _gemm_ws[key] = ws
    return ws


def pick_tile(h, w):
    """128-pixel output tile (tile_h, tile_w) wasting the fewest pixels for an h x w map."""
    best = None
    for tw in (128, 64, 32, 16, 8, 4, 2, 1):
        th = 128 // tw
        tiles = -(-h // th) * -(-w // tw)
        key = (tiles, -tw)
        if best is None or key < best[0]:
            best = (key, th, tw)
    return best[1], best[2]


# ---- arithmetic of the dense contractions over fp32 tensors: 0 = TF32 operands, 1 = "3xTF32" split (near-fp32,
#      strict parity). fp16 tensors always run as precision 2 (fp16 operands, fp32 accumulate): the engine selects
#      that mode by allocating its activations / weights in fp16 (EngineConfig.precision == "f16").
PRECISION = [0]
PRECISION_NAMES = {"tf32": 0, "fp32x3": 1, "f16": 0}


class precision(object):
    """context manager selecting the contraction arithmetic of every conv_gemm launched inside it"""

    def __init__(self, name):
        self.value = PRECISION_NAMES[name] if isinstance(name, str) else int(name)

    def __enter__(self):
        self.saved = PRECISION[0]
        PRECISION[0] = self.value

    def __exit__(self, *a):
        PRECISION[0] = self.saved
        return False


# ---- strict mode (3xTF32): weights split ONCE. presplit(w) returns a tensor equal to w whose storage continues with the
#      low parts lo = w - trunc_tf32(w) (as `taps` more [rows, K] slices); conv_gemm recognises it by its address and lets
#      the kernel fetch lo by TMA instead of splitting the staged weight tile on every k-block of every launch.
_PRESPLIT = {}


def presplit(w):
    """w: contiguous fp32 CUDA weight [rows, K] or [taps, rows, K] -> the same values as a view of a [2 * taps, rows, K]
    tensor whose second half holds the low parts of the 3xTF32 split"""
    assert w.is_cuda and w.dtype == torch.float32 and w.is_contiguous() and w.dim() in (2, 3)
    w3 = w if w.dim() == 3 else w.view(1, *w.shape)
    taps = w3.shape[0]
    combo = torch.empty(2 * taps, w3.shape[1], w3.shape[2], device=w.device, dtype=torch.float32)
    combo[:taps].copy_(w3)
    hi = (w3.view(torch.int32) & -8192).view(torch.float32)            # truncation to TF32: clear the low 13 mantissa bits
    combo[taps:].copy_(w3 - hi)
    out = combo[:taps] if w.dim() == 3 else combo[0]
    # keyed by address, valid while the returned tensor lives (a freed weight's address may be handed to an activation)
    _PRESPLIT[out.data_ptr()] = (weakref.ref(out), taps, tuple(w3.shape[1:]))
    return out


# ---- strict mode, "3xFP16" (precision 3): the SPLIT-FP16 storage format (include/mega_b200.h). A split-fp16 tensor is an
#      fp32-typed torch tensor (same shape / strides / bytes) whose every aligned group of 32 values holds 32 hi halves then
#      32 lo halves; which tensors are in that format is tracked by STORAGE (every view of a buffer shares it). conv_gemm runs
#      precision 3 when its weights were packed by pack_weights_split16 (A must then be a split-fp16 tensor) and writes
#      split-fp16 exactly when `out` is marked; the residual may be either.
SPLIT16 = [_os.environ.get("MEGA_B200_SPLIT16", "1") != "0"]     # strict engines use the format (0: 3xTF32 everywhere)
SPLIT16_ATT = [_os.environ.get("MEGA_B200_SPLIT16_ATT", "1") != "0"]   # ... also for the relation stages' feature rows
_SPLIT16_BUFS = {}
_SPLIT16_W = {}


def mark_split16(t):
    """declare the storage of `t` split-fp16 (the caller fills it through conv_gemm / pack_split16)"""
    assert t.dtype == torch.float32
    st = t.untyped_storage()
    _SPLIT16_BUFS[st.data_ptr()] = weakref.ref(st)
    return t


def unmark_split16(t):
    _SPLIT16_BUFS.pop(t.untyped_storage().data_ptr(), None)
    return t


def is_split16(t):
    if t is None or t.dtype != torch.float32:
        return False
    st = t.untyped_storage()
    r = _SPLIT16_BUFS.get(st.data_ptr())
    if r is None:
        return False
    if r() is None:          # a freed buffer's address handed to a new tensor
        del _SPLIT16_BUFS[st.data_ptr()]
        return False
    return True


def pack_split16(x, out=None):
    """fp32 values -> split-fp16; contiguous, numel % 32 == 0. out=None converts IN PLACE (and marks x)"""
    require_cuda(x, out)
    dst = x if out is None else out
    assert x.dtype == torch.float32 and x.is_contiguous() and dst.is_contiguous() and dst.numel() == x.numel()
    assert not is_split16(x) or out is not None, "already split-fp16"
    check(lib.mega_split16_pack(ptr(x), ptr(dst), x.numel(), stream_ptr()), "mega_split16_pack")
    return mark_split16(dst)


def unpack_split16(x, out):
    """split-fp16 -> fp32 values in `out` (contiguous, distinct storage)"""
    require_cuda(x, out)
    assert x.is_contiguous() and out.is_contiguous() and out.numel() == x.numel() and out.dtype == torch.float32
    check(lib.mega_split16_unpack(ptr(x), ptr(out), x.numel(), stream_ptr()), "mega_split16_unpack")
    return out


def split16_encode(x):
    """torch restatement of the format (any device): fp32 [..., K] (K % 32 == 0) -> fp32-typed tensor of the same shape
    holding [32 hi halves | 32 lo halves] per group of 32 values"""
    assert x.dtype == torch.float32 and x.shape[-1] % 32 == 0
    xc = x.contiguous()
    hi = xc.clamp(-65504.0, 65504.0).half()
    lo = (xc - hi.float()).clamp(-65504.0, 65504.0).half()
    g = xc.shape[:-1] + (xc.shape[-1] // 32, 1, 32)
    both = torch.cat([hi.view(g), lo.view(g)], dim=-2)                  # [..., K/32, 2, 32] halves
    return both.reshape(xc.shape[:-1] + (2 * xc.shape[-1],)).view(torch.float32)


def split16_decode(p):
    """inverse of split16_encode (fp32 sums hi + lo)"""
    h = p.contiguous().view(torch.float16)
    g = h.view(p.shape[:-1] + (p.shape[-1] // 32, 2, 32)).float()
    return (g[..., 0, :] + g[..., 1, :]).reshape(p.shape)


def pack_weights_split16(w, scale=None):
    """w: fp32 weight [rows, K] or [taps, rows, K] (K % 32 == 0) -> split-fp16 tensor of the same shape holding w * 2^e, e
    chosen so that max |w| 2^e lies in [2^13, 2^14) (the low halves of all weights down to 2^-17 of the largest then stay
    normal fp16 numbers); conv_gemm multiplies the accumulator by 2^-e (exact). scale [rows]: a per-output-channel factor
    (FrozenBatchNorm) folded into the weights first -- the precision-3 kernel adds a bias only."""
    assert w.dtype == torch.float32 and w.dim() in (2, 3) and w.shape[-1] % 32 == 0
    if scale is not None:
        w = w * scale.to(w.device).float().view(-1, 1)
    m = float(w.abs().max())
    e = 0 if m == 0.0 else 13 - int(math.floor(math.log2(m)))
    e = max(-24, min(e, 40))
    out = split16_encode(w * (2.0 ** e))
    _SPLIT16_W[out.data_ptr()] = (weakref.ref(out), 2.0 ** -e)
    return out


def _split16_weight(w):
    r = _SPLIT16_W.get(w.data_ptr())
    if r is None:
        return None
    if r[0]() is None:
        del _SPLIT16_W[w.data_ptr()]
        return None
    return r[1]


def _split16_fmt(t):
    """None: plain tensor; else the power of two its split-fp16 values must be multiplied by (1.0 for activations, 2^-e for
    tensors made by pack_weights_split16 -- either may serve as the A or the B operand)"""
    if t is None or t.dtype != torch.float32:
        return None
    s = _split16_weight(t)
    if s is not None:
        return s
    return 1.0 if is_split16(t) else None


# ---- per-shape kernel configuration (block_n, stream_k, max_ctas), filled by autotune()
TUNED = {}
AUTOTUNE = [False]
BLOCK_NS = (32, 64, 96, 128, 160, 192, 256)


def save_tuned(path):
    """persist the autotuned (block_n, stream_k) table (keyed by problem signature)"""
    import json
    with open(path, "w") as fh:
        json.dump({"device": torch.cuda.get_device_name(0), "entries": [[list(k), list(v)] for k, v in TUNED.items()]}, fh)


def load_tuned(path):
    import json
    import os
    if not os.path.exists(path):
        return 0
    with open(path) as fh:
        data = json.load(fh)
    if torch.cuda.is_available() and data.get("device") != torch.cuda.get_device_name(0):
        return 0
    for k, v in data["entries"]:
        if len(k) == 22:      # tables written before the fp16 modes existed: out_f16 = 0
            k = list(k) + [0]
        TUNED.setdefault(tuple(bool(x) if isinstance(x, bool) else x for x in k), tuple(v))
    return len(data["entries"])


def _shape_key(d):
    return (d.a_n, d.a_h, d.a_w, d.a_c, d.a_stride_w, d.b_n, d.b_k, d.taps_r, d.taps_s, d.dil, d.k_per_tap, d.n_img,
            d.out_h, d.out_w, d.cout, d.tile_h, d.tile_w, d.batch, bool(d.residual), d.out_ld, d.out_c_off,
            d.precision, d.out_f16) + ((d.stride_h, d.stride_w) if (d.stride_h, d.stride_w) != (1, 1) else ())


def _candidates(cout, prec=0, out_f16=0):
    cands = []
    for bn in ((64, 128) if prec in (1, 3) else BLOCK_NS):
        if out_f16 and bn % 64:
            continue
        if bn > MAX_BN[0]:
            continue
        if bn >= 2 * cout and bn > (64 if out_f16 else 32):
            continue
        for sk in (0, 1):
            cands.append((bn, sk))
    return cands


def _autotune(d):
    """time every (block_n, stream_k) candidate for this exact problem on the device (CUDA events,
    3 warm + 5 timed launches each) and remember the fastest; outputs are overwritten identically"""
    best = None
    for bn, sk in _candidates(d.cout, d.precision, d.out_f16):
        d.block_n, d.stream_k = bn, sk
        try:
            for _ in range(2):
                check(lib.mega_conv_gemm(ctypes.byref(d), stream_ptr()), "mega_conv_gemm")
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(8):
                check(lib.mega_conv_gemm(ctypes.byref(d), stream_ptr()), "mega_conv_gemm")
            e1.record()
            e1.synchronize()
            t = e0.elapsed_time(e1) / 8
        except _lib.MegaError:
            continue
        if best is None or t < best[0]:
            best = (t, bn, sk)
    return best


def _autotune_chain(d):
    """same, for a layer that is being recorded into a chain: every candidate is timed as a ONE-layer chain (the
    persistent chain kernel is the code that will run it; launch overhead is the same constant for all candidates)"""
    best = None
    dev = torch.device("cuda", torch.cuda.current_device())
    for bn, sk in _candidates(d.cout, d.precision, d.out_f16):
        c = _copy_desc(d)
        c.block_n, c.stream_k = bn, sk
        try:
            ch = ConvChain([c], dev, max_ctas=d.max_ctas)
            hook, TIMING_HOOK[0] = TIMING_HOOK[0], None
            try:
                for _ in range(2):
                    ch.launch()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(8):
                    ch.launch()
                e1.record()
                e1.synchronize()
            finally:
                TIMING_HOOK[0] = hook
            LAUNCHES[0] -= 10
            t = e0.elapsed_time(e1) / 8
        except _lib.MegaError:
            continue
        if best is None or t < best[0]:
            best = (t, bn, sk)
    return best


def pick_config(cout, m_tiles, batch, kb_per_tile, out_f16=False):
    """(block_n, stream_k) when no autotuned entry exists. Deep reductions balance best at k-block
    granularity (stream-K, widest tile); shallow ones run whole tiles, with the tile width chosen to
    minimise waves x bytes staged per k-block on 148 SMs."""
    if kb_per_tile >= 48:
        for bn in (32, 64, 128):
            if cout <= bn and not (out_f16 and bn % 64):
                return bn, 1
        return min(256, MAX_BN[0]), 1
    best = None
    for bn in BLOCK_NS:
        if out_f16 and bn % 64:
            continue
        if bn > MAX_BN[0]:
            continue
        if bn >= 2 * cout and bn > (64 if out_f16 else 32):
            continue
        tiles = m_tiles * (-(-cout // bn)) * batch
        cost = (-(-tiles // 148)) * (128 + bn)
        if best is None or cost < best[0] or (cost == best[0] and bn > best[1]):
            best = (cost, bn)
    return best[1], 0


def pick_block_n(cout, m_tiles=0, batch=1):
    return pick_config(cout, max(m_tiles, 1), batch, 1)[0]


def conv_gemm(a, w, out, *, taps=(1, 1), dil=1, pad=0, scale=None, bias=None, residual=None,
              relu=False, tile=None, block_n=None, cout=None, k=None, batch=1, a_c_off=0,
              a_n_off=0, b_k_off=0, b_n_off=0, out_c_off=0, out_n_off=0, res_c_off=0, res_n_off=0, bias_z_off=0,
              max_ctas=0, stream_k=None, out_hw=None, n_img=None, stride=(1, 1), pad_w=None):
    """out[n,h,w,:] = act(scale * conv(a, w) + bias + residual)   (tcgen05 tensor cores, fp32 accumulate)

    a   : [N,H,W,C] fp32 or fp16 view (innermost stride 1; other strides multiples of 16 bytes)
    w   : [taps, rows, K] same dtype as a (K contiguous)
    out : [N,Ho,Wo,>=cout] fp32 view, or fp16 when a is fp16 (innermost stride 1); residual: same dtype as out
    fp32 operands run as TF32 (or the 3xTF32 split under ops.precision("fp32x3")), fp16 operands as kind::f16.
    relu: False / True / "leaky" (LeakyReLU 0.1). stride = (stride_h, stride_w) of the convolution; pad_w: left padding
    when it differs from `pad` (rows). `out` (and `residual`) may be strided views in w / h / n (e.g. every other
    pixel of a larger map).
    """
    require_cuda(a, w, out, scale, bias, residual)
    f16 = a.dtype == torch.float16
    assert a.dtype == w.dtype and a.dtype in (torch.float32, torch.float16), (a.dtype, w.dtype)
    assert out.dtype == torch.float32 or (f16 and out.dtype == torch.float16), (a.dtype, out.dtype)
    assert residual is None or residual.dtype == out.dtype
    out_f16 = out.dtype == torch.float16
    assert a.dim() == 4 and w.dim() == 3 and out.dim() == 4
    assert a.stride(3) == 1 and w.stride(2) == 1 and out.stride(3) == 1
    n, h, wd, c = a.shape
    t, rows, kk = w.shape
    assert t == taps[0] * taps[1]
    on, oh, ow, oc = out.shape
    if out_hw is not None:
        oh, ow = out_hw
    d = ConvGemmDesc()
    d.a = ptr(a)
    d.a_n, d.a_h, d.a_w, d.a_c = n, h, wd, c
    d.a_stride_w, d.a_stride_h, d.a_stride_n = a.stride(2), a.stride(1), a.stride(0)
    d.b = ptr(w)
    d.b_n, d.b_k = rows, kk
    d.b_stride_n, d.b_stride_tap = w.stride(1), w.stride(0)
    d.taps_r, d.taps_s, d.dil, d.pad = taps[0], taps[1], dil, pad
    d.k_per_tap = k if k is not None else kk
    d.out = ptr(out)
    d.out_ld = out.stride(2)
    d.n_img, d.out_h, d.out_w = (on if n_img is None else n_img), oh, ow
    d.cout = cout if cout is not None else rows
    d.scale, d.bias, d.residual = ptr(scale), ptr(bias), ptr(residual)
    d.res_ld = residual.stride(-2) if residual is not None else 0
    if oh > 1:
        d.out_stride_h = out.stride(1)
    if d.n_img > 1 or batch > 1:
        d.out_stride_n = out.stride(0)
    if residual is not None and residual.dim() == 4:
        if oh > 1:
            d.res_stride_h = residual.stride(1)
        if d.n_img > 1 or batch > 1:
            d.res_stride_n = residual.stride(0)
    d.relu = 2 if relu == "leaky" else (1 if relu else 0)
    d.stride_h, d.stride_w = stride
    if pad_w is not None:
        d.pad_w_set, d.pad_w = 1, pad_w
    th, tw = tile if tile is not None else pick_tile(oh, ow)
    d.tile_h, d.tile_w = th, tw
    m_tiles = d.n_img * (-(-oh // th)) * (-(-ow // tw))
    d.batch = batch
    kb_per_tile = taps[0] * taps[1] * (-(-d.k_per_tap // (64 if f16 else 32)))
    d.precision = 2 if f16 else PRECISION[0]
    d.out_f16 = 1 if out_f16 else 0
    fa, fb = _split16_fmt(a), _split16_fmt(w)
    if fa is not None or fb is not None:
        assert fa is not None and fb is not None, \
            "conv_gemm: both operands must be split-fp16 (ops.pack_split16 / pack_weights_split16) or neither (A %s, B %s)" % (
                "split" if fa is not None else "plain", "split" if fb is not None else "plain")
        assert scale is None, "conv_gemm: split-fp16 contractions take no scale (fold it: pack_weights_split16(w, scale))"
        d.precision = 3
        d.out_f16 = 1 if is_split16(out) else 0
        d.res_split = 1 if is_split16(residual) else 0
        d.acc_scale = fa * fb
    else:
        assert not (is_split16(out) or is_split16(residual)), \
            "conv_gemm: split-fp16 output / residual need split-fp16 operands"
    d.pdl = 1 if PDL[0] else 0
    auto_bn, auto_sk = pick_config(d.cout, m_tiles, batch, kb_per_tile, out_f16)
    if d.precision in (1, 3):
        auto_bn = 64 if d.cout <= 64 else 128
        if block_n not in (None, 64, 128):
            block_n = auto_bn
    d.block_n = block_n if block_n is not None else auto_bn
    d.stream_k = auto_sk if stream_k is None else int(stream_k)
    d.a_c_off, d.a_n_off, d.b_k_off, d.b_n_off = a_c_off, a_n_off, b_k_off, b_n_off
    d.out_c_off, d.out_n_off, d.res_c_off, d.res_n_off = out_c_off, out_n_off, res_c_off, res_n_off
    d.bias_z_off = bias_z_off
    d.max_ctas = max_ctas
    if SM_LIMIT[0] > 0:
        d.max_ctas = min(max_ctas, SM_LIMIT[0]) if max_ctas > 0 else SM_LIMIT[0]
    if d.precision == 1 and batch == 1:
        ps = _PRESPLIT.get(w.data_ptr())
        if ps is not None and ps[0]() is None:
            del _PRESPLIT[w.data_ptr()]
            ps = None
        if ps is not None and ps[1] == t and ps[2] == (rows, kk) and w.stride(1) == kk:
            d.b_lo_tap_off = t
            d.b_stride_tap = rows * kk
    ws = gemm_workspace(a.device)
    d.workspace = ptr(ws)
    d.workspace_bytes = ws.numel()
    if block_n is None and stream_k is None:
        key = _shape_key(d) + ((MAX_BN[0],) if MAX_BN[0] != 256 else ())
        cfg = TUNED.get(key)
        aliased = residual is not None and residual.data_ptr() == out.data_ptr()   # in-place: not idempotent
        if (cfg is None and AUTOTUNE[0] and not aliased and _CHAIN_MODE[0] != "skip"
                and not torch.cuda.is_current_stream_capturing()):
            best = _autotune_chain(d) if _CHAIN_MODE[0] == "record" else _autotune(d)
            if best is not None:
                cfg = TUNED[key] = (best[1], best[2], best[0])
        if cfg is not None:
            d.block_n, d.stream_k = cfg[0], cfg[1]
    _launch_conv_gemm(d)
    return out


def linear(x, w, out, *, bias=None, relu=False, residual=None, block_n=None, max_ctas=0, stream_k=None):
    """out[m,:] = act(x[m,:] @ w.T + bias + residual[m,:]); x [M,K], w [N,K], out [M,N]."""
    m, kdim = x.shape
    nrows = w.shape[0]
    a4 = x.as_strided((1, 1, m, kdim), (x.stride(0) * m, x.stride(0) * m, x.stride(0), 1))
    o4 = out.as_strided((1, 1, m, out.shape[1]), (out.stride(0) * m, out.stride(0) * m, out.stride(0), 1))
    r4 = None
    if residual is not None:
        r4 = residual.as_strided((1, 1, m, residual.shape[1]),
                                 (residual.stride(0) * m, residual.stride(0) * m, residual.stride(0), 1))
    w3 = w.as_strided((1, nrows, kdim), (w.stride(0) * nrows, w.stride(0), 1))
    return conv_gemm(a4, w3, o4, bias=bias, relu=relu, residual=r4, tile=(1, 128), cout=nrows, block_n=block_n,
                     max_ctas=max_ctas, stream_k=stream_k)


# --------------------------------------------------------------------------- non-GEMM kernels
_ws_cache = {}


def _workspace(key, nbytes, device):
    """persistent byte workspace per (kind, device): kernels never allocate device memory."""
    ws = _ws_cache.get((key, device))
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        _ws_cache[(key, device)] = ws
    return ws


def nms_device(boxes, scores, thresh, keep=None, count=None):
    """-> (keep int64 [n] buffer, count int32 [1]) on the device; no synchronisation."""
    require_cuda(boxes, scores)
    n = boxes.shape[0]
    boxes = boxes.contiguous().float()
    scores = scores.contiguous().float()
    if keep is None:
        keep = torch.empty(max(n, 1), dtype=torch.int64, device=boxes.device)
    if count is None:
        count = torch.zeros(1, dtype=torch.int32, device=boxes.device)
    nbytes = lib.mega_nms_workspace_bytes(n)
    if nbytes < 0:
        raise _lib.MegaError("nms: n=%d exceeds the single-pass capacity (8192 boxes)" % n)
    ws = _workspace("nms", max(nbytes, 256), boxes.device)
    check(lib.mega_nms(ptr(boxes), ptr(scores), n, float(thresh), ptr(ws), ws.numel(), ptr(keep), ptr(count),
                       stream_ptr()), "mega_nms")
    LAUNCHES[0] += 4
    return keep, count


def rpn_select(head, n_img, h, w, base_anchors, im_w, im_h, pre_nms, post_nms, nms_thresh, min_size=0.0,
               stride=16, out=None, want_anchor=False):
    """head: [n_img, h, w, ld] fp32 (ld >= 5A). Returns (boxes [n_img,post,4], scores, anchor_idx|None, count)."""
    require_cuda(head, base_anchors)
    a = base_anchors.shape[0]
    ld = head.shape[-1]
    dev = head.device
    if out is None:
        boxes = torch.empty(n_img, post_nms, 4, device=dev)
        scores = torch.empty(n_img, post_nms, device=dev)
        count = torch.empty(n_img, dtype=torch.int32, device=dev)
        anchor = torch.empty(n_img, post_nms, dtype=torch.int32, device=dev) if want_anchor else None
    else:
        boxes, scores, anchor, count = out
    nbytes = lib.mega_rpn_select_workspace_bytes(n_img, h, w, a, pre_nms)
    if nbytes < 0:
        raise _lib.MegaError("rpn_select: pre_nms_top_n=%d exceeds 8192" % pre_nms)
    ws = _workspace("rpn%d" % n_img, nbytes, dev)
    check(lib.mega_rpn_select(ptr(head), head.stride(0), ld, n_img, h, w, a, stride, ptr(base_anchors), float(im_w),
                              float(im_h), pre_nms, post_nms, float(nms_thresh), float(min_size), ptr(ws), ws.numel(),
                              ptr(boxes), ptr(scores), ptr(anchor), ptr(count), stream_ptr()), "mega_rpn_select")
    LAUNCHES[0] += 4
    return boxes, scores, anchor, count


def roi_align_nchw(inp, rois, scale, ph, pw, sampling_ratio, out=None):
    require_cuda(inp, rois)
    inp = inp.contiguous().float()
    rois = rois.contiguous().float()
    n, c, h, w = inp.shape
    k = rois.shape[0]
    if out is None:
        out = torch.empty(k, c, ph, pw, device=inp.device)
    check(lib.mega_roi_align_forward_nchw(ptr(inp), n, c, h, w, ptr(rois), k, float(scale), ph, pw, sampling_ratio,
                                          ptr(out), stream_ptr()), "mega_roi_align_forward_nchw")
    LAUNCHES[0] += 1
    return out


def roi_align_nhwc(feat, boxes, roi_batch, scale, ph, pw, sampling_ratio, out):
    """feat [N,H,W,C] fp32 or fp16; boxes [K,4]; roi_batch int32 [K] or None; out [K, ph*pw*C] (dtype of feat)."""
    require_cuda(feat, boxes, roi_batch, out)
    n, h, w, c = feat.shape
    k = boxes.shape[0]
    assert out.dtype == feat.dtype
    fn = lib.mega_roi_align_forward_nhwc_f16 if feat.dtype == torch.float16 else lib.mega_roi_align_forward_nhwc
    if is_split16(feat):
        # split-fp16 map -> split-fp16 rows (marks `out`); maps beyond the separable kernel's 64 x 64 cells go through fp32
        if h <= 64 and w <= 64 and c % 128 == 0 and ph <= 7 and pw <= 7:
            fn = lib.mega_roi_align_forward_nhwc_split16
            mark_split16(out)
        else:
            plain = unpack_split16(feat.contiguous(), torch.empty_like(feat))
            unmark_split16(out)
            roi_align_nhwc(plain, boxes, roi_batch, scale, ph, pw, sampling_ratio, out)
            return pack_split16(out)
    else:
        unmark_split16(out)
    check(fn(ptr(feat), c, h, w, feat.stride(0), ptr(boxes), boxes.stride(0), 0,
                                          ptr(roi_batch), k, float(scale), ph, pw, sampling_ratio, ptr(out),
                                          out.stride(0), stream_ptr()), "mega_roi_align_forward_nhwc")
    LAUNCHES[0] += 1
    return out


def stem_im2col(img, out, kpad=160):
    """img fp32 NCHW -> im2col rows, fp32 or fp16 by out.dtype"""
    require_cuda(img, out)
    n, c, h, w = img.shape
    assert c == 3 and img.is_contiguous() and img.dtype == torch.float32
    fn = lib.mega_stem_im2col_f16 if out.dtype == torch.float16 else lib.mega_stem_im2col
    check(fn(ptr(img), n, h, w, kpad, ptr(out), stream_ptr()), "mega_stem_im2col")
    LAUNCHES[0] += 1
    return out


def stem_prep(img, out):
    """img [N,3,H,W] fp32 -> out [N, H+6, WP, 8] (zero border of 3 pixels, 3 real channels)"""
    require_cuda(img, out)
    n, c, h, w = img.shape
    assert c == 3 and img.is_contiguous() and img.dtype == torch.float32 and out.shape[1] == h + 6 and out.shape[3] == 8
    check(lib.mega_stem_prep(ptr(img), n, h, w, out.shape[2], ptr(out), 1 if out.dtype == torch.float16 else 0,
                             stream_ptr()), "mega_stem_prep")
    LAUNCHES[0] += 1
    return out


def maxpool3x3s2(x, out):
    require_cuda(x, out)
    n, h, w, c = x.shape
    assert x.dtype == out.dtype
    fn = lib.mega_maxpool3x3s2_nhwc_f16 if x.dtype == torch.float16 else lib.mega_maxpool3x3s2_nhwc
    check(fn(ptr(x), n, h, w, c, ptr(out), stream_ptr()), "mega_maxpool3x3s2_nhwc")
    LAUNCHES[0] += 1
    return out


def _as_f32_rows(t):
    """rows of fp16 features are moved as rows of half as many 32-bit words"""
    return t.view(torch.float32) if t.dtype == torch.float16 else t


def gather_rows(src, idx, dst, n_rows=None, row_len=None):
    require_cuda(src, idx, dst)
    assert idx.dtype == torch.int32 and src.dtype == dst.dtype
    if src.dtype == torch.float16:
        assert row_len is None
        src, dst = _as_f32_rows(src), _as_f32_rows(dst)
    n_rows = idx.numel() if n_rows is None else n_rows
    row_len = src.shape[-1] if row_len is None else row_len
    if copy_batch.active[0] is not None:
        copy_batch.active[0].append(_copy_job(src, idx, dst, None, n_rows, row_len))
        return dst
    check(lib.mega_gather_rows(ptr(src), src.stride(-2), ptr(idx), n_rows, row_len, ptr(dst), dst.stride(-2),
                               stream_ptr()), "mega_gather_rows")
    LAUNCHES[0] += 1
    return dst


def copy_rows(src, dst, n_rows, row_len=None, src_idx=None, dst_idx=None):
    """dst[dst_idx[i]] = src[src_idx[i]] for i < n_rows (either index optional); 2-D row views."""
    require_cuda(src, dst, src_idx, dst_idx)
    assert src.dtype == dst.dtype
    if src.dtype == torch.float16:
        assert row_len is None
        src, dst = _as_f32_rows(src), _as_f32_rows(dst)
    row_len = src.shape[-1] if row_len is None else row_len
    if copy_batch.active[0] is not None:
        copy_batch.active[0].append(_copy_job(src, src_idx, dst, dst_idx, n_rows, row_len))
        return dst
    check(lib.mega_copy_rows(ptr(src), src.stride(-2), ptr(src_idx), ptr(dst), dst.stride(-2), ptr(dst_idx), n_rows,
                             row_len, stream_ptr()), "mega_copy_rows")
    LAUNCHES[0] += 1
    return dst


class copy_batch(object):
    """with ops.copy_batch(): the gather_rows / copy_rows calls inside are collected and issued as ONE launch on exit
    (they must be independent of each other)"""
    active = [None]

    def __enter__(self):
        copy_batch.active[0] = []
        return self

    def __exit__(self, et, ev, tb):
        jobs, copy_batch.active[0] = copy_batch.active[0], None
        if et is not None or not jobs:
            return False
        for i in range(0, len(jobs), 16):
            part = jobs[i:i + 16]
            arr = (_lib.CopyJob * len(part))(*part)
            check(lib.mega_copy_rows_batch(arr, len(part), stream_ptr()), "mega_copy_rows_batch")
            LAUNCHES[0] += 1
        return False


def _copy_job(src, src_idx, dst, dst_idx, n_rows, row_len):
    j = _lib.CopyJob()
    j.src, j.src_ld, j.src_idx = src.data_ptr(), src.stride(-2), (src_idx.data_ptr() if src_idx is not None else None)
    j.dst, j.dst_ld, j.dst_idx = dst.data_ptr(), dst.stride(-2), (dst_idx.data_ptr() if dst_idx is not None else None)
    j.n_rows, j.row_len = n_rows, row_len
    return j


def transpose_2d(x, out, n_img, rows, cols):
    require_cuda(x, out)
    check(lib.mega_transpose_2d(ptr(x), n_img, rows, cols, ptr(out), stream_ptr()), "mega_transpose_2d")
    LAUNCHES[0] += 1
    return out


def relation_softmax(logits, n_rows, ldm, scale, boxes_q=None, boxes_k=None, wg=None, bg=None, dim_mat=None,
                     m_valid=None, m_host=0, n_valid=None, n_valid_off=0, probs_f16=None, host_w=None):
    """in place over fp32 logits [16, n_rows, ldm]; with probs_f16 (fp16, same shape) the probabilities go there -- or, when
    probs_f16 is an fp32-typed tensor marked split-fp16, in the split-fp16 format"""
    split = probs_f16 is not None and probs_f16.dtype == torch.float32
    if split:
        assert is_split16(probs_f16) and probs_f16.numel() == logits.numel() and ldm % 32 == 0
    if host_w is not None and boxes_q is not None:
        # (wg [16,64], bg [16], dim_mat [8]) as contiguous fp32 HOST tensors: they travel in the kernel parameters
        require_cuda(logits, boxes_q, boxes_k, m_valid, n_valid, probs_f16)
        wg_h, bg_h, dim_h = host_w
        assert not wg_h.is_cuda and wg_h.dtype == torch.float32 and wg_h.is_contiguous() and wg_h.numel() == 1024
        assert probs_f16 is None or split or probs_f16.dtype == torch.float16
        fn = lib.mega_relation_softmax_pe_split16 if split else lib.mega_relation_softmax_pe
        check(fn(ptr(logits), ptr(probs_f16), n_rows, ldm, ptr(boxes_q), ptr(boxes_k),
                                           ptr(wg_h), ptr(bg_h), ptr(dim_h), ptr(m_valid), m_host, ptr(n_valid),
                                           n_valid_off, float(scale), stream_ptr()), "mega_relation_softmax_pe")
        LAUNCHES[0] += 1
        return logits
    require_cuda(logits, boxes_q, boxes_k, wg, bg, dim_mat, m_valid, n_valid, probs_f16)
    if probs_f16 is not None:
        assert split or probs_f16.dtype == torch.float16
        fn = lib.mega_relation_softmax_split16 if split else lib.mega_relation_softmax_f16
        check(fn(ptr(logits), ptr(probs_f16), n_rows, ldm, ptr(boxes_q), ptr(boxes_k),
                                            ptr(wg), ptr(bg), ptr(dim_mat), ptr(m_valid), m_host, ptr(n_valid),
                                            n_valid_off, float(scale), stream_ptr()), "mega_relation_softmax_f16")
    else:
        check(lib.mega_relation_softmax(ptr(logits), n_rows, ldm, ptr(boxes_q), ptr(boxes_k), ptr(wg), ptr(bg),
                                        ptr(dim_mat), ptr(m_valid), m_host, ptr(n_valid), n_valid_off, float(scale),
                                        stream_ptr()), "mega_relation_softmax")
    LAUNCHES[0] += 1
    return logits


def box_postprocess(logits, deltas, proposals, count, num_classes, im_w, im_h, score_thresh, nms_thresh, max_det,
                    weights, out):
    """logits [R, ld] / deltas [R, ld] views (may alias one buffer); out = (boxes, scores, labels int64, count)."""
    require_cuda(logits, deltas, proposals, count)
    r = proposals.shape[0]
    nbytes = lib.mega_box_postprocess_workspace_bytes(r, num_classes)
    if nbytes < 0:
        raise _lib.MegaError("box_postprocess: at most 512 proposals per image")
    ws = _workspace("post", nbytes, logits.device)
    ob, os_, ol, oc = out
    check(lib.mega_box_postprocess(ptr(logits), logits.stride(0), ptr(deltas), deltas.stride(0), ptr(proposals),
                                   ptr(count), r, num_classes, float(im_w), float(im_h), float(score_thresh),
                                   float(nms_thresh), max_det, *[float(x) for x in weights], ptr(ws), ws.numel(),
                                   ptr(ob), ptr(os_), ptr(ol), ob.shape[0], ptr(oc), stream_ptr()),
          "mega_box_postprocess")
    LAUNCHES[0] += 2
    return out


# --------------------------------------------------------------------------- FGFA helpers (csrc/fgfa.cu)
def _is16(t):
    return 1 if t.dtype == torch.float16 else 0


def fgfa_pool_image(img, out):
    """img [1,3,H,W] or [3,H,W] fp32 -> out [ceil(H/2), ceil(W/2), 4] = avg_pool2d(img / 255, 2, ceil_mode)"""
    require_cuda(img, out)
    h, w = img.shape[-2:]
    assert img.dtype == torch.float32 and img.is_contiguous()
    check(lib.mega_fgfa_pool_image(ptr(img), h, w, ptr(out), _is16(out), stream_ptr()), "mega_fgfa_pool_image")
    LAUNCHES[0] += 1
    return out


def fgfa_build_pairs(ring, slots, key_pos, pairs):
    """ring [S, hq, wq, 4]; slots int32 [L] (device); pairs [L, hq+6, wq+8, 8]"""
    require_cuda(ring, slots, pairs)
    s, hq, wq, _ = ring.shape
    assert ring.dtype == pairs.dtype and slots.dtype == torch.int32
    check(lib.mega_fgfa_build_pairs(ptr(ring), ring.stride(0), ptr(slots), slots.numel(), key_pos, hq, wq, ptr(pairs),
                                    _is16(ring), stream_ptr()), "mega_fgfa_build_pairs")
    LAUNCHES[0] += 1
    return pairs


def avgpool2_nhwc(x, out):
    require_cuda(x, out)
    n, h, w, c = x.shape
    assert x.dtype == out.dtype and x.stride(3) == 1 and out.stride(3) == 1
    check(lib.mega_avgpool2_nhwc(ptr(x), n, h, w, c, x.stride(2), ptr(out), out.stride(2), _is16(x), stream_ptr()),
          "mega_avgpool2_nhwc")
    LAUNCHES[0] += 1
    return out


def fgfa_aggregate(ring, slots, key_pos, flow, out, feat_channels, embed_channels, weights_out=None):
    """ring [S, h, w, ld] ([feats | embeds] per pixel); flow [L, h, w, fl] fp32; out [h, w, >= feat_channels]"""
    require_cuda(ring, slots, flow, out, weights_out)
    s, h, w, ld = ring.shape
    assert flow.dtype == torch.float32 and ring.dtype == out.dtype
    check(lib.mega_fgfa_aggregate(ptr(ring), ring.stride(0), ld, feat_channels, embed_channels, ptr(slots), slots.numel(),
                                  key_pos, ptr(flow), flow.stride(2), h, w, ptr(out), out.stride(-2), ptr(weights_out),
                                  _is16(ring), stream_ptr()), "mega_fgfa_aggregate")
    LAUNCHES[0] += 1
    return out


def dff_warp_scale(key_feats, flow, scale, out):
    """key_feats [h, w, C]; flow [h, w, fl] fp32 (x, y in cells); scale [h, w, >=C]; out [h, w, >=C] = warp(key_feats) * scale"""
    require_cuda(key_feats, flow, scale, out)
    h, w, c = key_feats.shape
    assert flow.dtype == torch.float32 and key_feats.dtype == scale.dtype == out.dtype
    assert key_feats.stride(2) == 1 and scale.stride(2) == 1 and out.stride(2) == 1 and key_feats.stride(0) == w * key_feats.stride(1)
    check(lib.mega_dff_warp_scale(ptr(key_feats), key_feats.stride(1), c, ptr(flow), flow.stride(1), ptr(scale),
                                  scale.stride(1), h, w, ptr(out), out.stride(1), _is16(key_feats), stream_ptr()),
          "mega_dff_warp_scale")
    LAUNCHES[0] += 1
    return out


# ---------------------------------------------------------------------------------------------- device VID evaluator
VID_EVAL_MAX_RANGES = 4


def vid_eval_pack(pred_boxlists, gt_boxlists, motion_ious=None):
    """BoxLists -> flat arrays of mega_vid_eval_match, one torch.cat per field, on the BoxLists' device. motion_ious: per
    image a sequence of motion IoUs for its GT (or None); entries beyond the GT count are dropped and missing ones are
    NaN (never ignored), as calc_detection_vid_prec_rec does."""
    assert len(pred_boxlists) == len(gt_boxlists)
    det_n = torch.tensor([p.bbox.shape[0] for p in pred_boxlists], dtype=torch.int64)
    gt_n = torch.tensor([g.bbox.shape[0] for g in gt_boxlists], dtype=torch.int64)
    zero = torch.zeros(1, dtype=torch.int64)
    packed = {
        "det_boxes": torch.cat([p.bbox.reshape(-1, 4) for p in pred_boxlists]).float().contiguous(),
        "det_scores": torch.cat([p.get_field("scores").reshape(-1) for p in pred_boxlists]).float().contiguous(),
        "det_labels": torch.cat([p.get_field("labels").reshape(-1) for p in pred_boxlists]).int().contiguous(),
        "det_off": torch.cat([zero, det_n.cumsum(0)]),
        "gt_boxes": torch.cat([g.bbox.reshape(-1, 4) for g in gt_boxlists]).float().contiguous(),
        "gt_labels": torch.cat([g.get_field("labels").reshape(-1) for g in gt_boxlists]).int().contiguous(),
        "gt_off": torch.cat([zero, gt_n.cumsum(0)]),
        "gt_motion": None,
    }
    if motion_ious is not None:
        parts = []
        for m, g in zip(motion_ious, gt_n.tolist()):
            row = torch.full((g,), float("nan"), dtype=torch.float64)
            if m is not None and len(m) > 0:
                m = torch.as_tensor(m, dtype=torch.float64).reshape(-1)[:g]
                row[:m.numel()] = m
            parts.append(row)
        packed["gt_motion"] = torch.cat(parts) if parts else torch.zeros(0, dtype=torch.float64)
    labels = torch.cat([packed["det_labels"], packed["gt_labels"]])
    if labels.numel() == 0:
        raise ValueError("vid_eval: no detections and no ground truth")
    lo, hi = int(labels.min()), int(labels.max())
    if lo < 0:
        raise ValueError("vid_eval: negative class label %d" % lo)
    packed["num_classes"] = hi + 1
    return packed


def vid_eval(packed, ranges, empty_weights, iou_thresh=0.5, want_prec_rec=False, device="cuda"):
    """Scores packed BoxLists (vid_eval_pack) for up to 4 motion ranges on the GPU, on the current stream, without
    synchronising. Returns device tensors: ap [R, C] (NaN where a class has no positives), n_pos [R, C], seen [C] (label
    occurs: its precision curve exists), det_count [C], order [N] (detections by ascending (class, score); class c's
    block follows those of the classes below it), match / ignore [R, N], and with want_prec_rec prec / rec [R, N] (class c's
    curve in ranking order at the offset of its block in order; rec is NaN for classes without positives)."""
    dev = torch.device(device)
    r = len(ranges)
    if not 1 <= r <= VID_EVAL_MAX_RANGES or len(empty_weights) != r:
        raise _lib.MegaError("vid_eval: 1..%d ranges with one empty weight each" % VID_EVAL_MAX_RANGES)
    t = {k: (v.to(dev, non_blocking=True) if torch.is_tensor(v) else v) for k, v in packed.items()}
    require_cuda(t["det_boxes"], t["gt_boxes"])
    n, g, c = t["det_scores"].numel(), t["gt_labels"].numel(), packed["num_classes"]
    nbytes = lib.mega_vid_eval_workspace_bytes(n, g, c, r)
    if nbytes < 0:
        raise _lib.MegaError("vid_eval: %d detections / %d GT / %d classes / %d ranges exceed the evaluator's limits "
                             "(< 2^31 boxes, <= 512 classes)" % (n, g, c, r))
    ws = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=dev)
    out = {
        "match": torch.empty(r, n, dtype=torch.int8, device=dev),
        "ignore": torch.empty(r, n, dtype=torch.float64, device=dev),
        "n_pos": torch.empty(r, c, dtype=torch.int64, device=dev),
        "seen": torch.empty(c, dtype=torch.int32, device=dev),
        "det_count": torch.empty(c, dtype=torch.int32, device=dev),
        "order": torch.empty(n, dtype=torch.int32, device=dev),
        "ap": torch.empty(r, c, dtype=torch.float64, device=dev),
        "prec": torch.empty(r, n, dtype=torch.float64, device=dev) if want_prec_rec else None,
        "rec": torch.full((r, n), float("nan"), dtype=torch.float64, device=dev) if want_prec_rec else None,
    }
    rng = (ctypes.c_double * (2 * r))(*[float(x) for lh in ranges for x in lh])
    empty = (ctypes.c_double * r)(*[float(x) for x in empty_weights])
    n_img = t["det_off"].numel() - 1
    s = stream_ptr()
    check(lib.mega_vid_eval_match(ptr(t["det_boxes"]), ptr(t["det_scores"]), ptr(t["det_labels"]), ptr(t["det_off"]),
                                  ptr(t["gt_boxes"]), ptr(t["gt_labels"]), ptr(t["gt_motion"]), ptr(t["gt_off"]), n_img,
                                  n, g, c, r, rng, empty, float(iou_thresh), ptr(ws), ws.numel(), ptr(out["match"]),
                                  ptr(out["ignore"]), ptr(out["n_pos"]), ptr(out["seen"]), ptr(out["det_count"]), s),
          "mega_vid_eval_match")
    check(lib.mega_vid_eval_rank(n, g, c, r, ptr(ws), ws.numel(), ptr(out["order"]), s), "mega_vid_eval_rank")
    check(lib.mega_vid_eval_scan_ap(ptr(out["match"]), ptr(out["ignore"]), ptr(out["order"]), ptr(out["det_count"]),
                                    ptr(out["n_pos"]), n, g, c, r, ptr(ws), ws.numel(), ptr(out["prec"]), ptr(out["rec"]),
                                    ptr(out["ap"]), s), "mega_vid_eval_scan_ap")
    LAUNCHES[0] += 2 + 3 * ((32 + (c - 1).bit_length() + 7) // 8)      # match, scan / AP, 3 per radix pass
    return out
