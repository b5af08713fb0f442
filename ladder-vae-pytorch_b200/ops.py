"""torch.autograd glue over the C-ABI kernels.

Tensors that cross this layer are *logical* NCHW (what the reference's modules exchange) but
*physically* NHWC: ``nhwc(x)`` returns the contiguous (B,H,W,C) view the kernels consume and
``as_nchw(y)`` re-labels a kernel output without copying.  Nothing here computes on the CPU
and nothing falls back to ATen for the hot ops; a missing library raises.
"""
from __future__ import annotations

import ctypes
import struct
import threading
from contextlib import contextmanager
from typing import List, Optional

import torch
from torch.autograd import Function

from . import _capi

call = _capi.call

ACT_IDS = {None: 0, "none": 0, "relu": 1, "leakyrelu": 2, "elu": 3, "selu": 4}


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _dt(t) -> int:
    if t.dtype == torch.float32:
        return 0
    if t.dtype == torch.bfloat16:
        return 1
    raise TypeError("lvae_b200 kernels take float32 or bfloat16 activations, got %s" % t.dtype)


def _require_cuda(t):
    if not t.is_cuda:
        raise RuntimeError("lvae_b200 has no CPU path: tensors must live on a CUDA (sm_100a) device")


def nhwc(x: torch.Tensor) -> torch.Tensor:
    """logical NCHW -> contiguous (B,H,W,C) (zero-copy when x is already NHWC-physical)."""
    y = x.permute(0, 2, 3, 1)
    return y if y.is_contiguous() else y.contiguous()


def as_nchw(y: torch.Tensor) -> torch.Tensor:
    """(B,H,W,C) contiguous kernel output -> logical NCHW view."""
    return y.permute(0, 3, 1, 2)


# --------------------------------------------------------------------------- RNG + injection
class _Rng(threading.local):
    def __init__(self):
        self.state = {}        # device index -> int64[2] tensor (seed, offset)
        self.seed = None
        self.stream_id = 0
        self.rank = 0          # folded into the Philox key (data-parallel replicas must not share noise)


_rng = _Rng()


def manual_seed(seed: int) -> None:
    _rng.seed = int(seed)
    _rng.state = {}
    _rng.stream_id = 0


def _philox_key() -> int:
    base = _rng.seed if _rng.seed is not None else (torch.initial_seed() & 0x7FFFFFFFFFFFFFFF)
    return (base ^ ((_rng.rank * 0x9E3779B97F4A7C15) & 0x7FFFFFFFFFFFFFFF)) & 0x7FFFFFFFFFFFFFFF


def rng_state(device) -> torch.Tensor:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    st = _rng.state.get(idx)
    if st is None:
        st = torch.tensor([_philox_key(), 0], dtype=torch.int64, device=torch.device("cuda", idx))
        _rng.state[idx] = st
    return st


def fold_rank(rank: int) -> None:
    """Give this process its own Philox key (seed ^ f(rank)); idempotent, keeps the offsets of existing states."""
    if int(rank) == _rng.rank:
        return
    _rng.rank = int(rank)
    for st in _rng.state.values():
        st[0:1].fill_(_philox_key())


@contextmanager
def shared_key():
    """Temporarily the SAME Philox key on every rank (the importance-weighted evaluator numbers its samples globally: sample k
    of a batch is (key, offset k) on whichever rank computes it); the per-rank key of a training engine comes back after."""
    rank = _rng.rank
    fold_rank(0)
    try:
        yield
    finally:
        fold_rank(rank)


def next_stream_id() -> int:
    _rng.stream_id += 1
    return _rng.stream_id


def set_stream_id(v: int) -> None:
    _rng.stream_id = int(v)


RNG_STEP = 1 << 36      # Philox offset advance per step / importance sample (no site of one step draws that many quads)


def rng_advance(device, inc: int = RNG_STEP) -> None:
    call("lvae_rng_advance", rng_state(device).data_ptr(), inc, _stream())


class StepContext(threading.local):
    """Per-forward side inputs: injected eps / dropout masks (parity tests) or one pre-drawn
    mask arena for all Dropout2d sites of a forward (one launch instead of ~300)."""

    def __init__(self):
        self.eps: Optional[List[torch.Tensor]] = None
        self.masks: Optional[List[torch.Tensor]] = None
        self.mask_arena: Optional[torch.Tensor] = None
        self.mask_cursor = 0
        # (3, L, B) fp32 rows [kl_samplewise | logprob_p | logprob_q] of the L stochastic layers of one top-down pass: every
        # layer's kernel writes its row, lvae_kl_bookkeeping reads the matrices (no torch.stack, no per-layer reductions)
        self.kl_rows: Optional[torch.Tensor] = None
        self.kl_cursor = 0


_ctx = StepContext()


@contextmanager
def inject(eps=None, masks=None):
    """Feed fixed noise to the next forward: ``eps`` = list of (B,Z,h,w) tensors in execution
    (top-down) order, ``masks`` = list of (B,C,1,1) or (B,C) keep masks already scaled by 1/(1-p)."""
    old = (_ctx.eps, _ctx.masks)
    _ctx.eps = list(eps) if eps is not None else None
    _ctx.masks = list(masks) if masks is not None else None
    try:
        yield
    finally:
        _ctx.eps, _ctx.masks = old


def pop_eps():
    if _ctx.eps is None:
        return None
    if not _ctx.eps:
        raise RuntimeError("injected eps list exhausted")
    return _ctx.eps.pop(0)


def prepare_masks(n_sites: int, batch: int, channels: int, p: float, device) -> None:
    """Draw all Dropout2d masks of one forward in a single launch."""
    if _ctx.masks is not None or n_sites == 0 or not p:
        _ctx.mask_arena = None
        return
    arena = torch.empty((n_sites, batch, channels), dtype=torch.float32, device=device)
    call("lvae_dropout_masks", arena.data_ptr(), arena.numel(), float(p), rng_state(device).data_ptr(),
         next_stream_id(), _stream())
    _ctx.mask_arena, _ctx.mask_cursor = arena, 0


def begin_kl_rows(n_layers: int, batch: int, device) -> None:
    """LadderVAE.topdown_pass (inference): reserve one row per stochastic layer for this pass."""
    _ctx.kl_rows = torch.empty((3, n_layers, batch), dtype=torch.float32, device=device)
    _ctx.kl_cursor = 0


def end_kl_rows():
    rows, _ctx.kl_rows = _ctx.kl_rows, None
    return rows


def _take_kl_row(batch: int, device):
    """(kl, logp, logq) output vectors of one stochastic block: the next row of the pass's matrices, or fresh tensors."""
    r = _ctx.kl_rows
    if r is not None and _ctx.kl_cursor < r.shape[1] and r.shape[2] == batch and r.device == device:
        i = r.shape[1] - 1 - _ctx.kl_cursor        # the top-down pass visits layers L-1 .. 0: row index = layer index
        _ctx.kl_cursor += 1
        return r[0, i], r[1, i], r[2, i]
    v = torch.empty((3, batch), dtype=torch.float32, device=device)
    return v[0], v[1], v[2]


def clear_masks() -> None:
    _ctx.mask_arena = None
    _ctx.mask_cursor = 0


def next_mask(batch: int, channels: int, p: float, device) -> Optional[torch.Tensor]:
    """(B,C) fp32 keep mask scaled by 1/(1-p) for one Dropout2d site (None when p == 0)."""
    if _ctx.masks is not None:
        if not _ctx.masks:
            raise RuntimeError("injected dropout mask list exhausted")
        m = _ctx.masks.pop(0)
        return m.reshape(batch, channels).to(device=device, dtype=torch.float32).contiguous()
    if not p:
        return None
    a = _ctx.mask_arena
    if a is not None and _ctx.mask_cursor < a.shape[0] and a.shape[1] == batch and a.shape[2] == channels:
        m = a[_ctx.mask_cursor]
        _ctx.mask_cursor += 1
        return m
    m = torch.empty((batch, channels), dtype=torch.float32, device=device)
    call("lvae_dropout_masks", m.data_ptr(), m.numel(), float(p), rng_state(device).data_ptr(),
         next_stream_id(), _stream())
    return m


# --------------------------------------------------------------------------- gradient sinks
def grad_sink(param) -> Optional[torch.Tensor]:
    """Engine-owned flat gradient arena slice for this parameter (kernels accumulate into it
    directly, autograd is bypassed for parameter gradients); None -> return grads normally."""
    return getattr(param, "_lvae_grad_sink", None)


# Gradient-readiness tracking for the data-parallel engine: the arena is cut into buckets in the order the backward pass
# produces gradients; when the last parameter gradient of a bucket has been issued, the engine's flush callback unpacks the
# bucket's packed weight gradients and starts its NCCL all-reduce on the communication stream while the backward goes on.
_grad_track = {"on": False, "record": None, "bucket_of": {}, "remaining": [], "pending": [], "seen": set(), "flush": None}


def grad_track_begin(bucket_of, counts, flush, record=None) -> None:
    _grad_track.update(on=True, record=record, bucket_of=bucket_of, remaining=list(counts), pending=[], seen=set(), flush=flush)


def grad_track_end() -> None:
    """Flush whatever became ready at the last gradient site and stop tracking."""
    check_no_pending_bn1()
    t = _grad_track
    if t["on"]:
        for k in t["pending"]:
            t["flush"](k)
    t.update(on=False, record=None, pending=[], flush=None)


def grad_site() -> None:
    """Called at the top of every function that produces parameter gradients (conv / BatchNorm / head backward), before it
    announces its own parameters: everything the earlier sites announced has been launched by now, so the buckets they
    completed can go out.  (A site announces weight AND bias before it launches: flushing from inside the announcement
    would reduce a bucket ahead of the kernel that writes its last gradient.)"""
    t = _grad_track
    if t["on"] and t["pending"]:
        for k in t["pending"]:
            t["flush"](k)
        t["pending"] = []


def _grad_note(param) -> None:
    t = _grad_track
    pid = id(param)
    if pid in t["seen"]:
        return
    t["seen"].add(pid)
    if t["record"] is not None:
        t["record"].add(pid)
    k = t["bucket_of"].get(pid)
    if k is None or not t["remaining"]:
        return
    t["remaining"][k] -= 1
    if t["remaining"][k] == 0:
        t["pending"].append(k)


def _param_grad_buffer(param):
    sink = grad_sink(param)
    if sink is not None:
        if _grad_track["on"]:
            _grad_note(param)
        return sink, True
    return torch.zeros_like(param, dtype=torch.float32, memory_format=torch.contiguous_format), False


# --------------------------------------------------------------------------- packed weights
_PACK_FMT = "<QQiiiiii"   # must match LvaePackDesc in csrc/conv_generic.cu
_pack_epoch = [0]         # bumped whenever weights were updated behind torch's version counters


def bump_pack_epoch() -> None:
    """Our fused optimizer writes parameters through raw pointers; this invalidates every
    cached GEMM-layout copy so the next forward re-packs."""
    _pack_epoch[0] += 1



_hook_dirty = [False]


def note_conv_call(hooked: bool) -> None:
    """Forward hooks on conv modules (boilr's data_dependent_init, experiment_manager.py:62-72) rewrite `weight.data` in
    place AFTER the module's forward, which torch's version counter does not see.  A hooked call marks the packed-weight
    caches suspect; the first conv module called without hooks afterwards (the stem, at the top of the next forward)
    invalidates them all."""
    if hooked:
        _hook_dirty[0] = True
    elif _hook_dirty[0]:
        _hook_dirty[0] = False
        bump_pack_epoch()


class WeightPack:
    """GEMM-ready copy of one conv weight (see lvae_pack_weights).  Re-packed when the
    parameter's version counter or storage changes (i.e. after every optimizer step).
    modes 0/1: [K][ld] rows for the CUDA-core kernel; modes 2/3: bf16 K-major operand tiles
    [tap][k-block][Npad][64] for the tcgen05 kernel (forward / dgrad)."""

    def __init__(self, O: int, I: int, taps: int, mode: int):
        self.O, self.I, self.taps, self.mode = O, I, taps, mode
        if mode >= 2:
            nreal, kreal = (O, I) if mode == 2 else (I, O)
            self.ld = 64
            self.rows = taps * ((kreal + 63) // 64) * ((nreal + 15) // 16 * 16)
        else:
            n = O if mode == 0 else I
            self.ld = (n + 3) // 4 * 4
            self.rows = taps * (I if mode == 0 else O)
        self.buf = None
        self.desc = None
        self.desc_src = None
        self.key = None

    def alloc(self, weight: torch.Tensor, dtype: torch.dtype) -> bytes:
        """(Re)allocate the packed buffer and return the raw LvaePackDesc for it."""
        if self.mode >= 2:
            dtype = torch.bfloat16
        self.buf = torch.empty((self.rows, self.ld), dtype=dtype, device=weight.device)
        raw = struct.pack(_PACK_FMT, weight.data_ptr(), self.buf.data_ptr(), self.O, self.I, self.taps,
                          self.mode, self.ld, 0 if dtype == torch.float32 else 1)
        assert len(raw) == _capi.lib().lvae_pack_desc_size()
        self.desc = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(weight.device)
        self.desc_src = weight.data_ptr()
        return raw

    def get(self, weight: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
        if self.mode >= 2:
            dtype = torch.bfloat16
        key = (weight.data_ptr(), weight._version, dtype, weight.device, _pack_epoch[0])
        if self.key == key:
            return self.buf
        if self.buf is None or self.buf.dtype != dtype or self.buf.device != weight.device or \
                self.desc_src != weight.data_ptr():
            self.alloc(weight, dtype)
        call("lvae_pack_weights", self.desc.data_ptr(), 1, _stream())
        self.key = key
        return self.buf

    def mark_fresh(self, weight, dtype):
        """The engine packed every weight in one batched launch; record that this one is current."""
        if self.mode >= 2:
            dtype = torch.bfloat16
        self.key = (weight.data_ptr(), weight._version, dtype, weight.device, _pack_epoch[0])


_tc_enabled = [True]


def set_tensor_cores(flag: bool) -> None:
    """Route eligible bf16 convolutions to the tcgen05 kernel (default) or keep them on the CUDA-core one."""
    _tc_enabled[0] = bool(flag)


def _pow2(v: int) -> bool:
    return v > 0 and (v & (v - 1)) == 0


TC_REJECTED, TC_RESIDENT, TC_STREAMED = 0, 1, 2
_tc_plans = {}


def conv_tc_plan(cin: int, n: int, k: int, two_inputs: bool, h: int, w: int, out_f32: bool) -> int:
    """How lvae_conv2d_tc holds the weights of this launch shape: TC_REJECTED, TC_RESIDENT or TC_STREAMED.  The library's
    own rule (lvae_conv2d_tc_plan, the code the launch runs), asked once per shape."""
    key = (cin, n, k, bool(two_inputs), h, w, bool(out_f32))
    plan = _tc_plans.get(key)
    if plan is None:
        plan = _tc_plans[key] = int(_capi.lib().lvae_conv2d_tc_plan(*(int(v) for v in key)))
    return plan


class ConvSpec:
    """Static geometry + packed-weight caches of one conv module (Conv2d or ConvTranspose2d)."""

    def __init__(self, cout, cin, k, stride, pad, transposed=False, output_padding=0):
        self.cout, self.cin, self.k, self.stride, self.pad = cout, cin, k, stride, pad
        self.transposed, self.output_padding = transposed, output_padding
        self.out_fp32 = False         # bf16 pipeline: keep this conv's output in fp32 (stochastic / likelihood inputs)
        taps = k * k
        if not transposed:            # weight (Cout, Cin, k, k)
            self.pack_fwd = WeightPack(cout, cin, taps, 0)    # rows (tap, ci) -> cols co
            self.pack_bwd = WeightPack(cout, cin, taps, 1)    # rows (tap, co) -> cols ci
        else:                         # weight (Cin, Cout, k, k): O' = Cin, I' = Cout
            self.pack_fwd = WeightPack(cin, cout, taps, 1)    # rows (tap, ci) -> cols co
            self.pack_bwd = WeightPack(cin, cout, taps, 0)    # rows (tap, co) -> cols ci
        self.tc_shape = (not transposed) and stride == 1 and k in (1, 3) and pad == k // 2
        self.pack_tc_fwd = WeightPack(cout, cin, taps, 2) if self.tc_shape else None
        self.pack_tc_bwd = WeightPack(cout, cin, taps, 3) if self.tc_shape else None
        # stride-2 3x3 64 -> 64 (the down / up-sampling convs): lvae_conv2d_tc_s2.  With d0, d1 = the weight tensor's first
        # two dims, the "gather" kind multiplies by blocks [N = d0][K = d1] (mode 2), the "transposed" kind by [N = d1][K = d0]
        # (mode 3).  Conv2d: forward = gather, dgrad = transposed; ConvTranspose2d: the other way round.
        self.s2_shape = (k == 3 and stride == 2 and pad == 1 and cin == 64 and cout == 64
                         and (not transposed or output_padding == 1))
        d0, d1 = (cin, cout) if transposed else (cout, cin)
        self.pack_s2_gather = WeightPack(d0, d1, taps, 2) if self.s2_shape else None
        self.pack_s2_scatter = WeightPack(d0, d1, taps, 3) if self.s2_shape else None

    def packs(self, bf16: bool):
        """Packs the engine refreshes in its one batched launch per step.  In the bf16 pipeline the convolutions that run on
        the tensor cores only need their tcgen05 operand tiles; a CUDA-core fallback (odd image size) re-packs on demand."""
        if bf16 and self.tc_shape and self.cin % 64 == 0:
            return [self.pack_tc_fwd, self.pack_tc_bwd]
        out = [self.pack_fwd, self.pack_bwd]
        if bf16 and self.tc_shape:
            out += [self.pack_tc_fwd, self.pack_tc_bwd]
        if bf16 and self.s2_shape:
            out += [self.pack_s2_gather, self.pack_s2_scatter]
        return out

    def s2_ok(self, t, small_h: int, small_w: int) -> bool:
        """tcgen05 path for the stride-2 convs: bf16 (B,H,W,64) operand, the smaller grid a power of two, W <= 64."""
        return (_tc_enabled[0] and self.s2_shape and t.dtype == torch.bfloat16 and t.shape[3] == 64
                and _pow2(small_h) and _pow2(small_w) and small_w <= 64)

    def out_hw(self, h, w):
        if not self.transposed:
            return ((h + 2 * self.pad - self.k) // self.stride + 1, (w + 2 * self.pad - self.k) // self.stride + 1)
        return ((h - 1) * self.stride - 2 * self.pad + self.k + self.output_padding,
                (w - 1) * self.stride - 2 * self.pad + self.k + self.output_padding)

    def tc_forward_ok(self, xn, x2n) -> bool:
        if not (_tc_enabled[0] and self.tc_shape and xn.dtype == torch.bfloat16 and self.cout <= 256):
            return False
        B, H, W, C = xn.shape
        if not (_pow2(H) and _pow2(W) and W <= 128 and C % 64 == 0 and C <= 256):
            return False
        if x2n is not None and x2n.shape[3] != C:
            return False
        return conv_tc_plan(C, self.cout, self.k, x2n is not None, H, W, self.out_fp32) != TC_REJECTED

    def tc_dgrad_ok(self, gyn, out_f32: bool = False) -> bool:
        if not (_tc_enabled[0] and self.tc_shape and self.cin <= 256):
            return False
        B, H, W, N = gyn.shape
        return (_pow2(H) and _pow2(W) and W <= 128 and N % 64 == 0 and N <= 256
                and conv_tc_plan(N, self.cin, self.k, False, H, W, out_f32) != TC_REJECTED)


# Weight gradients depend only on saved activations and the output gradient, and nothing reads them before the
# optimizer: the engine lets them run on a side stream (a parallel branch of the captured graph) so that the
# small, latency-bound wgrad kernels overlap the dgrad / BatchNorm chain.
_side = {"streams": None, "keep": [], "next": 0, "log": {}}     # log: stream slot (-1 = current stream) -> packed-gradient ids


def set_side_stream(streams) -> None:
    """streams: list of side streams (weight-gradient launches rotate over them) or None."""
    if streams is not None and not isinstance(streams, (list, tuple)):
        streams = [streams]
    _side["streams"] = list(streams) if streams else None
    _side["keep"] = []
    _side["next"] = 0
    _side["log"] = {}


def packed_grad_log():
    """{stream slot: [packed-gradient ids whose wgrad was issued there since set_side_stream]} (slot -1: current stream)."""
    return _side["log"]


def join_side_stream() -> None:
    sts = _side["streams"]
    if sts:
        for st in sts:
            torch.cuda.current_stream().wait_stream(st)
    _side["keep"] = []


@contextmanager
def _wgrad_stream(sunk: bool, keep):
    """Issue the enclosed weight-gradient launches on the next side stream, after the current stream's work so far, when
    side streams are set and the gradients go to engine-owned sinks (else on the current stream).  keep: the operands, held
    until join_side_stream.  Yields the stream slot for packed_grad_log (-1: the current stream)."""
    sts = _side["streams"]
    if not (sts and sunk):
        yield -1
        return
    slot = _side["next"] % len(sts)
    _side["next"] += 1
    sts[slot].wait_event(torch.cuda.current_stream().record_event())
    _side["keep"].append(keep)
    with torch.cuda.stream(sts[slot]):
        yield slot


_wgrad_ws = {}
stats = {"tc_fwd": 0, "tc_dgrad": 0, "tc_wgrad": 0, "cc_fwd": 0, "cc_dgrad": 0, "cc_wgrad": 0}   # path counters (tests)


def _wgrad_workspace(device) -> torch.Tensor:
    """Scratch packed gradient of lvae_conv2d_wgrad_tc (stream-ordered reuse: one per stream)."""
    key = (device, torch.cuda.current_stream().cuda_stream)
    ws = _wgrad_ws.get(key)
    if ws is None:
        ws = torch.empty(512 * 128, dtype=torch.float32, device=device)        # one packed gradient (<= 5 pairs x 128 x 64)
        _wgrad_ws[key] = ws
    return ws


_wgrad_tc_fits = {}


def wgrad_tc_plan(N: int, k: int, two_inputs: bool):
    """dY windows ((width, first dY channel), ...) of the tensor-core weight gradient of a stride-1 conv with N output
    channels (a multiple of 64), or () when the kernel cannot take it.  What fits is the library's own rule
    (lvae_wgrad_tc_packed_size > 0); a shape that does not fit TMEM runs over 128- or 64-channel windows of dY (a 3x3 conv
    with N = 128: two launches).  PackedGradArena gives a packed gradient exactly to the single-launch shapes."""
    def fits(n):
        key = (n, k, bool(two_inputs))
        ok = _wgrad_tc_fits.get(key)
        if ok is None:
            ok = _wgrad_tc_fits[key] = int(_capi.lib().lvae_wgrad_tc_packed_size(n, k, int(bool(two_inputs)))) > 0
        return ok
    if N <= 0 or N % 64 or N > 256:
        return ()
    if N <= 128 and fits(N):
        return ((N, 0),)
    for n in (128, 64):
        if n < N and N % n == 0 and fits(n):
            return tuple((n, c0) for c0 in range(0, N, n))
    return ()


def wgrad_tc_windows(N: int, k: int, two_inputs: bool, xC: int):
    """(first X channel, width, first dY channel) of every launch of the tensor-core weight gradient when each input has
    xC > 64 channels: the dY windows of wgrad_tc_plan, once per 64-channel X window.  () when the kernel cannot take it."""
    if xC % 64 or xC > 256:
        return ()
    return tuple((x0, n, c0) for x0 in range(0, xC, 64) for n, c0 in wgrad_tc_plan(N, k, two_inputs))


def _tc_fusable(N, out_f32, nsplit=0) -> bool:
    """Can the conv's epilogue carry a fused per-channel reduction (TMA-store path of lvae_conv2d_tc, with or without a
    residual)?"""
    return N == 64 and not out_f32 and not nsplit


def _conv_tc(x, x2, wp, bias, out_scale, res, N, ksize, flip, out_f32, nsplit=0, stats_acc=None, bnb=None, gate=None, fold=None):
    """Launch the tcgen05 kernel.  Returns y, or (y, y2) when nsplit splits the output columns.
    stats_acc: (2,64) float64 accumulator for the output's per-channel statistics; bnb = (x, save, gamma, beta, acc, act):
    BatchNorm-backward sums over the output (both fused into the epilogue)."""
    B, H, W, C = x.shape
    odt = torch.float32 if out_f32 else torch.bfloat16
    if nsplit:
        y = torch.empty((B, H, W, nsplit), dtype=odt, device=x.device)
        y2 = torch.empty((B, H, W, N - nsplit), dtype=odt, device=x.device)
    else:
        y, y2 = torch.empty((B, H, W, N), dtype=odt, device=x.device), None
    streamed = conv_tc_plan(C, N, ksize, x2 is not None, H, W, out_f32) == TC_STREAMED
    if streamed:
        key = "tc_dgrad_streamed" if flip else "tc_fwd_streamed"
        stats[key] = stats.get(key, 0) + 1
    if res is not None and not out_f32:
        # bf16 residual: added in the TMA-store epilogue (resident weights, N % 64 == 0, N <= 128), else by scattered row stores
        key = "res_tma" if (N % 64 == 0 and N <= 128 and not streamed) else "res_scattered"
        stats[key] = stats.get(key, 0) + 1
    fuse = None
    gate_out = None
    if stats_acc is not None or bnb is not None or gate is not None or fold is not None:
        f = _capi.ConvFuse()
        f.stats_acc = _p(stats_acc)
        if fold is not None:            # eval-mode BatchNorm + activation of the consumer: (gamma, beta, mean, var, eps, act)
            fg, fb, fm, fv, feps, fact = fold[:6]
            f.fold_gamma, f.fold_beta, f.fold_mean, f.fold_var = fg.data_ptr(), fb.data_ptr(), fm.data_ptr(), fv.data_ptr()
            f.fold_eps, f.fold_act = float(feps), int(fact)
            if len(fold) > 6 and fold[6] is not None:     # + the eval-mode BatchNorm in front of the conv: (gamma, beta, mean, var, eps)
                pg, pb, pm, pv, peps = fold[6]
                f.pre_gamma, f.pre_beta, f.pre_mean, f.pre_var = pg.data_ptr(), pb.data_ptr(), pm.data_ptr(), pv.data_ptr()
                f.pre_eps = float(peps)
        if gate is not None:            # (residual input (B,H,W,64) bf16, activation id): gated residual output in the epilogue
            gx, gact = gate
            gate_out = torch.empty_like(gx)
            f.gate_x, f.gate_out, f.gate_act = gx.data_ptr(), gate_out.data_ptr(), int(gact)
            f.gate_skip_h = 0 if _gate_keep_h[0] else 1     # no backward will run (no_grad caller): h = [a | g] is not stored
        if bnb is not None:
            bx, bsave, bgamma, bbeta, bacc, bact = bnb
            f.bnb_x, f.bnb_save, f.bnb_gamma, f.bnb_beta = bx.data_ptr(), bsave.data_ptr(), bgamma.data_ptr(), bbeta.data_ptr()
            f.bnb_acc, f.bnb_act = bacc.data_ptr(), int(bact)
        fuse = ctypes.addressof(f)
    call("lvae_conv2d_tc_ex", x.data_ptr(), _p(x2), wp.data_ptr(), _p(bias), _p(out_scale), _p(res), y.data_ptr(), _p(y2),
         nsplit, B, H, W, C, N, ksize, 1 if flip else 0, 1 if out_f32 else 0, fuse, _stream())
    if gate is not None:
        return y, gate_out
    return (y, y2) if nsplit else y


def _gather(x, x2, wp, ld, bias, in_scale, out_scale, res, B, Hi, Wi, C1, C2, Ho, Wo, N, k, stride, pad, mode, out_dtype):
    y = torch.empty((B, Ho, Wo, N), dtype=out_dtype, device=x.device)
    call("lvae_conv2d_gather", x.data_ptr(), _p(x2), wp.data_ptr(), _p(bias), _p(in_scale), _p(out_scale), _p(res),
         y.data_ptr(), B, Hi, Wi, C1, C2, Ho, Wo, N, ld, k, k, stride, pad, mode, _dt(x), _stream())
    return y


def conv_forward_raw(spec: ConvSpec, xn, x2n, weight, bias, out_scale, resn, stats_acc=None, window=None):
    """(conv(cat(xn, x2n)) + bias) * out_scale + resn on NHWC tensors.  bf16 activations on eligible shapes run on
    the tensor cores (lvae_conv2d_tc), everything else on the CUDA-core implicit GEMM (lvae_conv2d_gather)."""
    B, Hi, Wi, C1 = xn.shape
    C2 = x2n.shape[3] if x2n is not None else 0
    padded = x2n is None and C1 > spec.cin          # zero-padded input channels (bf16 copy of z): tensor-core path only
    assert padded or C1 + C2 == spec.cin, "conv input channels %d+%d != %d" % (C1, C2, spec.cin)
    Ho, Wo = spec.out_hw(Hi, Wi)
    want_f32 = spec.out_fp32 and xn.dtype == torch.bfloat16
    if x2n is None and resn is None and not want_f32 and spec.s2_shape:
        hs, ws = (Hi, Wi) if spec.transposed else (Ho, Wo)
        if spec.s2_ok(xn, hs, ws):
            stats["tc_fwd"] += 1
            pack = spec.pack_s2_scatter if spec.transposed else spec.pack_s2_gather
            y = torch.empty((B, Ho, Wo, spec.cout), dtype=torch.bfloat16, device=xn.device)
            call("lvae_conv2d_tc_s2", xn.data_ptr(), pack.get(weight, torch.bfloat16).data_ptr(), _p(bias), _p(out_scale),
                 y.data_ptr(), B, hs, ws, spec.cout, 1 if spec.transposed else 0, _stream())
            return (y, False) if stats_acc is not None else y
    if (spec.cout <= 4 and spec.k == 3 and spec.stride == 1 and spec.pad == 1 and not spec.transposed and x2n is None
            and resn is None and out_scale is None and xn.dtype == torch.bfloat16 and C1 == 64 and spec.cin == 64):
        # narrow head (Bernoulli parameter_net, 64 -> 1): a GEMM tile would be 63/64 padding
        stats["narrow_fwd"] = stats.get("narrow_fwd", 0) + 1
        y = torch.empty((B, Ho, Wo, spec.cout), dtype=torch.float32 if want_f32 else torch.bfloat16, device=xn.device)
        rp, ip = window if window is not None else (0, 0)     # xn may be a window of a larger NHWC tensor (zero-copy crop)
        call("lvae_conv3x3_narrow_ex", xn.data_ptr(), weight.data_ptr(), _p(bias), y.data_ptr(), B, Hi, Wi, spec.cout,
             1 if want_f32 else 0, int(rp), int(ip), _stream())
        return (y, False) if stats_acc is not None else y
    assert window is None, "only the narrow head convolution reads a windowed input"
    if padded and not spec.tc_forward_ok(xn, x2n):
        xn, C1 = xn[..., :spec.cin].contiguous(), spec.cin
    if spec.tc_forward_ok(xn, x2n) and (resn is None or resn.dtype == (torch.float32 if want_f32 else torch.bfloat16)):
        wp = spec.pack_tc_fwd.get(weight, torch.bfloat16)
        stats["tc_fwd"] += 1
        fused = stats_acc is not None and _tc_fusable(spec.cout, want_f32)
        y = _conv_tc(xn, x2n, wp, bias, out_scale, resn, spec.cout, spec.k, False, want_f32,
                     stats_acc=stats_acc if fused else None)
        return (y, fused) if stats_acc is not None else y
    wp = spec.pack_fwd.get(weight, xn.dtype)
    if resn is not None and resn.dtype != xn.dtype:
        resn = resn.to(xn.dtype)
    stats["cc_fwd"] += 1
    y = _gather(xn, x2n, wp, spec.pack_fwd.ld, bias, None, out_scale, resn, B, Hi, Wi, C1, C2, Ho, Wo,
                spec.cout, spec.k, spec.stride, spec.pad, 1 if spec.transposed else 0, xn.dtype)
    y = y.float() if want_f32 else y
    return (y, False) if stats_acc is not None else y


def conv_backward_raw(spec: ConvSpec, xn, x2n, weight, bias, out_scale, gyn, need_x=True, need_w=True, need_b=True,
                      dx_scale=None, bnb=None):
    """Data and parameter gradients of conv_forward_raw.  ``out_scale`` is the forward's Dropout2d mask (gyn is the
    gradient wrt the masked output; pass None when gyn is already the gradient wrt the raw conv output).
    ``dx_scale`` (B, Cin) is folded into the dgrad epilogue: the returned dx is multiplied by it (the mask of the
    conv that produced xn).  Returns (gx, gx2, gw, gb); gw / gb are None when accumulated into a gradient sink."""
    grad_site()
    if gyn.dtype != xn.dtype:
        lp = _lowp_grad_take(gyn, xn.dtype) if gyn.dtype == torch.float32 else None
        gyn = lp if lp is not None else gyn.to(xn.dtype)
    B, Hi, Wi, C1 = xn.shape
    C2 = x2n.shape[3] if x2n is not None else 0
    _, Ho, Wo, N = gyn.shape
    gx = gx2 = gw = gb = None
    conv_backward_raw.last_fused = False
    padded = x2n is None and C1 > spec.cin
    use_tc = xn.dtype == torch.bfloat16 and spec.tc_dgrad_ok(gyn, padded)
    if padded and not use_tc:
        xn, C1, padded = xn[..., :spec.cin].contiguous(), spec.cin, False
    # stride-2 convs on the tensor cores: dgrad of Conv2d = "transposed" kind over the dy grid, dgrad of ConvTranspose2d =
    # "gather" kind onto the (smaller) x grid; their weight gradients read the stride-2-shifted operand through an
    # element-strided tensor map
    hs2, ws2 = (Hi, Wi) if spec.transposed else (Ho, Wo)
    s2 = x2n is None and spec.s2_ok(gyn, hs2, ws2) and xn.dtype == torch.bfloat16 and C1 == 64
    use_s2, use_s2w = need_x and s2, need_w and s2
    if (use_tc or use_s2 or use_s2w) and out_scale is not None:
        # TMA-fed operands never pass through registers: apply the Dropout2d mask in a separate pass
        gys = torch.empty_like(gyn)
        call("lvae_channel_scale", gyn.data_ptr(), out_scale.data_ptr(), gys.data_ptr(), B, Ho * Wo, N, _dt(gyn), _stream())
        gyn, out_scale = gys, None
    if need_x:
        if use_s2:
            stats["tc_dgrad"] += 1
            pack = spec.pack_s2_gather if spec.transposed else spec.pack_s2_scatter
            gx = torch.empty((B, Hi, Wi, 64), dtype=torch.bfloat16, device=gyn.device)
            call("lvae_conv2d_tc_s2", gyn.data_ptr(), pack.get(weight, torch.bfloat16).data_ptr(), None, _p(dx_scale),
                 gx.data_ptr(), B, hs2, ws2, 64, 0 if spec.transposed else 1, _stream())
        elif use_tc:
            wpb = spec.pack_tc_bwd.get(weight, torch.bfloat16)
            stats["tc_dgrad"] += 1
            if x2n is None:
                fuse_bnb = bnb is not None and not padded and _tc_fusable(spec.cin, False)
                # padded (conv_out of a stochastic block reading the 64-channel bf16 copy of z): the gradient goes to the
                # fp32, Z-channel z the autograd graph holds -> fp32 epilogue, no padding channels
                gx = _conv_tc(gyn, None, wpb, None, dx_scale, None, spec.cin, spec.k, True, padded,
                              bnb=bnb if fuse_bnb else None)
                if fuse_bnb:
                    stats["bnb_fused"] = stats.get("bnb_fused", 0) + 1
                    conv_backward_raw.last_fused = True
            else:
                assert dx_scale is None
                gx, gx2 = _conv_tc(gyn, None, wpb, None, None, None, spec.cin, spec.k, True, False, nsplit=C1)
        else:
            wpb = spec.pack_bwd.get(weight, gyn.dtype)
            stats["cc_dgrad"] += 1
            gcat = _gather(gyn, None, wpb, spec.pack_bwd.ld, None, out_scale, dx_scale, None, B, Ho, Wo, N, 0, Hi, Wi,
                           spec.cin, spec.k, spec.stride, spec.pad, 0 if spec.transposed else 1, gyn.dtype)
            if x2n is None:
                gx = gcat
            else:
                assert dx_scale is None
                gx, gx2 = gcat[..., :C1], gcat[..., C1:]
    if need_w:
        gwbuf, sunk = _param_grad_buffer(weight)
        gbbuf, bsunk = (None, True)
        if bias is not None and need_b:
            gbbuf, bsunk = _param_grad_buffer(bias)
        tc_ok = use_tc and out_scale is None and gyn.dtype == torch.bfloat16 and C2 in (0, C1)
        plan = wgrad_tc_plan(N, spec.k, C2 > 0) if (tc_ok and C1 == 64) else ()
        wins = wgrad_tc_windows(N, spec.k, C2 > 0, C1) if (tc_ok and C1 > 64) else ()
        with _wgrad_stream(sunk and bsunk, (xn, x2n, gyn, out_scale)) as slot:
            if wins:
                # wider inputs: one launch per (64-channel X window, dY window); the dY window's first X window adds the bias
                stats["tc_wgrad"] += 1
                stats["tc_wgrad_xwin"] = stats.get("tc_wgrad_xwin", 0) + 1
                row = spec.cin * spec.k * spec.k * 4
                for x0, n, c0 in wins:
                    call("lvae_conv2d_wgrad_tc_ex", xn.data_ptr(), _p(x2n), gyn.data_ptr(), gwbuf.data_ptr() + c0 * row,
                         None if (gbbuf is None or x0) else gbbuf.data_ptr() + c0 * 4,
                         _wgrad_workspace(xn.device).data_ptr(), B, Hi, Wi, n, spec.k, 0, 0, N, c0, C1, x0, _stream())
            elif plan:
                stats["tc_wgrad"] += 1
                gp = getattr(weight, "_lvae_gp", None) if (sunk and bsunk) else None
                if gp is not None:
                    # engine-owned packed gradient: every CTA reduce-adds into it, the engine unpacks them in batched launches
                    assert plan == ((N, 0),), "packed gradient of a conv whose weight gradient is split"
                    _side["log"].setdefault(slot, []).append(weight._lvae_gp_id)
                    call("lvae_conv2d_wgrad_tc_acc", xn.data_ptr(), _p(x2n), gyn.data_ptr(), gp.data_ptr(), B, Hi, Wi, N, spec.k,
                         0, 0, _stream())
                else:
                    # a split launch covers output channels [c0, c0 + n): rows c0.. of dw (N, cin, k, k) and of dbias
                    row = spec.cin * spec.k * spec.k * 4
                    for n, c0 in plan:
                        call("lvae_conv2d_wgrad_tc", xn.data_ptr(), _p(x2n), gyn.data_ptr(), gwbuf.data_ptr() + c0 * row,
                             None if gbbuf is None else gbbuf.data_ptr() + c0 * 4, _wgrad_workspace(xn.device).data_ptr(),
                             B, Hi, Wi, n, spec.k, spec.cin if padded else 0, 0, N, c0, _stream())
            elif use_s2w:
                stats["tc_wgrad"] += 1
                big, small = (gyn, xn) if spec.transposed else (xn, gyn)
                gp = getattr(weight, "_lvae_gp", None) if (sunk and bsunk) else None
                if gp is not None:
                    _side["log"].setdefault(slot, []).append(weight._lvae_gp_id)
                    call("lvae_conv2d_wgrad_tc_s2_acc", big.data_ptr(), small.data_ptr(), gp.data_ptr(), B, hs2, ws2, _stream())
                else:
                    call("lvae_conv2d_wgrad_tc_s2", big.data_ptr(), small.data_ptr(), gwbuf.data_ptr(),
                         None if spec.transposed else _p(gbbuf), _wgrad_workspace(xn.device).data_ptr(), B, hs2, ws2, _stream())
                if spec.transposed and gbbuf is not None:      # the bias gradient sums the large grid
                    call("lvae_colsum", gyn.data_ptr(), None, gbbuf.data_ptr(), B, Ho * Wo, N, _dt(gyn), _stream())
            elif not spec.transposed:
                stats["cc_wgrad"] += 1
                call("lvae_conv2d_wgrad", xn.data_ptr(), _p(x2n), gyn.data_ptr(), None, _p(out_scale),
                     gwbuf.data_ptr(), _p(gbbuf), B, Hi, Wi, C1, C2, Ho, Wo, N, spec.k, spec.k, spec.stride,
                     spec.pad, _dt(xn), _stream())
            else:
                # roles swap: "input" = dy (scaled), "output grad" = x; result is (Cin, Cout, k, k)
                stats["cc_wgrad"] += 1
                call("lvae_conv2d_wgrad", gyn.data_ptr(), None, xn.data_ptr(), _p(out_scale), None,
                     gwbuf.data_ptr(), None, B, Ho, Wo, N, 0, Hi, Wi, C1, spec.k, spec.k, spec.stride, spec.pad,
                     _dt(xn), _stream())
                if gbbuf is not None:
                    call("lvae_colsum", gyn.data_ptr(), _p(out_scale), gbbuf.data_ptr(), B, Ho * Wo, N, _dt(gyn), _stream())
        gw = None if sunk else gwbuf
        gb = None if (bsunk or gbbuf is None) else gbbuf
    return gx, gx2, gw, gb


class Conv2dFn(Function):
    """y = (conv(cat(x, x2)) + bias) * out_scale[b, c] + res   (Conv2d or ConvTranspose2d)."""

    @staticmethod
    def forward(ctx, x, x2, weight, bias, out_scale, res, spec: ConvSpec, stats_bn=None, x_lowp=None):
        _require_cuda(x)
        # x_lowp: the kernel's actual operand when the caller already holds a bf16, channel-padded copy of x (the stochastic
        # kernel writes z both as fp32 and as the 64-channel bf16 operand of conv_out); x itself then only carries the autograd
        # edge, and the data gradient comes back in x's own shape and dtype (fp32 epilogue): no pad / slice / cast passes
        window = None
        xv = x.permute(0, 2, 3, 1)
        if (x_lowp is None and x2 is None and res is None and out_scale is None and not torch.is_grad_enabled()
                and not xv.is_contiguous() and spec.cout == 1 and spec.k == 3 and spec.stride == 1 and spec.pad == 1
                and not spec.transposed and xv.dtype == torch.bfloat16 and xv.shape[3] == 64 == spec.cin
                and xv.stride(3) == 1 and xv.stride(2) == 64):
            # a cropped view of an NHWC activation (ops.crop under no_grad): the narrow head conv reads the window in place
            xn, window = xv, (xv.stride(1), xv.stride(0))
        else:
            xn = nhwc(x_lowp) if x_lowp is not None else nhwc(x)
        x2n = nhwc(x2) if x2 is not None else None
        resn = nhwc(res) if res is not None else None
        if out_scale is not None:
            out_scale = out_scale.reshape(xn.shape[0], spec.cout)
        spec._last_stats = None
        if stats_bn is not None and stats_bn.training and stats_bn.num_features == spec.cout == 64:
            # the consumer is a BatchNorm in train mode: its statistics ride in this conv's epilogue when the tcgen05 path runs
            acc = bn_scratch(stats_bn, xn.device)[0]
            _bn_clean(stats_bn, acc, "fwd")
            y, fused = conv_forward_raw(spec, xn, x2n, weight, bias, out_scale, resn, stats_acc=acc)
            if fused:
                spec._last_stats = (acc, y.shape[0] * y.shape[1] * y.shape[2], _bn_epoch[0])
        else:
            y = conv_forward_raw(spec, xn, x2n, weight, bias, out_scale, resn, window=window)
        ctx.spec = spec
        ctx.save_for_backward(xn, x2n, weight, bias, out_scale)
        ctx.has_res = res is not None
        return as_nchw(y)

    @staticmethod
    def backward(ctx, gy):
        spec = ctx.spec
        xn, x2n, weight, bias, out_scale = ctx.saved_tensors
        need_x = ctx.needs_input_grad[0] or (x2n is not None and ctx.needs_input_grad[1])
        gx, gx2, gw, gb = conv_backward_raw(spec, xn, x2n, weight, bias, out_scale, nhwc(gy), need_x,
                                            ctx.needs_input_grad[2], ctx.needs_input_grad[3])
        gres = gy if ctx.has_res and ctx.needs_input_grad[5] else None
        return (as_nchw(gx) if gx is not None else None, as_nchw(gx2) if gx2 is not None else None, gw, gb, None,
                gres, None, None, None)


def conv2d(x, weight, bias, spec: ConvSpec, x2=None, out_scale=None, res=None, stats_bn=None, x_lowp=None):
    """stats_bn: the train-mode BatchNorm2d that consumes the output next (its statistics are then accumulated by this
    conv's epilogue and handed over through the output tensor, like a gated block does for its successor)."""
    out = Conv2dFn.apply(x, x2, weight, bias, out_scale, res, spec, stats_bn, x_lowp)
    if stats_bn is not None and getattr(spec, "_last_stats", None) is not None:
        out._lvae_stats = spec._last_stats
        spec._last_stats = None
    return out


# --------------------------------------------------------------------------- BatchNorm (+ nonlinearity)
class BnActFn(Function):
    """y = act(batch_norm(x)); bn may be absent (plain activation).  Running statistics and
    num_batches_tracked are updated on the device in train mode."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, nbt, acc, training, momentum, eps, act, out_dtype):
        _require_cuda(x)
        xn = nhwc(x)
        B, H, W, C = xn.shape
        Pn = B * H * W
        y = torch.empty((B, H, W, C), dtype=out_dtype or xn.dtype, device=xn.device)
        mean = rstd = None
        if gamma is not None:
            stats = torch.empty((2, C), dtype=torch.float32, device=xn.device)
            mean, rstd = stats[0], stats[1]
            if training:
                call("lvae_bn_stats", xn.data_ptr(), acc.data_ptr(), Pn, C, _dt(xn), _stream())
                call("lvae_bn_finalize", acc.data_ptr(), mean.data_ptr(), rstd.data_ptr(), _p(running_mean),
                     _p(running_var), _p(nbt), Pn, C, float(momentum), float(eps), _stream())
            else:
                call("lvae_bn_eval_prepare", running_mean.data_ptr(), running_var.data_ptr(), mean.data_ptr(),
                     rstd.data_ptr(), C, float(eps), _stream())
        call("lvae_bn_act_fwd", xn.data_ptr(), y.data_ptr(), _p(mean), _p(rstd), _p(gamma), _p(beta), Pn, C, act,
             _dt(xn), _dt(y), _stream())
        ctx.save_for_backward(xn, mean, rstd, gamma, beta)
        ctx.acc, ctx.training, ctx.act = acc, training, act
        return as_nchw(y)

    @staticmethod
    def backward(ctx, gy):
        grad_site()
        xn, mean, rstd, gamma, beta = ctx.saved_tensors
        gyn = nhwc(gy)
        if gyn.dtype != xn.dtype:
            gyn = gyn.to(xn.dtype)
        B, H, W, C = xn.shape
        Pn = B * H * W
        gx = torch.empty_like(xn)
        gg = gb = None
        gsunk = bsunk = True
        if gamma is not None:
            gg, gsunk = _param_grad_buffer(gamma)
            gb, bsunk = _param_grad_buffer(beta)
        call("lvae_bn_act_bwd", gyn.data_ptr(), xn.data_ptr(), gx.data_ptr(), _p(mean), _p(rstd), _p(gamma), _p(beta),
             _p(ctx.acc), _p(gg), _p(gb), Pn, C, ctx.act, 1 if ctx.training else 0, _dt(xn), _stream())
        return (as_nchw(gx), None if gsunk else gg, None if bsunk else gb, None, None, None, None, None, None, None,
                None, None)


def bn_act(x, bn, act_id: int, out_dtype=None):
    """bn: our BatchNorm2d module or None."""
    if bn is None:
        return BnActFn.apply(x, None, None, None, None, None, None, False, 0.0, 0.0, act_id, out_dtype)
    training = bn.training or (bn.running_mean is None)
    return BnActFn.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var,
                         bn.num_batches_tracked if training else None, bn.stat_acc(x.device), training,
                         bn.momentum if bn.momentum is not None else 0.1, bn.eps, act_id, out_dtype)


# --------------------------------------------------------------------------- BatchNorm scratch arena
BN_STRIPES = 8
_bn_epoch = [0]
_whole_block = [True]
_gate_keep_h = [True]     # set per call by residual_block(): autograd.Function.forward always runs with grad mode off
# Fused paths of the gated blocks.  Always on: they are flags only so that tests/test_conv_gate_gpu.py and
# tests/test_block_stack_fusion_gpu.py can turn them off for their reference runs.
# _gate_chain: conv2 + gate conv + gate as ONE launch, the 1x1 GEMM reading the staged conv2 tile (lvae_conv_gate_tc; on a
# B200 in round 2: bit-identical tensors, 17.41 -> 16.71 ms per CIFAR-15 step).  _eval_bn_pre / _eval_bn_fold: eval-mode
# BatchNorm1 on conv1's operand path / BatchNorm2 folded into conv1's epilogue.  _stack_fusion: see below.
_gate_chain = [True]
_eval_bn_pre = [True]
_eval_bn_fold = [True]
_stack_fusion = [True]


def _conv_gate_chain(a2, w2p, bias2, mask2, wgp, gbias, xn, gact, stats_acc, keep):
    """lvae_conv_gate_tc: returns (c2, h, out); c2 and h are None when nothing will run backward (keep = False)."""
    B, H, W, _ = a2.shape
    out = torch.empty_like(xn)
    c2 = torch.empty_like(a2) if keep else None
    h = torch.empty((B, H, W, 128), dtype=torch.bfloat16, device=a2.device) if keep else None
    call("lvae_conv_gate_tc", a2.data_ptr(), w2p.data_ptr(), _p(bias2), _p(mask2), wgp.data_ptr(), _p(gbias), xn.data_ptr(),
         _p(c2), _p(h), out.data_ptr(), _p(stats_acc), B, H, W, int(gact), _stream())
    return c2, h, out


def set_whole_block(flag: bool) -> None:
    """Run default residual blocks as one autograd node with the hand-scheduled backward (default) or op by op."""
    _whole_block[0] = bool(flag)


def whole_block_enabled() -> bool:
    return _whole_block[0]



def new_forward_epoch() -> int:
    """A model zeroed its BatchNorm scratch arena: accumulators stamped with an older epoch are clean again."""
    check_no_pending_bn1()
    _bn_epoch[0] += 1
    return _bn_epoch[0]


# Cross-block fusion of the backward pass: inside a stack of directly adjacent gated residual blocks (models/lvae_layers.py
# _BlockStack) the LAST launch of block k's backward (BatchNorm1-backward apply + residual gradient -> dx) and the FIRST launch
# of block k-1's backward (gate backward on that very dx) are two elementwise passes over the same pixels.  Block k hands its
# apply over instead of launching it (keyed by the storage of the dx tensor it returns); block k-1 runs both as one kernel
# (lvae_bn_act_bwd2_gate).  Only when the stack guarantees that block k is the sole consumer of block k-1's output -- the
# gradient then reaches block k-1 unaccumulated, as the same tensor -- and only with engine-owned gradient sinks.
_private_out = [False]
_defer_bn1_next = [False]
_pending_bn1 = {}


def mark_block_output_private(flag: bool = True) -> None:
    """Called by the block stack right before it runs a block whose output is consumed by the next gated block only."""
    _private_out[0] = bool(flag) and _stack_fusion[0]


def check_no_pending_bn1() -> None:
    if _pending_bn1:
        n = len(_pending_bn1)
        _pending_bn1.clear()
        raise RuntimeError("lvae_b200: %d deferred BatchNorm-backward apply pass(es) were never picked up by the preceding "
                           "block's backward: their input gradients were not computed (cross-block fusion, ops._stack_fusion)" % n)


def bn_scratch(bn, device):
    """(3, 8, 2, C) float64 scratch of one BatchNorm2d: [0] forward sum / sum-of-squares, [1] backward sums, [2] statistics
    of the output of the residual block this BatchNorm opens; each 8-way striped (see csrc/elementwise.cu).  Clean
    (all zero) at first use in a forward epoch when it lives in a model arena; otherwise zeroed on demand."""
    acc = getattr(bn, "_lvae_scratch", None)
    if acc is None or acc.device != device:
        acc = torch.zeros((3, BN_STRIPES, 2, bn.num_features), dtype=torch.float64, device=device)
        bn._lvae_scratch = acc
        bn._lvae_scratch_owned = True
        bn._lvae_epoch_fwd = bn._lvae_epoch_bwd = -1
    return acc


def _bn_clean(bn, acc_rows, which: str):
    """Make sure the accumulator rows are zero before accumulating into them."""
    attr = "_lvae_epoch_" + which
    arena_clean = (not getattr(bn, "_lvae_scratch_owned", True)) and getattr(bn, attr, -1) != _bn_epoch[0]
    if not arena_clean:
        acc_rows.zero_()
    setattr(bn, attr, _bn_epoch[0])


class ResidualBlockFn(Function):
    """One whole ResidualBlock of type 'bacdbacd' or 'bacdbac' (lib/nn.py:62-99), gated (+ GateLayer2d :108-126) or not,
    with a hand-made backward schedule.  mask1 / mask2 are the Dropout2d masks behind conv1 / conv2 (either may be None).
    Gated:
        forward : [stats] BN1+act -> conv1 (*mask1) -> stats, BN2+act -> conv2 (*mask2) -> 1x1 gate conv ->
                  act(a)*sigmoid(b) + x  (+ statistics of the output for the next block's BN1)
        backward: gate' -> 1x1 dgrad (*mask2 in its epilogue) / wgrad -> conv2 dgrad / wgrad -> BN2' (*mask1 fused)
                  -> conv1 dgrad / wgrad -> BN1' (+ residual gradient fused)
    Ungated (gate conv None): conv2 (*mask2) + x in one epilogue, which also accumulates the output statistics; backward
        gout * mask2 -> conv2 dgrad / wgrad -> BN2' (*mask1 fused) -> conv1 dgrad / wgrad -> BN1' (+ residual gradient fused)
    Dropout2d masks are folded into neighbouring kernels' epilogues and BatchNorm needs no finalize / parameter kernels."""

    @staticmethod
    def forward(ctx, x, g1, b1, w1, cb1, g2, b2, w2, cb2, wg, gbias, m1, m2, blk, x_stats, training):
        _require_cuda(x)
        xn = nhwc(x)
        B, H, W, C = xn.shape
        Pn, dev, dt = B * H * W, xn.device, _dt(xn)
        bn1, bn2, conv1, conv2, gconv, act, gact = blk
        sc1, sc2 = bn_scratch(bn1, dev), bn_scratch(bn2, dev)
        saves = torch.empty((2, 2, C), dtype=torch.float32, device=dev)

        def bn_fwd(inp, bn, sc, save, gamma, beta, given_acc=None):
            acc = None
            if training:
                if given_acc is not None:
                    acc = given_acc
                else:
                    acc = sc[0]
                    _bn_clean(bn, acc, "fwd")
                    call("lvae_bn_stats", inp.data_ptr(), acc.data_ptr(), Pn, C, dt, _stream())
            out = torch.empty_like(inp)
            call("lvae_bn_act_fwd2", inp.data_ptr(), out.data_ptr(), _p(acc), gamma.data_ptr(), beta.data_ptr(),
                 save.data_ptr(), _p(bn.running_mean), _p(bn.running_var), _p(bn.num_batches_tracked) if training else None,
                 Pn, C, act, 1 if training else 0, float(bn.momentum if bn.momentum is not None else 0.1), float(bn.eps),
                 dt, dt, _stream())
            return out

        acc2 = None
        # eval mode under no_grad (the IW evaluator's sample passes): BatchNorm2 is a fixed per-channel affine map, so it rides
        # with the activation in conv1's epilogue -- one launch and one read + write of the tensor less per block
        fold2 = (_eval_bn_fold[0] and not training and not _gate_keep_h[0] and C == 64 and m1 is None
                 and xn.dtype == torch.bfloat16 and bn2.running_mean is not None and conv1.spec.cout == 64
                 and not conv1.spec.out_fp32 and conv1.spec.tc_forward_ok(xn, None))
        # ... and BatchNorm1 + activation on conv1's operand tile as it lands in shared memory (halo tiles: 16x16 and larger)
        pre1 = fold2 and _eval_bn_pre[0] and conv1.spec.k == 3 and H % 16 == 0 and W % 8 == 0 and bn1.running_mean is not None
        a1 = None if pre1 else bn_fwd(xn, bn1, sc1, saves[0], g1, b1, x_stats)
        if fold2:
            stats["tc_fwd"] += 1
            stats["bn_fold"] = stats.get("bn_fold", 0) + 1
            stats["bn_pre"] = stats.get("bn_pre", 0) + (1 if pre1 else 0)
            y1 = None
            a2 = _conv_tc(xn if pre1 else a1, None, conv1.spec.pack_tc_fwd.get(w1, torch.bfloat16), cb1, None, None, 64,
                          conv1.spec.k, False, False,
                          fold=(g2, b2, bn2.running_mean, bn2.running_var, bn2.eps, act,
                                (g1, b1, bn1.running_mean, bn1.running_var, bn1.eps) if pre1 else None))
        elif training and C == 64:
            acc2 = sc2[0]
            _bn_clean(bn2, acc2, "fwd")
            y1, fused = conv_forward_raw(conv1.spec, a1, None, w1, cb1, m1, None, stats_acc=acc2)   # BN2 statistics in the epilogue
            if not fused:
                call("lvae_bn_stats", y1.data_ptr(), acc2.data_ptr(), Pn, C, dt, _stream())
        else:
            y1 = conv_forward_raw(conv1.spec, a1, None, w1, cb1, m1, None)
        if not fold2:
            a2 = bn_fwd(y1, bn2, sc2, saves[1], g2, b2, acc2)
        out_stats = y2 = h = None
        if gconv is None:
            # ungated: out = conv2(a2) * mask2 + x, the residual added in the TMA-store epilogue; in training the same epilogue
            # accumulates the statistics of out for the next block's BN1 (bf16, 64 channels: free there -- elsewhere the
            # consumer's BatchNorm computes them)
            if (training and C == 64 and xn.dtype == torch.bfloat16 and not conv2.spec.out_fp32
                    and conv2.spec.tc_forward_ok(a2, None)):
                out_stats = sc1[2]
                _bn_clean(bn1, out_stats, "out")
                out, fused = conv_forward_raw(conv2.spec, a2, None, w2, cb2, m2, xn, stats_acc=out_stats)
                if not fused:
                    call("lvae_bn_stats", out.data_ptr(), out_stats.data_ptr(), Pn, C, dt, _stream())
            else:
                out = conv_forward_raw(conv2.spec, a2, None, w2, cb2, m2, xn)
        else:
            gspec = gconv.spec
            # conv2, the 1x1 gate conv and the gate itself as one launch (csrc/conv_gate_tcgen05.cu)
            chain = (_gate_chain[0] and C == 64 and gspec.cout == 128 and gspec.k == 1 and conv2.spec.k == 3 and conv2.spec.cout == 64
                     and xn.dtype == torch.bfloat16 and not gspec.out_fp32 and not conv2.spec.out_fp32
                     and conv2.spec.tc_forward_ok(a2, None) and gspec.tc_forward_ok(a2, None)
                     and (m2 is None or (m2.dtype == torch.float32 and m2.is_contiguous())))
            if not chain:
                y2 = conv_forward_raw(conv2.spec, a2, None, w2, cb2, m2, None)
            if training and 256 % (C // 4) == 0:
                out_stats = sc1[2]                        # statistics of this block's output, for the next block's BN1
                _bn_clean(bn1, out_stats, "out")
            if chain:
                stats["tc_fwd"] += 2
                stats["gate_chain"] = stats.get("gate_chain", 0) + 1
                y2, h, out = _conv_gate_chain(a2, conv2.spec.pack_tc_fwd.get(w2, torch.bfloat16), cb2, m2,
                                              gspec.pack_tc_fwd.get(wg, torch.bfloat16), gbias, xn, gact, out_stats, _gate_keep_h[0])
            elif (C == 64 and gspec.cout == 128 and xn.dtype == torch.bfloat16 and not gspec.out_fp32
                    and gspec.tc_forward_ok(y2, None)):
                # gate, residual add and the output statistics ride in the epilogue of the 1x1 gate conv
                stats["tc_fwd"] += 1
                stats["gate_fused"] = stats.get("gate_fused", 0) + 1
                h, out = _conv_tc(y2, None, gspec.pack_tc_fwd.get(wg, torch.bfloat16), gbias, None, None, 128, gspec.k, False, False,
                                  stats_acc=out_stats, gate=(xn, gact))
            else:
                h = conv_forward_raw(gspec, y2, None, wg, gbias, None, None)
                out = torch.empty_like(xn)
                if out_stats is not None:
                    call("lvae_gate_fwd_stats", h.data_ptr(), xn.data_ptr(), out.data_ptr(), out_stats.data_ptr(), Pn, C, gact, dt, _stream())
                else:
                    call("lvae_gate_fwd", h.data_ptr(), xn.data_ptr(), out.data_ptr(), Pn, C, gact, dt, _stream())
        ctx.save_for_backward(xn, a1, y1, a2, y2, h, saves, g1, b1, w1, cb1, g2, b2, w2, cb2, wg, gbias, m1, m2)
        ctx.blk, ctx.training = blk, training
        ctx.defer_bn1 = bool(_defer_bn1_next[0])
        _defer_bn1_next[0] = False
        blk[0]._lvae_last_out_stats = (out_stats, Pn, _bn_epoch[0]) if out_stats is not None else None
        return as_nchw(out)

    @staticmethod
    def backward(ctx, gout):
        xn, a1, y1, a2, y2, h, saves, g1, b1, w1, cb1, g2, b2, w2, cb2, wg, gbias, m1, m2 = ctx.saved_tensors
        bn1, bn2, conv1, conv2, gconv, act, gact = ctx.blk
        training = ctx.training
        B, H, W, C = xn.shape
        Pn, dev, dt = B * H * W, xn.device, _dt(xn)
        gn = nhwc(gout)
        if gn.dtype != xn.dtype:
            gn = gn.to(xn.dtype)
        ng = ctx.needs_input_grad
        if gconv is None:
            # ungated: the gradient wrt conv2's raw output is gout * mask2 (applied by conv_backward_raw); never handed a
            # deferred BatchNorm1 apply (residual_block marks only gated blocks' outputs private)
            dy2, scale2, gwg, ggb = gn, m2, None, None
        else:
            gsp = gconv.spec
            # gate
            dh = torch.empty_like(h)
            pend = _pending_bn1.pop(gn.data_ptr(), None)
            if pend is not None:
                # the consumer block deferred its BatchNorm1-backward apply: gn is its (still uncomputed) dx -- one pass writes
                # dx into gn and this block's gate gradient dh
                assert pend["shape"] == tuple(gn.shape) and gn.dtype == torch.bfloat16 and h.dtype == torch.bfloat16
                grad_site()
                pdg, _ = _param_grad_buffer(pend["gamma"])
                pdb, _ = _param_grad_buffer(pend["beta"])
                stats["bn1_gate_fused"] = stats.get("bn1_gate_fused", 0) + 1
                call("lvae_bn_act_bwd2_gate", pend["dy"].data_ptr(), pend["x"].data_ptr(), gn.data_ptr(), pend["save"].data_ptr(),
                     pend["gamma"].data_ptr(), pend["beta"].data_ptr(), pend["acc"].data_ptr(), pdg.data_ptr(), pdb.data_ptr(), None,
                     pend["add"].data_ptr(), h.data_ptr(), dh.data_ptr(), Pn, H * W, C, pend["act"], gact,
                     1 if pend["training"] else 0, _stream())
            else:
                call("lvae_gate_bwd", gn.data_ptr(), h.data_ptr(), dh.data_ptr(), Pn, C, gact, dt, _stream())
            # 1x1 gate conv: dgrad carries conv2's Dropout2d mask in its epilogue -> gradient wrt conv2's raw output
            dy2, _, gwg, ggb = conv_backward_raw(gsp, y2, None, wg, gbias, None, dh, True, ng[9], ng[10], dx_scale=m2)
            scale2 = None
        sc1b, sc2b = bn_scratch(bn1, dev), bn_scratch(bn2, dev)
        acc1b, acc2b = sc1b[1], sc2b[1]
        _bn_clean(bn1, acc1b, "bwd")
        _bn_clean(bn2, acc2b, "bwd")
        # conv2 (dy2 is masked, or scale2 masks it); its dgrad epilogue also accumulates BN2's backward sums
        da2, _, gw2, gcb2 = conv_backward_raw(conv2.spec, a2, None, w2, cb2, scale2, dy2, True, ng[7], ng[8],
                                              bnb=(y1, saves[1], g2, b2, acc2b, act) if C == 64 else None)
        fused2 = conv_backward_raw.last_fused

        def bn_bwd(dy, xin, bn, acc, save, gamma, beta, post_scale, add, skip_reduce):
            grad_site()
            dgam, gsunk = _param_grad_buffer(gamma)
            dbet, bsunk = _param_grad_buffer(beta)
            dxo = torch.empty_like(xin)
            call("lvae_bn_act_bwd2", dy.data_ptr(), xin.data_ptr(), dxo.data_ptr(), save.data_ptr(), gamma.data_ptr(),
                 beta.data_ptr(), acc.data_ptr(), dgam.data_ptr(), dbet.data_ptr(), _p(post_scale), _p(add), Pn, H * W, C,
                 act, 1 if training else 0, dt, 1 if skip_reduce else 0, _stream())
            return dxo, (None if gsunk else dgam), (None if bsunk else dbet)

        # BN2 + act backward, conv1's mask fused -> gradient wrt conv1's raw output
        dy1, gg2, gb2 = bn_bwd(da2, y1, bn2, acc2b, saves[1], g2, b2, m1, None, fused2)
        da1, _, gw1, gcb1 = conv_backward_raw(conv1.spec, a1, None, w1, cb1, None, dy1, True, ng[3], ng[4],
                                              bnb=(xn, saves[0], g1, b1, acc1b, act) if C == 64 else None)
        fused1 = conv_backward_raw.last_fused
        # BN1 + act backward, residual gradient fused
        if (ctx.defer_bn1 and fused1 and xn.dtype == torch.bfloat16 and C % 8 == 0 and grad_sink(g1) is not None
                and grad_sink(b1) is not None and gn.dtype == torch.bfloat16):
            # handed over to the backward of the block that produced xn (see _pending_bn1): dx is returned uncomputed
            dx = torch.empty_like(xn)
            _pending_bn1[dx.data_ptr()] = dict(dy=da1, x=xn, add=gn, save=saves[0], gamma=g1, beta=b1, acc=acc1b, act=act,
                                               training=training, shape=tuple(xn.shape), keep=dx)
            return (as_nchw(dx), None, None, gw1, gcb1, gg2, gb2, gw2, gcb2, gwg, ggb, None, None, None, None, None)
        dx, gg1, gb1 = bn_bwd(da1, xn, bn1, acc1b, saves[0], g1, b1, None, gn, fused1)
        return (as_nchw(dx), gg1, gb1, gw1, gcb1, gg2, gb2, gw2, gcb2, gwg, ggb, None, None, None, None, None)


def residual_block(x, bn1, conv1, drop1, bn2, conv2, drop2, gate_layer, act_id):
    """A 'bacdbacd' / 'bacdbac' residual block as one autograd node (ResidualBlockFn).  drop1 / drop2: the Dropout2d modules
    behind conv1 / conv2, or None; gate_layer: the GateLayer2d of a gated block, None for an ungated one."""
    training = bn1.training
    # statistics of x computed by the kernel that produced it (previous block's last epilogue), if still valid
    x_stats = None
    st = getattr(x, "_lvae_stats", None)
    if training and st is not None and st[2] == _bn_epoch[0] and st[1] == x.shape[0] * x.shape[2] * x.shape[3]:
        x_stats = st[0]
    m1 = drop1.mask(x) if drop1 is not None else None
    m2 = drop2.mask(x) if drop2 is not None else None
    if m1 is not None:
        m1 = m1.reshape(x.shape[0], -1)
    if m2 is not None:
        m2 = m2.reshape(x.shape[0], -1)
    gconv = gate_layer.conv if gate_layer is not None else None
    blk = (bn1, bn2, conv1, conv2, gconv, act_id, getattr(gate_layer.nonlin, "act_id", 0) if gate_layer is not None else 0)
    _gate_keep_h[0] = torch.is_grad_enabled()
    # this block's output goes to the next block of the stack and nowhere else; only a gated block's backward picks the next
    # block's deferred BatchNorm1 apply up (lvae_bn_act_bwd2_gate), so only its output is marked private
    private = _private_out[0] and gconv is not None
    _private_out[0] = False
    # x is such a private output of the previous block: this block's BatchNorm1-backward apply may be handed over to it
    _defer_bn1_next[0] = bool(getattr(x, "_lvae_private", False)) and training and torch.is_grad_enabled() and x.requires_grad
    try:
        out = ResidualBlockFn.apply(x, bn1.weight, bn1.bias, conv1.weight, conv1.bias, bn2.weight, bn2.bias, conv2.weight,
                                    conv2.bias, gconv.weight if gconv is not None else None,
                                    gconv.bias if gconv is not None else None, m1, m2, blk, x_stats, training)
    finally:
        _defer_bn1_next[0] = False            # never leaks into another block if the forward raised before reading it
    stats["block_node"] = stats.get("block_node", 0) + 1
    if training and bn1._lvae_last_out_stats is not None:
        out._lvae_stats = bn1._lvae_last_out_stats
    if private and training and out.dtype == torch.bfloat16:
        out._lvae_private = True
    return out


# --------------------------------------------------------------------------- gate (+ residual)
class GateFn(Function):
    @staticmethod
    def forward(ctx, h, res, act):
        hn = nhwc(h)
        B, H, W, C2 = hn.shape
        C = C2 // 2
        resn = nhwc(res) if res is not None else None
        out = torch.empty((B, H, W, C), dtype=hn.dtype, device=hn.device)
        call("lvae_gate_fwd", hn.data_ptr(), _p(resn), out.data_ptr(), B * H * W, C, act, _dt(hn), _stream())
        ctx.save_for_backward(hn)
        ctx.act, ctx.has_res = act, res is not None
        return as_nchw(out)

    @staticmethod
    def backward(ctx, g):
        (hn,) = ctx.saved_tensors
        gn = nhwc(g)
        B, H, W, C2 = hn.shape
        dh = torch.empty_like(hn)
        call("lvae_gate_bwd", gn.data_ptr(), hn.data_ptr(), dh.data_ptr(), B * H * W, C2 // 2, ctx.act, _dt(hn), _stream())
        return as_nchw(dh), (g if ctx.has_res else None), None


def gate(h, res, act_id):
    return GateFn.apply(h, res, act_id)


# --------------------------------------------------------------------------- resampling helpers
class Upsample2xFn(Function):
    @staticmethod
    def forward(ctx, x):
        xn = nhwc(x)
        B, H, W, C = xn.shape
        y = torch.empty((B, 2 * H, 2 * W, C), dtype=xn.dtype, device=xn.device)
        call("lvae_upsample2x_fwd", xn.data_ptr(), y.data_ptr(), B, H, W, C, _dt(xn), _stream())
        ctx.shape = (B, H, W, C)
        return as_nchw(y)

    @staticmethod
    def backward(ctx, g):
        gn = nhwc(g)
        B, H, W, C = ctx.shape
        dx = torch.empty((B, H, W, C), dtype=gn.dtype, device=gn.device)
        call("lvae_upsample2x_bwd", gn.data_ptr(), dx.data_ptr(), B, H, W, C, _dt(gn), _stream())
        return as_nchw(dx)


def upsample2x(x):
    return Upsample2xFn.apply(x)


def _copy_window(src, dst, B, C, Hs, Ws, Hd, Wd, sy0, sx0, dy0, dx0, h, w, src_nchw, dst_nchw):
    call("lvae_copy_window", src.data_ptr(), dst.data_ptr(), B, C, Hs, Ws, Hd, Wd, sy0, sx0, dy0, dx0, h, w,
         1 if src_nchw else 0, 1 if dst_nchw else 0, _dt(src), _dt(dst), _stream())


def pad_image(x: torch.Tensor, size, out_dtype=torch.float32) -> torch.Tensor:
    """boilr pad_img_tensor on the *input image* (no gradient needed): NCHW user tensor ->
    zero-padded NHWC-physical activation (logical NCHW)."""
    _require_cuda(x)
    x = x.contiguous()
    if x.dtype != torch.float32:
        x = x.float()
    B, C, H, W = x.shape
    Hp, Wp = int(size[0]), int(size[1])
    dr, dc = Hp - H, Wp - W
    if dr < 0 or dc < 0:
        raise ValueError("trying to pad to a smaller size")
    if dr == 0 and dc == 0:
        y = torch.empty((B, Hp, Wp, C), dtype=out_dtype, device=x.device)
    else:
        y = torch.zeros((B, Hp, Wp, C), dtype=out_dtype, device=x.device)
    _copy_window(x, y, B, C, H, W, Hp, Wp, 0, 0, dr // 2, dc // 2, H, W, True, False)
    return as_nchw(y)


class CropFn(Function):
    """boilr crop_img_tensor (centred) on an NHWC-physical activation."""

    @staticmethod
    def forward(ctx, x, size):
        xn = nhwc(x)
        B, H, W, C = xn.shape
        h, w = int(size[0]), int(size[1])
        dr, dc = H - h, W - w
        if dr < 0 or dc < 0:
            raise ValueError("trying to crop to a larger size")
        y = torch.empty((B, h, w, C), dtype=xn.dtype, device=xn.device)
        _copy_window(xn, y, B, C, H, W, h, w, dr // 2, dc // 2, 0, 0, h, w, False, False)
        ctx.geom = (B, H, W, C, h, w, dr // 2, dc // 2)
        return as_nchw(y)

    @staticmethod
    def backward(ctx, g):
        B, H, W, C, h, w, y0, x0 = ctx.geom
        gn = nhwc(g)
        dx = torch.zeros((B, H, W, C), dtype=gn.dtype, device=gn.device)
        _copy_window(gn, dx, B, C, h, w, H, W, 0, 0, y0, x0, h, w, False, False)
        return as_nchw(dx), None


def crop(x, size):
    if tuple(x.shape[2:]) == tuple(int(s) for s in size):
        return x
    if not torch.is_grad_enabled() and x.is_cuda:
        # nothing runs backward (IW evaluator, sampling): the centred crop is a strided view of the NHWC buffer -- the Bernoulli
        # head's narrow conv reads the window in place, any other consumer makes it contiguous itself (ops.nhwc)
        xn = x.permute(0, 2, 3, 1)
        h, w = int(size[0]), int(size[1])
        dr, dc = xn.shape[1] - h, xn.shape[2] - w
        if dr < 0 or dc < 0:
            raise ValueError("trying to crop to a larger size")
        if xn.is_contiguous():
            return xn[:, dr // 2:dr // 2 + h, dc // 2:dc // 2 + w, :].permute(0, 3, 1, 2)
    return CropFn.apply(x, size)


# --------------------------------------------------------------------------- stochastic block core
_stoch_ws = {}


def _stoch_workspace(batch: int, device) -> torch.Tensor:
    """Zero-initialised scratch that lets lvae_stoch_fwd split one sample over several CTAs (stream-ordered reuse)."""
    key = (device, torch.cuda.current_stream().cuda_stream, batch)      # one buffer per batch size: its tickets stay zero
    ws = _stoch_ws.get(key)
    if ws is None:
        ws = torch.zeros(int(_capi.lib().lvae_stoch_ws_bytes(batch)), dtype=torch.uint8, device=device)
        _stoch_ws[key] = ws
    return ws


# fp32 gradient buffer (data_ptr) -> (the fp32 tensor itself, its bf16 copy written by the producing kernel, the buffer's version).  The entry keeps the
# fp32 tensor alive, so the address cannot be handed to another tensor while the entry exists (and autograd, seeing a second
# reference, never accumulates into it in place); a gradient that autograd summed with another one is a new tensor and misses.
_lowp_grads: dict = {}


def _lowp_grad_put(g32: torch.Tensor, g16: torch.Tensor) -> None:
    if len(_lowp_grads) > 256:           # entries nobody collected (a consumer that needed no gradient)
        _lowp_grads.clear()
    _lowp_grads[g32.data_ptr()] = (g32, g16, g32._version)


def _lowp_grad_take(g32: torch.Tensor, dtype: torch.dtype):
    """The bf16 copy of this very gradient tensor, if its producer wrote one (else None)."""
    ent = _lowp_grads.pop(g32.data_ptr(), None)
    if ent is None:
        return None
    k, g16, version = ent
    # (an in-place write to the fp32 buffer after the copy was taken moves its version counter: the copy is stale)
    if g16.dtype != dtype or tuple(g16.shape) != tuple(g32.shape) or k.data_ptr() != g32.data_ptr() or g32._version != version:
        return None
    return g16


class StochasticFn(Function):
    """Everything between conv_in_* and conv_out of NormalStochasticBlock2d (lib/stochastic.py:45-96)."""

    @staticmethod
    def forward(ctx, q_params, p_params, eps, forced, use_mode, analytical, lowp_copy):
        _require_cuda(p_params)
        ctx.set_materialize_grads(False)         # unused outputs (z, kl_spatial, logp, logq ...) arrive as None, not as zero tensors
        pn = nhwc(p_params).float()
        qn = nhwc(q_params).float() if q_params is not None else None
        ref = qn if qn is not None else pn
        p_broadcast = pn.shape[0] == 1 and ref.shape[0] != 1
        B, H, W, Z2 = ref.shape
        Z, hw = Z2 // 2, H * W
        dev = ref.device
        epsn = nhwc(eps).float() if eps is not None else None
        forcedn = nhwc(forced).float() if forced is not None else None
        z = torch.empty((B, H, W, Z), dtype=torch.float32, device=dev)
        # bf16 copy of z for conv_out, zero-padded to 64 channels so that the conv runs on the tensor cores
        zp = 64 if (lowp_copy and Z < 64) else Z
        z_lp = torch.empty((B, H, W, zp), dtype=torch.bfloat16, device=dev) if lowp_copy else None
        kl_row, logp, logq_row = _take_kl_row(B, dev)
        if qn is not None:
            kl, logq = kl_row, logq_row
            kls = torch.empty((B, H, W), dtype=torch.float32, device=dev)
        else:
            kl = logq = kls = None
        need_rng = epsn is None and forcedn is None and not use_mode
        call("lvae_stoch_fwd", _p(qn), pn.data_ptr(), 1 if p_broadcast else 0, _p(epsn), _p(forcedn),
             rng_state(dev).data_ptr() if need_rng else None, next_stream_id() if need_rng else 0,
             z.data_ptr(), _p(z_lp), zp, _p(kl), _p(kls), logp.data_ptr(), _p(logq), B, hw, Z,
             1 if use_mode else 0, 1 if analytical else 0, _stoch_workspace(B, dev).data_ptr(), _stream())
        ctx.save_for_backward(qn, pn, z)
        ctx.meta = (B, hw, Z, p_broadcast, analytical, 0 if forced is not None else (2 if use_mode else 1))
        ctx.q_dtype = q_params.dtype if q_params is not None else None
        ctx.p_dtype = p_params.dtype
        ctx.lowp = bool(lowp_copy)
        zo = as_nchw(z)
        zlo = as_nchw(z_lp) if z_lp is not None else None
        if zlo is not None:
            ctx.mark_non_differentiable(zlo)      # conv_out takes it as a side operand; the gradient flows through z
        return zo, zlo, kl, kls, logp, logq

    @staticmethod
    def backward(ctx, g_z, g_zlp, g_kl, g_kls, g_logp, g_logq):
        qn, pn, z = ctx.saved_tensors
        if qn is None:
            raise RuntimeError("backward through prior sampling is not supported")
        B, hw, Z, p_broadcast, analytical, z_kind = ctx.meta
        gz = nhwc(g_z).float() if g_z is not None else None
        cg = lambda t: t.contiguous().float() if t is not None else None
        g_kl, g_kls, g_logp, g_logq = cg(g_kl), cg(g_kls), cg(g_logp), cg(g_logq)
        dq = torch.empty_like(qn)
        dp = torch.empty((B,) + tuple(qn.shape[1:]), dtype=torch.float32, device=qn.device)
        # bf16 pipeline: the kernel also writes bf16 copies of dq / dp, which the tensor-core data / weight gradients of conv_in_q /
        # conv_in_p pick up from _lowp_grads instead of casting the fp32 gradient autograd hands them (29 ATen launches per step)
        dq_lp = torch.empty(qn.shape, dtype=torch.bfloat16, device=qn.device) if ctx.lowp and 2 * Z == 64 else None
        dp_lp = torch.empty(qn.shape, dtype=torch.bfloat16, device=qn.device) if dq_lp is not None and not p_broadcast else None
        call("lvae_stoch_bwd_ex", qn.data_ptr(), pn.data_ptr(), 1 if p_broadcast else 0, z.data_ptr(), _p(gz), _p(g_kl),
             _p(g_logp), _p(g_logq), _p(g_kls), dq.data_ptr(), dp.data_ptr(), _p(dq_lp), _p(dp_lp), B, hw, Z,
             1 if analytical else 0, z_kind, _stream())
        if dq_lp is not None and ctx.q_dtype == torch.float32:
            _lowp_grad_put(dq, dq_lp)
        if dp_lp is not None and ctx.p_dtype == torch.float32:
            _lowp_grad_put(dp, dp_lp)
        if p_broadcast:
            dps = torch.empty_like(pn)
            call("lvae_sum_batch", dp.data_ptr(), dps.data_ptr(), B, dps.numel(), 0, _stream())
            dp = dps
        dq, dp = as_nchw(dq), as_nchw(dp)
        if ctx.q_dtype != torch.float32:
            dq = dq.to(ctx.q_dtype)
        if ctx.p_dtype != torch.float32:
            dp = dp.to(ctx.p_dtype)
        return dq, dp, None, None, None, None, None


def stochastic_core(q_params, p_params, eps=None, forced=None, use_mode=False, analytical=False, lowp_copy=False):
    return StochasticFn.apply(q_params, p_params, eps, forced, use_mode, analytical, lowp_copy)


class KLBookFn(Function):
    """Free bits and the KL / log p bookkeeping of LadderVAE.forward (models/lvae.py:192-198,301-302; boilr free_bits_kl)
    as ONE launch over the (L,B) matrices the stochastic kernels filled, with a one-launch backward.
    apply(free_bits, L, rows_or_None, kl_0 .. kl_{L-1}, logp_0 .. logp_{L-1}) -> (kl_sep, kl, kl_avg_layerwise, kl_loss, logp)."""

    @staticmethod
    def forward(ctx, free_bits, L, rows, *vecs):
        kls, lps = vecs[:L], vecs[L:]
        B = kls[0].shape[0]
        dev = kls[0].device
        # the vectors are the rows of the pass's (3,L,B) matrix when LadderVAE.topdown_pass reserved it; anything else
        # (blocks called on their own, a batch-size change mid-pass) is gathered first
        in_place = (rows is not None and rows.shape[1] == L and rows.shape[2] == B and
                    all(kls[i].data_ptr() == rows[0, i].data_ptr() and lps[i].data_ptr() == rows[1, i].data_ptr() for i in range(L)))
        if in_place:
            stats["kl_rows_in_place"] = stats.get("kl_rows_in_place", 0) + 1
            klm, lpm = rows[0], rows[1]
        else:
            klm = torch.stack([k.float() for k in kls]).contiguous()
            lpm = torch.stack([v.float() for v in lps]).contiguous()
        kl_sep = torch.empty((B,), dtype=torch.float32, device=dev)
        scal = torch.empty((3,), dtype=torch.float32, device=dev)
        avg = torch.empty((L,), dtype=torch.float32, device=dev)
        coef = torch.empty((L, B), dtype=torch.float32, device=dev)
        call("lvae_kl_bookkeeping", klm.data_ptr(), lpm.data_ptr(), L, B, float(free_bits), kl_sep.data_ptr(), scal.data_ptr(),
             avg.data_ptr(), coef.data_ptr(), _stream())
        ctx.save_for_backward(coef)
        ctx.L, ctx.B = L, B
        ctx.set_materialize_grads(False)
        return kl_sep, scal[0], avg, scal[1], scal[2]

    @staticmethod
    def backward(ctx, g_sep, g_kl, g_avg, g_loss, g_lp):
        (coef,) = ctx.saved_tensors
        L, B = ctx.L, ctx.B
        dev = coef.device
        parts = [g_kl, g_loss, g_lp]
        if all(p is None for p in parts):
            gs = torch.zeros((3,), dtype=torch.float32, device=dev)
        else:
            z = None
            cols = []
            for p in parts:
                if p is None:
                    if z is None:
                        z = torch.zeros((), dtype=torch.float32, device=dev)
                    cols.append(z)
                else:
                    cols.append(p.float().reshape(()))
            gs = torch.stack(cols)
        gk = torch.empty((L, B), dtype=torch.float32, device=dev)
        gl = torch.empty((L, B), dtype=torch.float32, device=dev) if g_lp is not None else None
        call("lvae_kl_bookkeeping_bwd", coef.data_ptr(), gs.data_ptr(), _p(g_sep.contiguous().float() if g_sep is not None else None),
             _p(g_avg.contiguous().float() if g_avg is not None else None), L, B, gk.data_ptr(), _p(gl), _stream())
        return (None, None, None) + tuple(gk[i] for i in range(L)) + tuple((gl[i] if gl is not None else None) for i in range(L))


def kl_bookkeeping(kl_list, logp_list, free_bits: float, rows=None):
    """-> dict(kl_sep (B,), kl, kl_avg_layerwise (L,), kl_loss, logp) from the per-layer (B,) vectors."""
    L = len(kl_list)
    kl_sep, kl, avg, loss, lp = KLBookFn.apply(float(free_bits), L, rows, *kl_list, *logp_list)
    return {"kl_sep": kl_sep, "kl": kl, "kl_avg_layerwise": avg, "kl_loss": loss, "logp": lp}


# --------------------------------------------------------------------------- likelihoods
class BernoulliFn(Function):
    """sigmoid + Bernoulli log-likelihood (lib/likelihoods.py:61-62,385-388). Returns (prob, ll)."""

    @staticmethod
    def forward(ctx, logits, x):
        ln = nhwc(logits).float()
        B, H, W, C = ln.shape
        prob = torch.empty_like(ln)
        ll = None
        xc = None
        if x is not None:
            xc = x.contiguous().float()
            assert tuple(xc.shape) == (B, C, H, W), "image shape %s vs params %s" % (tuple(xc.shape), (B, C, H, W))
            ll = torch.empty((B,), dtype=torch.float32, device=ln.device)
        call("lvae_bernoulli_fwd", ln.data_ptr(), _p(xc), prob.data_ptr(), _p(ll), B, H * W, C, _stream())
        ctx.save_for_backward(prob, xc)
        ctx.in_dtype = logits.dtype
        return as_nchw(prob), ll

    @staticmethod
    def backward(ctx, g_prob, g_ll):
        prob, xc = ctx.saved_tensors
        B, H, W, C = prob.shape
        if xc is None or g_ll is None:
            if g_prob is None:
                return None, None
            gp = nhwc(g_prob).float()
            return as_nchw(gp * prob * (1 - prob)).to(ctx.in_dtype), None
        gp = nhwc(g_prob).float() if g_prob is not None else None
        dl = torch.empty_like(prob)
        call("lvae_bernoulli_bwd", prob.data_ptr(), xc.data_ptr(), g_ll.contiguous().float().data_ptr(), _p(gp),
             dl.data_ptr(), B, H * W, C, _stream())
        out = as_nchw(dl)
        return (out if ctx.in_dtype == torch.float32 else out.to(ctx.in_dtype)), None


def bernoulli_loglik(logits, x):
    return BernoulliFn.apply(logits, x)


def bernoulli_sample(prob):
    pn = nhwc(prob).float()
    B, H, W, C = pn.shape
    out = torch.empty((B, C, H, W), dtype=torch.float32, device=pn.device)
    call("lvae_bernoulli_sample", pn.data_ptr(), out.data_ptr(), B, H * W, C, rng_state(pn.device).data_ptr(),
         next_stream_id(), _stream())
    return out


class DmolFn(Function):
    """-discretized_mix_logistic_loss(2x-1, l) (lib/likelihoods.py:226-230,291-382) -> ll (B,)."""

    @staticmethod
    def forward(ctx, l, x):
        ln = nhwc(l).float()
        B, H, W, C = ln.shape
        if C != 100:
            raise RuntimeError("discretized logistic mixture expects 100 parameter channels, got %d" % C)
        xc = x.contiguous().float()
        assert tuple(xc.shape) == (B, 3, H, W), "image shape %s vs params %s" % (tuple(xc.shape), (B, 3, H, W))
        ll = torch.zeros((B,), dtype=torch.float32, device=ln.device)
        call("lvae_dmol_fwd", ln.data_ptr(), xc.data_ptr(), ll.data_ptr(), B, H * W, _stream())
        ctx.save_for_backward(ln, xc)
        ctx.in_dtype = l.dtype
        return ll

    @staticmethod
    def backward(ctx, g_ll):
        ln, xc = ctx.saved_tensors
        B, H, W, C = ln.shape
        dl = torch.empty_like(ln)
        call("lvae_dmol_bwd", ln.data_ptr(), xc.data_ptr(), g_ll.contiguous().float().data_ptr(), dl.data_ptr(), None, B,
             H * W, _stream())
        out = as_nchw(dl)
        return (out if ctx.in_dtype == torch.float32 else out.to(ctx.in_dtype)), None


def dmol_loglik(l, x):
    return DmolFn.apply(l, x)


class DmolHeadFn(Function):
    """parameter_net conv (64 or 128 -> 100, 3x3) + mixture-of-logistics log-likelihood as ONE autograd node on the bf16
    tensor-core path: the likelihood backward writes its gradient directly as the zero-padded bf16 operand
    (B,H,W,128) of the head conv's tcgen05 dgrad / wgrad (no fp32 round trip, no CUDA-core fallback for N = 100)."""

    @staticmethod
    def forward(ctx, h, weight, bias, x, spec):
        ctx.set_materialize_grads(False)
        hn = nhwc(h)
        B, H, W, C = hn.shape
        wp = spec.pack_tc_fwd.get(weight, torch.bfloat16)
        stats["tc_fwd"] += 1
        l = _conv_tc(hn, None, wp, bias, None, None, spec.cout, spec.k, False, True)      # fp32 (B,H,W,100)
        xc = x.contiguous().float()
        ll = torch.zeros((B,), dtype=torch.float32, device=hn.device)
        call("lvae_dmol_fwd", l.data_ptr(), xc.data_ptr(), ll.data_ptr(), B, H * W, _stream())
        ctx.save_for_backward(hn, l, xc, weight, bias)
        ctx.spec = spec
        lo = as_nchw(l)
        ctx.mark_non_differentiable(lo)
        return ll, lo

    @staticmethod
    def backward(ctx, g_ll, _g_l):
        grad_site()
        hn, l, xc, weight, bias = ctx.saved_tensors
        spec = ctx.spec
        if g_ll is None:
            if _g_l is not None:
                raise RuntimeError("DmolHeadFn: gradients through the raw likelihood parameters are not supported")
            return None, None, None, None, None
        B, H, W, C = hn.shape
        dl = torch.empty((B, H, W, 128), dtype=torch.bfloat16, device=hn.device)
        call("lvae_dmol_bwd", l.data_ptr(), xc.data_ptr(), g_ll.contiguous().float().data_ptr(), None, dl.data_ptr(), B,
             H * W, _stream())
        gh = None
        if ctx.needs_input_grad[0]:
            wpb = spec.pack_tc_bwd.get(weight, torch.bfloat16)
            stats["tc_dgrad"] += 1
            gh = as_nchw(_conv_tc(dl, None, wpb, None, None, None, spec.cin, spec.k, True, False))
        gw = gb = None
        if ctx.needs_input_grad[1]:
            gwbuf, sunk = _param_grad_buffer(weight)
            gbbuf, bsunk = _param_grad_buffer(bias)
            with _wgrad_stream(sunk and bsunk, (hn, dl)):
                stats["tc_wgrad"] += 1
                # five accumulator pairs x 128 columns would not fit TMEM: two launches over 64 output channels each
                taps = spec.k * spec.k
                if C == 64:
                    for c0 in (0, 64):
                        call("lvae_conv2d_wgrad_tc", hn.data_ptr(), None, dl.data_ptr(),
                             gwbuf.data_ptr() + c0 * spec.cin * taps * 4, gbbuf.data_ptr() + c0 * 4,
                             _wgrad_workspace(hn.device).data_ptr(), B, H, W, 64, spec.k, 0, min(64, spec.cout - c0), 128, c0,
                             _stream())
                else:
                    # ... and, per dY window, one launch per 64-channel X window (the first adds the bias gradient)
                    stats["tc_wgrad_xwin"] = stats.get("tc_wgrad_xwin", 0) + 1
                    for x0 in range(0, C, 64):
                        for c0 in (0, 64):
                            call("lvae_conv2d_wgrad_tc_ex", hn.data_ptr(), None, dl.data_ptr(),
                                 gwbuf.data_ptr() + c0 * spec.cin * taps * 4, None if x0 else gbbuf.data_ptr() + c0 * 4,
                                 _wgrad_workspace(hn.device).data_ptr(), B, H, W, 64, spec.k, 0, min(64, spec.cout - c0), 128,
                                 c0, C, x0, _stream())
            gw, gb = (None if sunk else gwbuf), (None if bsunk else gbbuf)
        return gh, gw, gb, None, None


def dmol_head(h, conv, x):
    """Fused head when the tensor-core path applies; returns (ll, params) or None."""
    hn_ok = h.dtype == torch.bfloat16 and conv.spec.cout == 100 and conv.spec.cin in (64, 128) and _tc_enabled[0] \
        and conv.spec.tc_shape and _pow2(h.shape[2]) and _pow2(h.shape[3]) and h.shape[3] <= 128
    if hn_ok and conv.spec.cin != 64:
        # wider input: the forward (N = 100, fp32 output) and the dgrad (N = cin) must be launches the library takes
        H, W, k = h.shape[2], h.shape[3], conv.spec.k
        hn_ok = (conv_tc_plan(conv.spec.cin, 100, k, False, H, W, True) != TC_REJECTED
                 and conv_tc_plan(128, conv.spec.cin, k, False, H, W, False) != TC_REJECTED)
    if not hn_ok:
        return None
    return DmolHeadFn.apply(h, conv.weight, conv.bias, x, conv.spec)


def dmol_sample(l):
    ln = nhwc(l).float()
    B, H, W, C = ln.shape
    out = torch.empty((B, 3, H, W), dtype=torch.float32, device=ln.device)
    call("lvae_dmol_sample", ln.data_ptr(), out.data_ptr(), B, H * W, rng_state(ln.device).data_ptr(), next_stream_id(),
         _stream())
    return out


# --------------------------------------------------------------------------- IW bound
def iw_lse_update(ll, kl_sep, state, first: bool):
    call("lvae_iw_lse_update", ll.data_ptr(), kl_sep.data_ptr(), state.data_ptr(), ll.numel(), 1 if first else 0, _stream())


def iw_lse_combine(states, k_total: int):
    R, B, _ = states.shape
    out = torch.empty((B,), dtype=torch.float32, device=states.device)
    call("lvae_iw_lse_combine", states.data_ptr(), out.data_ptr(), R, B, int(k_total), _stream())
    return out
