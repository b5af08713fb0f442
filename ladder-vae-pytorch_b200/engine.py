"""Step engines: the training step and the importance-weighted evaluation as replayable CUDA
graphs over flat parameter / gradient arenas, data-parallel across one process per GPU.

What the reference does per step in Python (experiment/experiment_manager.py:322-367 forward_pass,
:78-80 Adamax over ~1700 tensors, :346-350 L2 loop, boilr's train loop) is here one captured
graph: rng advance -> grad arena memset -> batched weight re-pack -> LadderVAE forward -> loss ->
backward (kernels accumulate parameter gradients straight into the arena) -> [NCCL all-reduce of
the arena in buckets, outside the graph] -> fused Adamax + L2 norm.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, Optional

import torch
import torch.distributed as dist

from . import _capi, ops
from .lib.nn import Conv2d, ConvTranspose2d

call = _capi.call


def _stream():
    return torch.cuda.current_stream().cuda_stream


def shard_samples(k_total: int, rank: int, world: int):
    """Contiguous split of K importance samples over ranks (first ranks take the remainder)."""
    base, rem = divmod(k_total, world)
    n = base + (1 if rank < rem else 0)
    start = rank * base + min(rank, rem)
    return start, n


def bucket_ranges(numel: int, bucket_bytes: int = 25 << 20, elem_bytes: int = 4):
    """[start, end) element ranges of the gradient arena, one NCCL call each."""
    per = max(1, bucket_bytes // elem_bytes)
    return [(s, min(numel, s + per)) for s in range(0, numel, per)]


def bucket_ranges_aligned(starts, numel: int, bucket_bytes: int = 25 << 20, elem_bytes: int = 4):
    """Like bucket_ranges, but every cut falls on a tensor boundary (`starts` = sorted start offsets of the tensors in the
    arena): a bucket is reduced as soon as its last gradient is out, so no tensor may straddle two buckets."""
    per = max(1, bucket_bytes // elem_bytes)
    cuts, begin = [0], 0
    for s in list(starts)[1:]:
        if s - begin >= per:
            cuts.append(s)
            begin = s
    return [(a, b) for a, b in zip(cuts, cuts[1:] + [numel])]


def all_reduce_buckets(flat: torch.Tensor, buckets, group=None) -> None:
    """Sum-all-reduce a flat gradient arena bucket by bucket (NCCL on GPUs; device agnostic)."""
    for s, e in buckets:
        dist.all_reduce(flat[s:e], op=dist.ReduceOp.SUM, group=group)


def gather_states(state: torch.Tensor, group=None) -> torch.Tensor:
    """All-gather the per-rank (B,2) running (max, sum-exp) states into (R,B,2)."""
    world = dist.get_world_size(group)
    out = torch.empty((world * state.shape[0],) + tuple(state.shape[1:]), dtype=state.dtype, device=state.device)
    dist.all_gather_into_tensor(out, state.contiguous(), group=group)
    return out.view((world,) + tuple(state.shape))


def grad_ready_order(model: torch.nn.Module):
    """Trainable parameters in the order the backward pass finishes their gradients: likelihood head, final top-down
    blocks, top-down layers bottom -> top, bottom-up layers top -> bottom, stem (the reverse of LadderVAE.forward,
    models/lvae.py:172-214; autograd runs the later-created nodes first), each module's own parameters reversed.  Buckets
    of the gradient arena cut in this order complete one after the other during the backward, so their all-reduce can
    start early.  Any other model: reversed registration order."""
    groups = []
    if all(hasattr(model, a) for a in ("likelihood", "final_top_down", "top_down_layers", "bottom_up_layers", "first_bottom_up")):
        groups = [model.likelihood, model.final_top_down, *list(model.top_down_layers),
                  *reversed(list(model.bottom_up_layers)), model.first_bottom_up]
    seen, out = set(), []
    for g in groups:
        for p in reversed(list(g.parameters())):
            if p.requires_grad and id(p) not in seen:
                seen.add(id(p))
                out.append(p)
    for p in reversed(list(model.parameters())):
        if p.requires_grad and id(p) not in seen:
            seen.add(id(p))
            out.append(p)
    return out


class ParamArena:
    """All trainable parameters of a model as views into one flat fp32 buffer (laid out in gradient-ready order), with a
    parallel gradient buffer that the wgrad / BatchNorm / prior kernels accumulate into directly."""

    def __init__(self, model: torch.nn.Module):
        params = grad_ready_order(model)
        if not params:
            raise RuntimeError("model has no trainable parameters")
        dev = params[0].device
        if dev.type != "cuda":
            raise RuntimeError("lvae_b200 has no CPU path: move the model to a CUDA device first")
        sizes = [((p.numel() + 3) // 4) * 4 for p in params]          # keep every view 16-byte aligned
        self.numel = sum(sizes)
        self.flat = torch.zeros(self.numel, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(self.numel, dtype=torch.float32, device=dev)
        self.params, off = params, 0
        self.offsets = {}
        for p, n in zip(params, sizes):
            self.offsets[id(p)] = off
            view = self.flat[off:off + p.numel()].view(p.shape)
            view.copy_(p.data)
            p.data = view
            sink = self.grad[off:off + p.numel()].view(p.shape)
            p._lvae_grad_sink = sink
            p.grad = sink
            off += n

    def detach_sinks(self):
        for p in self.params:
            if hasattr(p, "_lvae_grad_sink"):
                del p._lvae_grad_sink
            if hasattr(p, "_lvae_gp"):
                del p._lvae_gp


class PackedGradArena:
    """Packed weight gradients of every convolution the tcgen05 wgrad kernel serves (lvae_conv2d_wgrad_tc_acc adds
    into them with TMA reduce-stores), and the device table that lets ONE launch per step re-lay all of them into the
    (O,I,kh,kw) gradient arena and clear them again."""

    def __init__(self, model: torch.nn.Module):
        lib = _capi.lib()
        convs = []
        for m in model.modules():
            if isinstance(m, (Conv2d, ConvTranspose2d)):
                sp = m.spec
                w = m.weight
                if not (w.requires_grad and hasattr(w, "_lvae_grad_sink")):
                    continue
                if sp.s2_shape:
                    # stride-2 resampling convs (lvae_conv2d_wgrad_tc_s2_acc): same packed layout as a 3x3 64 -> 64 conv.  A
                    # ConvTranspose2d's bias gradient sums the large grid (lvae_colsum), not the packed ones-row.
                    n = int(lib.lvae_wgrad_tc_packed_size(64, 3, 0))
                    if m.bias is None or hasattr(m.bias, "_lvae_grad_sink"):
                        convs.append((m, False, n))
                    continue
                if not sp.tc_shape:
                    continue
                two = sp.cin == 128 and sp.k == 1
                if not (sp.cin <= 64 or two):
                    continue
                # only convs whose weight gradient is one launch (ops.conv_backward_raw splits the others over dY windows)
                if ops.wgrad_tc_plan(sp.cout, sp.k, two) != ((sp.cout, 0),):
                    continue
                n = int(lib.lvae_wgrad_tc_packed_size(sp.cout, sp.k, int(two)))
                if m.bias is None or hasattr(m.bias, "_lvae_grad_sink"):
                    convs.append((m, two, n))
        self.n = len(convs)
        if not self.n:
            return
        dev = convs[0][0].weight.device
        self.flat = torch.zeros(sum(n for _, _, n in convs), dtype=torch.float32, device=dev)
        dsz = int(lib.lvae_wgrad_unpack_desc_size())
        host = ctypes.create_string_buffer(dsz * self.n)
        off = 0
        for i, (m, two, n) in enumerate(convs):
            gp = self.flat[off:off + n]
            off += n
            m.weight._lvae_gp = gp
            m.weight._lvae_gp_id = i
            bias_sink = m.bias._lvae_grad_sink if (m.bias is not None and not m.spec.transposed) else None
            call("lvae_wgrad_unpack_desc", ctypes.addressof(host) + i * dsz, gp.data_ptr(), m.weight._lvae_grad_sink.data_ptr(),
                 bias_sink.data_ptr() if bias_sink is not None else None, m.spec.cout, m.spec.k, int(two), m.spec.cin,
                 m.spec.cout, 1)      # clear Gp; ADD into the arena (a generic-path fallback may have written it too)
        self.dsz = dsz
        self.table = torch.frombuffer(bytearray(host.raw), dtype=torch.uint8).to(dev).view(self.n, dsz)
        self._sub = {}

    def unpack(self, ids=None):
        """Re-lay the packed gradients `ids` (default: all) into the gradient arena, on the current stream.  Sub-tables are
        cached per id tuple (built during the eager warm-up steps, so nothing is allocated under graph capture)."""
        if not self.n:
            return
        if ids is None:
            tab, n = self.table, self.n
        else:
            key = tuple(ids)
            if not key:
                return
            tab = self._sub.get(key)
            if tab is None:
                tab = self.table[torch.tensor(key, dtype=torch.long, device=self.table.device)].contiguous()
                self._sub[key] = tab
            n = len(key)
        call("lvae_wgrad_unpack_batched", tab.data_ptr(), n, 128, _stream())


class PackTable:
    """One device table of LvaePackDesc for every conv weight (both GEMM layouts): the whole
    model is re-packed by ONE launch per step."""

    def __init__(self, model: torch.nn.Module, dtype: torch.dtype):
        self.entries = []
        raws = []
        for m in model.modules():
            if isinstance(m, (Conv2d, ConvTranspose2d)):
                for pack in m.spec.packs(dtype == torch.bfloat16):
                    raws.append(pack.alloc(m.weight, dtype))
                    self.entries.append((pack, m.weight))
        self.dtype = dtype
        self.table = torch.frombuffer(bytearray(b"".join(raws)), dtype=torch.uint8).cuda()
        self.n = len(raws)

    def repack(self):
        call("lvae_pack_weights", self.table.data_ptr(), self.n, _stream())
        for pack, w in self.entries:
            pack.mark_fresh(w, self.dtype)


class TrainEngine:
    """ELBO training step (SURVEY.md 3.1) for a lvae_b200.LadderVAE on one GPU of a data-parallel job."""

    def __init__(self, model, batch_size: int, lr: float = 3e-4, weight_decay: float = 0.0, betas=(0.9, 0.999),
                 eps: float = 1e-8, beta_kl: float = 1.0, use_graph: bool = True, process_group=None,
                 bucket_bytes: int = 12 << 20, compute_l2: bool = True, wgrad_side_stream: bool = True,
                 overlap_allreduce: bool = True):
        _capi.device_check()
        self.model = model.train()
        self.batch_size = batch_size
        self.betas, self.eps = betas, eps
        self.pg = process_group
        inited = process_group is not None or dist.is_initialized()
        self.world = dist.get_world_size(process_group) if inited else 1
        self.rank = dist.get_rank(process_group) if inited else 0
        self.arena = ParamArena(model)
        dev = self.arena.flat.device
        self.device = dev
        # learning rate, weight decay and the KL weight live on the device: the captured graphs read them at replay, so
        # schedules (the reference's --beta-anneal, experiment_manager.py:339-344) need no recapture
        self._hyper = torch.tensor([lr, weight_decay], dtype=torch.float32, device=dev)
        self._beta = torch.tensor(float(beta_kl), dtype=torch.float32, device=dev)
        self._lr, self._wd, self._beta_kl = float(lr), float(weight_decay), float(beta_kl)
        if self.world > 1:
            ops.fold_rank(self.rank)        # replicas must not share eps / Dropout2d masks: one Philox key per rank
        self.exp_avg = torch.zeros_like(self.arena.flat)
        self.exp_inf = torch.zeros_like(self.arena.flat)
        self.step_count = torch.zeros((), dtype=torch.int64, device=dev)
        self.l2_acc = torch.zeros((), dtype=torch.float64, device=dev)
        self.l2 = torch.zeros((), dtype=torch.float32, device=dev)
        self.compute_l2 = compute_l2
        self.packs = PackTable(model, getattr(model, "compute_dtype", torch.float32))
        self.gpacks = PackedGradArena(model)
        self.buckets = bucket_ranges_aligned(sorted(self.arena.offsets.values()), self.arena.numel, bucket_bytes)
        # data parallel: bucket k of the gradient arena is all-reduced on the communication stream as soon as the backward has
        # issued its last gradient (the arena is in gradient-ready order), overlapping NCCL with the rest of the backward
        self.overlap = bool(overlap_allreduce) and self.world > 1
        self.comm_stream = torch.cuda.Stream(device=dev) if self.overlap else None
        starts = [s for s, _ in self.buckets]
        import bisect
        self._bucket_of = {pid: bisect.bisect_right(starts, off) - 1 for pid, off in self.arena.offsets.items()}
        self._gp_bucket = {}
        for m in model.modules():
            if isinstance(m, (Conv2d, ConvTranspose2d)) and hasattr(m.weight, "_lvae_gp_id"):
                ks = [self._bucket_of[id(m.weight)]] + ([self._bucket_of[id(m.bias)]] if m.bias is not None and id(m.bias) in self._bucket_of else [])
                self._gp_bucket[m.weight._lvae_gp_id] = min(ks)
        self._ready_counts = None          # parameters per bucket that announce their gradient (calibrated on the first step)
        self._flushed = set()
        self._unpacked = set()
        self.x = torch.zeros((batch_size, model.color_ch) + tuple(model.img_shape), dtype=torch.float32, device=dev)
        self.use_graph = use_graph
        n_side = int(wgrad_side_stream) if not isinstance(wgrad_side_stream, bool) else (3 if wgrad_side_stream else 0)
        # Side streams run at the lowest priority and the step is captured on a high-priority stream: when SMs free up the
        # block scheduler serves the dependent main chain (fwd / dgrad / BatchNorm) first, the weight gradients fill the rest.
        lo, hi = torch.cuda.Stream.priority_range() if hasattr(torch.cuda.Stream, "priority_range") else (0, -1)
        # measured on a B200 at the end of round 2 (three side streams): 14.41-14.44 ms per step with priorities vs 14.50 without
        self.side_stream = [torch.cuda.Stream(device=dev, priority=lo) for _ in range(n_side)] if n_side else None
        self.main_stream = torch.cuda.Stream(device=dev, priority=hi)
        self.graph_fb: Optional[torch.cuda.CUDAGraph] = None
        self.graph_opt: Optional[torch.cuda.CUDAGraph] = None
        self.out: Dict[str, torch.Tensor] = {}
        self.launches_per_step = 0
        if self.world > 1:                      # all replicas start from rank 0's weights
            dist.broadcast(self.arena.flat, 0, group=self.pg)
            for b in model.buffers():
                dist.broadcast(b, 0, group=self.pg)

    # -- hyper-parameters (device resident; setting them is a tiny H2D copy, no recapture) ------
    @property
    def lr(self):
        return self._lr

    @lr.setter
    def lr(self, v):
        self._lr = float(v)
        self._hyper[0:1].copy_(torch.tensor([self._lr], dtype=torch.float32), non_blocking=True)

    @property
    def wd(self):
        return self._wd

    @wd.setter
    def wd(self, v):
        self._wd = float(v)
        self._hyper[1:2].copy_(torch.tensor([self._wd], dtype=torch.float32), non_blocking=True)

    @property
    def beta_kl(self):
        return self._beta_kl

    @beta_kl.setter
    def beta_kl(self, v):
        self._beta_kl = float(v)
        self._beta.copy_(torch.tensor(self._beta_kl, dtype=torch.float32), non_blocking=True)

    # -- checkpoint / resume of the optimizer side (the model's own state_dict holds the parameters) ------
    def state_dict(self):
        """Adamax moments in the layout of torch.optim.Adamax's per-parameter state (keyed by parameter name), the step
        count, hyper-parameters and the Philox state."""
        names = {id(p): n for n, p in self.model.named_parameters()}
        state, off = {}, 0
        for p in self.arena.params:
            n = p.numel()
            state[names[id(p)]] = {"exp_avg": self.exp_avg[off:off + n].view(p.shape).clone(),
                                   "exp_inf": self.exp_inf[off:off + n].view(p.shape).clone()}
            off += ((n + 3) // 4) * 4
        return {"state": state, "step": int(self.step_count), "lr": self._lr, "weight_decay": self._wd,
                "beta_kl": self._beta_kl, "betas": tuple(self.betas), "eps": self.eps,
                "rng": ops.rng_state(self.device).clone().cpu()}

    def load_state_dict(self, sd):
        names = {id(p): n for n, p in self.model.named_parameters()}
        off = 0
        for p in self.arena.params:
            n = p.numel()
            st = sd["state"][names[id(p)]]
            self.exp_avg[off:off + n].view(p.shape).copy_(st["exp_avg"])
            self.exp_inf[off:off + n].view(p.shape).copy_(st["exp_inf"])
            off += ((n + 3) // 4) * 4
        self.step_count.fill_(int(sd["step"]))
        self.lr, self.wd, self.beta_kl = sd["lr"], sd["weight_decay"], sd["beta_kl"]
        if sd.get("rng") is not None:
            ops.rng_state(self.device).copy_(sd["rng"])
        ops.bump_pack_epoch()

    # -- pieces ---------------------------------------------------------------------------
    def _forward_backward(self):
        # Philox streams are numbered from 0 in every step (the per-step offset advance keeps steps apart), so an eager
        # step and a graph replay of the same step draw identical eps / Dropout2d masks
        ops.set_stream_id(0)
        ops.rng_advance(self.device)
        self.arena.grad.zero_()
        self.packs.repack()
        out = self.model(self.x)
        recons = (-out["ll"]).mean()
        loss = recons + out["kl_loss"] * self._beta
        ops.set_side_stream(self.side_stream)          # (None: everything on this stream; also resets the wgrad log)
        self._flushed, self._unpacked = set(), set()
        record = None
        if self.overlap:
            if self._ready_counts is None:
                record = set()                         # first step: learn which parameters announce their gradients
                ops.grad_track_begin(self._bucket_of, [], self._flush_bucket, record)
            else:
                ops.grad_track_begin(self._bucket_of, self._ready_counts, self._flush_bucket)
        try:
            loss.backward()
            ops.grad_track_end()
            if record is not None:
                counts = [0] * len(self.buckets)
                for pid in record:
                    counts[self._bucket_of[pid]] += 1
                # a bucket that also holds gradients autograd accumulates by itself (no announcement) waits for the end
                silent = [0] * len(self.buckets)
                for pid, k in self._bucket_of.items():
                    if pid not in record:
                        silent[k] += 1
                self._ready_counts = [c if (c > 0 and silent[k] == 0) else -1 for k, c in enumerate(counts)]
            # re-lay the remaining packed weight gradients where their wgrads ran: each side stream unpacks its own
            # convolutions (concurrently with the main stream's tail), then the streams join
            self._unpack_ready(None)
            if self.overlap:
                for k in range(len(self.buckets)):
                    self._flush_bucket(k)
                torch.cuda.current_stream().wait_stream(self.comm_stream)
        finally:
            ops.grad_track_end()
            ops.join_side_stream()
            ops.set_side_stream(None)
        elbo = (out["ll"] - out["kl_sep"]).mean()
        self.out = {"loss": loss.detach(), "elbo": elbo.detach(), "recons": recons.detach(), "kl": out["kl"].detach(),
                    "kl_avg_layerwise": out["kl_avg_layerwise"].detach()}

    def _unpack_ready(self, bucket):
        """Unpack the packed weight gradients issued so far (of `bucket`, or all that are left) on the streams that ran them."""
        for slot, ids in ops.packed_grad_log().items():
            todo = [i for i in ids if i not in self._unpacked and (bucket is None or self._gp_bucket.get(i) == bucket)]
            if not todo:
                continue
            self._unpacked.update(todo)
            if slot >= 0 and self.side_stream is not None:
                with torch.cuda.stream(self.side_stream[slot]):
                    self.gpacks.unpack(todo)
            else:
                self.gpacks.unpack(todo)

    def _flush_bucket(self, k):
        """All gradients of bucket k have been issued: unpack its packed weight gradients and all-reduce it on the
        communication stream (behind everything issued so far on the main and side streams)."""
        if k in self._flushed:
            return
        self._flushed.add(k)
        self._unpack_ready(k)
        cs = self.comm_stream
        cs.wait_stream(torch.cuda.current_stream())
        for st in (self.side_stream or []):
            cs.wait_stream(st)
        s, e = self.buckets[k]
        with torch.cuda.stream(cs):
            dist.all_reduce(self.arena.grad[s:e], op=dist.ReduceOp.SUM, group=self.pg)

    def _all_reduce(self):
        if self.world > 1 and not self.overlap:
            all_reduce_buckets(self.arena.grad, self.buckets, self.pg)

    def _optimizer(self):
        a = self.arena
        if self.compute_l2:        # the L2 norm of the updated parameters (experiment_manager.py:346-350) rides on the Adamax pass
            call("lvae_adamax_step_l2", a.flat.data_ptr(), a.grad.data_ptr(), self.exp_avg.data_ptr(), self.exp_inf.data_ptr(),
                 a.numel, self._lr, self.betas[0], self.betas[1], self.eps, self._wd, self.step_count.data_ptr(),
                 1.0 / self.world, self._hyper.data_ptr(), self.l2_acc.data_ptr(), self.l2.data_ptr(), _stream())
        else:
            call("lvae_adamax_step", a.flat.data_ptr(), a.grad.data_ptr(), self.exp_avg.data_ptr(), self.exp_inf.data_ptr(),
                 a.numel, self._lr, self.betas[0], self.betas[1], self.eps, self._wd, self.step_count.data_ptr(),
                 1.0 / self.world, self._hyper.data_ptr(), _stream())
        self.out["l2"] = self.l2

    def _eager_step(self):
        self._forward_backward()
        self._all_reduce()
        self._optimizer()

    def _capture(self):
        # Warm-up on a side stream (allocates pack buffers, BatchNorm scratch, sub-tables of the packed-gradient unpack).
        # The two eager steps are real steps on the caller's first batch, so everything they mutate is put back before
        # the capture: parameters, Adamax moments, step count, BatchNorm running statistics, the Philox state.  The first
        # step(x) in graph mode therefore applies exactly one update, like use_graph=False and like the reference.
        snap = [(t, t.clone()) for t in (self.arena.flat, self.exp_avg, self.exp_inf, self.step_count,
                                         ops.rng_state(self.device))]
        snap += [(b, b.clone()) for b in self.model.buffers()]
        gstep = getattr(self.model, "global_step", 0)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                self._eager_step()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        for t, c in snap:
            t.copy_(c)
        self.model.global_step = gstep
        torch.cuda.synchronize()
        # Parameters changed behind torch's version counters (Adamax and the restore above write through raw pointers):
        # every cached GEMM-layout weight copy is stale.  The batched re-pack at the top of the step refreshes the table's
        # packs; any OTHER pack a convolution falls back to (CUDA-core layouts of the 64 -> 1 Bernoulli head, odd sizes)
        # now misses its cache key during capture, so its on-demand lvae_pack_weights launch becomes a node of the graph
        # and runs on every replay.
        ops.bump_pack_epoch()
        n0 = _capi.launch_count()
        self.graph_fb = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph_fb, stream=self.main_stream):
            self._forward_backward()
        self.graph_opt = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph_opt, pool=self.graph_fb.pool()):
            self._optimizer()
        self.launches_per_step = _capi.launch_count() - n0

    # -- public ---------------------------------------------------------------------------
    def step(self, x: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """One optimisation step.  ``x``: (B,C,H,W) in [0,1], host (ideally pinned) or device;
        None re-uses the resident batch.  Returns device scalars (no host sync)."""
        if x is not None:
            self.x.copy_(x, non_blocking=True)
        if not self.use_graph:
            n0 = _capi.launch_count()
            self._eager_step()
            self.launches_per_step = _capi.launch_count() - n0
        else:
            if self.graph_fb is None:
                self._capture()
            self.graph_fb.replay()
            self._all_reduce()
            self.graph_opt.replay()
        ops.bump_pack_epoch()          # parameters changed behind torch's version counters
        self.model.global_step = getattr(self.model, "global_step", 0) + 1
        return self.out


class IWEvaluator:
    """Importance-weighted bound log p(x) >= logsumexp_k(ll_k - kl_k) - log K (SURVEY.md 3.3), with the
    K samples sharded over ranks and one (B,2) all-gather + combine per image batch."""

    def __init__(self, model, batch_size: int, use_graph: bool = True, process_group=None, reuse_bottomup: bool = True):
        _capi.device_check()
        self.model = model.eval()
        self.reuse_bottomup = reuse_bottomup      # False: full forward per sample, like the reference's loop
        self.bu = None
        self.pg = process_group
        inited = process_group is not None or dist.is_initialized()
        self.world = dist.get_world_size(process_group) if inited else 1
        self.rank = dist.get_rank(process_group) if inited else 0
        dev = next(model.parameters()).device
        self.device = dev
        self.x = torch.zeros((batch_size, model.color_ch) + tuple(model.img_shape), dtype=torch.float32, device=dev)
        self.state = torch.zeros((batch_size, 2), dtype=torch.float32, device=dev)
        self.use_graph = use_graph
        self.graph = None
        self.graph_bu = None
        self.launches_per_sample = 0
        self.launches_bottomup = 0

    def _bottomup(self):
        self.bu = self.model.bottomup_pass(self.model.pad_input(self.x)) if self.reuse_bottomup else None

    def _one_sample(self):
        ops.set_stream_id(0)             # sample k of an image batch = Philox offset k, stream ids numbered from 0
        ops.rng_advance(self.device)
        out = self.model.forward_from_bottomup(self.x, self.bu) if self.reuse_bottomup else self.model(self.x)
        ops.iw_lse_update(out["ll"], out["kl_sep"], self.state, False)

    def _reset(self):
        self.state[:, 0].fill_(-math.inf)
        self.state[:, 1].zero_()

    def local_state(self, x: torch.Tensor, k_total: int) -> torch.Tensor:
        """This rank's share of the K-sample bound for one image batch: (B,2) running (max, sum-exp) of ll - kl over the
        samples shard_samples() assigns to this rank."""
        k_start, k_local = shard_samples(k_total, self.rank, self.world)
        with torch.no_grad(), ops.shared_key():
            self.x.copy_(x, non_blocking=True)
            self._reset()
            if self.use_graph and self.graph is None:
                rng0 = ops.rng_state(self.device).clone()
                s = torch.cuda.Stream()
                s.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s):
                    self._bottomup()
                    self._one_sample()
                torch.cuda.current_stream().wait_stream(s)
                torch.cuda.synchronize()
                self._reset()
                n0 = _capi.launch_count()
                self.graph_bu = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph_bu):
                    self._bottomup()
                self.launches_bottomup = _capi.launch_count() - n0
                n0 = _capi.launch_count()
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph, pool=self.graph_bu.pool()):
                    self._one_sample()
                self.launches_per_sample = _capi.launch_count() - n0
                ops.rng_state(self.device).copy_(rng0)      # the warm-up sample must not shift the noise sequence
                self._reset()
            if self.use_graph:
                self.graph_bu.replay()
            else:
                self._bottomup()
            # Sample k of this batch always draws from Philox offset (base + k): a rank skips the samples of the ranks
            # before it, so the K samples are distinct across ranks (with the usual same-seed-everywhere setup they would
            # otherwise be `world` copies of K/world samples) and the bound does not depend on how K is sharded.
            if k_start:
                ops.rng_advance(self.device, k_start * ops.RNG_STEP)
            for _ in range(k_local):
                if self.use_graph:
                    self.graph.replay()
                else:
                    n0 = _capi.launch_count()
                    self._one_sample()
                    self.launches_per_sample = _capi.launch_count() - n0
            k_rest = k_total - k_start - k_local
            if k_rest:
                ops.rng_advance(self.device, k_rest * ops.RNG_STEP)      # every rank ends the batch at the same offset
            return self.state

    def bound(self, x: torch.Tensor, k_total: int) -> torch.Tensor:
        """Per-image IW bound (B,) for this image batch with k_total samples over all ranks."""
        state = self.local_state(x, k_total)
        with torch.no_grad():
            states = gather_states(state, self.pg) if self.world > 1 else state[None]
            return ops.iw_lse_combine(states.contiguous(), k_total)
