"""GPU: residual blocks of every 'bacd' layout (bacdbacd / bacdbac, gated or not, any Dropout2d placement) as one block node,
and the residual add on the TMA-store epilogue of the tensor-core convolution that the ungated node ends with."""
import os

import pytest
import torch

from oracle import lvae_oracle as O
from lvae_test_helpers import make_inputs, rel_err

pytestmark = pytest.mark.gpu


def _record(line):
    """Measured error levels go to the directory named by LVAE_RECORD_DIR (when set), so that the bf16 tolerances below
    rest on evidence."""
    d = os.environ.get("LVAE_RECORD_DIR")
    if not d:
        return
    try:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "measured_block_layouts.txt"), "a") as fh:
            fh.write(line + "\n")
    except OSError:
        pass


# ----------------------------------------------------------------------------------------------------- epilogue
def _conv(x, w, bias, mask, res, out_f32, k, stats_acc=None):
    from lvae_b200 import ops
    N = w.shape[0]
    spec = ops.ConvSpec(N, 64, k, 1, k // 2)
    return ops._conv_tc(x, None, spec.pack_tc_fwd.get(w, torch.bfloat16), bias, mask, res, N, k, False, out_f32,
                        stats_acc=stats_acc)


@pytest.mark.parametrize("B,H,W,k,N", [
    (256, 16, 16, 3, 64),     # halo tiles, 512 tiles: several per CTA
    (4, 8, 8, 3, 64),         # plain tiles
    (3, 4, 4, 3, 64),         # 48 pixels: one partial tile
    (2, 32, 32, 3, 64),       # halo tiles
    (5, 8, 8, 1, 128),        # two 64-column chunks per thread, partial last tile
])
@pytest.mark.parametrize("with_mask,with_bias", [(False, False), (True, True), (True, False), (False, True)])
def test_residual_on_tma_store_epilogue_is_exact(B, H, W, k, N, with_mask, with_bias):
    """bf16((acc + bias) * mask + res) rounded once: the fp32 output of the same launch without a residual, plus res in fp32,
    rounded to bf16, bit for bit.  The fused statistics are those of the stored sum."""
    from lvae_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + H + k)
    x = torch.randn((B, H, W, 64), device="cuda", generator=g).to(torch.bfloat16)
    res = torch.randn((B, H, W, N), device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn((N, 64, k, k), device="cuda", generator=g) * (1.0 / (8 * k))
    bias = torch.randn(N, device="cuda", generator=g) if with_bias else None
    mask = ((torch.rand((B, N), device="cuda", generator=g) > 0.3).float() / 0.7) if with_mask else None
    n0 = dict(ops.stats)
    y = _conv(x, w, bias, mask, res, False, k)
    assert ops.stats.get("res_tma", 0) == n0.get("res_tma", 0) + 1
    assert ops.stats.get("res_scattered", 0) == n0.get("res_scattered", 0)
    ref = (_conv(x, w, bias, mask, None, True, k) + res.float()).to(torch.bfloat16)
    torch.cuda.synchronize()
    assert torch.equal(y, ref), float((y.float() - ref.float()).abs().max())
    if N == 64:
        acc = torch.zeros((8, 2, 64), dtype=torch.float64, device="cuda")
        y2 = _conv(x, w, bias, mask, res, False, k, stats_acc=acc)
        assert torch.equal(y2, ref)
        s = acc.sum(0)
        yd = ref.double().reshape(-1, 64)
        assert rel_err(s[0], yd.sum(0)) < 1e-5
        assert rel_err(s[1], (yd * yd).sum(0)) < 1e-5


# ----------------------------------------------------------------------------------------------------- node vs op by op
LAYOUTS = [  # (block type, gated, dropout)
    ("bacdbacd", False, 0.2), ("bacdbac", False, 0.3), ("bacdbac", False, None), ("bacdbac", True, 0.3),
    ("bacdbac", True, None), ("bacdbacd", False, 0.0),
]


def _mnist3(block_type, gated, dropout):
    cfg = O.baseline_config("mnist3")
    cfg.res_block_type, cfg.gated, cfg.dropout = block_type, gated, dropout
    return cfg


def _build(cfg, seed, dtype):
    import lvae_b200
    model = lvae_b200.LadderVAE(**cfg.kwargs())
    model.load_state_dict(O.make_params(cfg, seed), strict=True)
    model = model.cuda()
    if dtype == torch.bfloat16:
        model.set_compute_dtype(torch.bfloat16)
    return model


def _train_once(cfg, dtype, node, B=8):
    import lvae_b200
    from lvae_b200 import ops
    ops.set_whole_block(node)
    try:
        model = _build(cfg, 41, dtype)
        x, eps, masks = make_inputs(cfg, B, 77, True)
        n0 = ops.stats.get("block_node", 0)
        with lvae_b200.inject(eps=[e.float().cuda() for e in eps[0]],
                              masks=[m.float().cuda() for m in masks] if masks else None):
            out = model(x.float().cuda())
        loss = (-out["ll"]).mean() + out["kl_loss"]
        loss.backward()
        torch.cuda.synchronize()
        nodes = ops.stats.get("block_node", 0) - n0
        return (float(loss), {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None},
                {k: v.clone() for k, v in model.state_dict().items() if "running" in k}, nodes)
    finally:
        ops.set_whole_block(True)


# bf16 bounds: about 3x the largest differences measured on a B200 over LAYOUTS (profiles/block_layouts_r03.txt: loss 9.0e-5,
# gradients 4.8e-2 of the tensor's largest entry, running statistics 2.0e-3; eval outputs 1.0e-3)
BF16_TOL = {"loss": 3e-4, "grad": 0.15, "running": 6e-3}


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("block_type,gated,dropout", LAYOUTS)
def test_node_matches_op_by_op_training(block_type, gated, dropout, dtype):
    cfg = _mnist3(block_type, gated, dropout)
    a = _train_once(cfg, dtype, True)
    b = _train_once(cfg, dtype, False)
    assert a[3] > 0 and b[3] == 0
    gmax = max(float(v.abs().max()) for v in b[1].values())
    e_loss = abs(a[0] - b[0]) / abs(b[0])
    e_grad = max(float((a[1][n] - gr).abs().max()) / max(float(gr.abs().max()), 1e-3 * gmax) for n, gr in b[1].items())
    e_run = max(rel_err(a[2][k], v) for k, v in b[2].items())
    _record("node vs op by op, train, %s gated=%s p=%s %s: loss rel %.2e, grad rel(max) %.2e, running rel(max) %.2e" % (
        block_type, gated, dropout, str(dtype).split(".")[-1], e_loss, e_grad, e_run))
    assert set(a[1]) == set(b[1])
    if dtype == torch.float32:          # as tests/test_model_gpu.py::test_whole_block_schedule_matches_op_by_op
        assert e_loss < 1e-5 and e_grad < 1e-4 and e_run < 1e-5, (e_loss, e_grad, e_run)
    else:
        assert e_loss < BF16_TOL["loss"] and e_grad < BF16_TOL["grad"] and e_run < BF16_TOL["running"], (e_loss, e_grad, e_run)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("block_type,gated,dropout", LAYOUTS)
def test_node_matches_op_by_op_eval(block_type, gated, dropout, dtype):
    import lvae_b200
    from lvae_b200 import ops
    from lvae_b200.engine import IWEvaluator
    cfg = _mnist3(block_type, gated, dropout)
    x, eps, _ = make_inputs(cfg, 8, 78, False)
    res = {}
    for node in (True, False):
        ops.set_whole_block(node)
        try:
            model = _build(cfg, 42, dtype).eval()
            with torch.no_grad(), lvae_b200.inject(eps=[e.float().cuda() for e in eps[0]]):
                out = model(x.float().cuda())
            lvae_b200.manual_seed(3)
            bound = IWEvaluator(model, 8, use_graph=False).bound(x.float().cuda(), 4)
            res[node] = (out["ll"].double(), out["kl_sep"].double(), bound.double())
        finally:
            ops.set_whole_block(True)
    errs = [rel_err(a, b) for a, b in zip(res[True], res[False])]
    _record("node vs op by op, eval, %s gated=%s p=%s %s: ll / kl_sep / IW-4 bound rel %s" % (
        block_type, gated, dropout, str(dtype).split(".")[-1], ["%.2e" % e for e in errs]))
    lim = 1e-5 if dtype == torch.float32 else 3e-3
    assert max(errs) < lim, errs


# ----------------------------------------------------------------------------------------------------- float64 oracle
@pytest.mark.parametrize("block_type,dropout", [("bacdbacd", 0.2), ("bacdbac", None)])
def test_ungated_node_gradients_match_oracle(block_type, dropout):
    """Every gradient tensor of a small ungated model (fp32, block node) against the float64 oracle."""
    import lvae_b200
    from lvae_b200 import ops
    from oracle.make_golden import small_cfg
    cfg = small_cfg(res_block_type=block_type, gated=False, dropout=dropout)
    B = 4
    model = lvae_b200.LadderVAE(**cfg.kwargs())
    model.load_state_dict(O.make_params(cfg, 5), strict=True)
    model = model.cuda()
    x, eps, masks = make_inputs(cfg, B, 55, True)
    n0 = ops.stats.get("block_node", 0)
    with lvae_b200.inject(eps=[e.float().cuda() for e in eps[0]], masks=[m.float().cuda() for m in masks] if masks else None):
        out = model(x.float().cuda())
    ((-out["ll"]).mean() + out["kl_loss"]).backward()
    assert ops.stats.get("block_node", 0) > n0
    st = O.TrainState(cfg, O.make_params(cfg, 5, torch.float64))
    o2, t2 = st.step(x, eps[0], masks, update=False)
    assert rel_err((-out["ll"]).mean() + out["kl_loss"], t2["loss"]) < 1e-4
    gmax = max(float(st.P[n].grad.abs().max()) for n in st.names if st.P[n].grad is not None)
    for n, p in model.named_parameters():
        gr = st.P[n].grad
        if gr is None:
            continue
        err = float((p.grad.double().cpu() - gr).abs().max())
        assert err < 1e-3 * max(float(gr.abs().max()), 1e-3 * gmax), (n, err, float(gr.abs().max()))


# ----------------------------------------------------------------------------------------------------- coverage
def _count_forward(cfg, B=2):
    from lvae_b200 import ops
    from lvae_b200.lib.nn import ResidualBlock
    model = _build(cfg, 43, torch.bfloat16)
    n_blocks = sum(1 for m in model.modules() if isinstance(m, ResidualBlock))
    n_ungated = sum(1 for m in model.modules() if isinstance(m, ResidualBlock) and not m.gated)
    x, _, _ = make_inputs(cfg, B, 79, True)
    n0 = dict(ops.stats)
    out = model(x.float().cuda())
    ((-out["ll"]).mean() + out["kl_loss"]).backward()
    torch.cuda.synchronize()
    d = {k: ops.stats.get(k, 0) - n0.get(k, 0) for k in ("block_node", "res_tma", "res_scattered")}
    return n_blocks, n_ungated, d


def test_every_residual_block_of_an_ungated_cifar15_takes_the_node():
    """Stem, bottom-up, top-down and final blocks: one node each, and no bf16 residual conv on the scattered epilogue."""
    cfg = O.baseline_config("cifar15")
    cfg.gated = False
    n_blocks, n_ungated, d = _count_forward(cfg)
    assert n_blocks > 30 and n_ungated > 30          # the merge layers' blocks are always gated (conv2 + gate chain, no res)
    assert d["block_node"] == n_blocks, (n_blocks, d)
    assert d["res_tma"] == n_ungated and d["res_scattered"] == 0, (n_ungated, d)


@pytest.mark.parametrize("block_type,batchnorm", [("cabdcabd", True), ("bacdbacd", False)])
def test_step_by_step_layouts_take_the_node_zero_times(block_type, batchnorm):
    cfg = O.baseline_config("mnist3")
    cfg.res_block_type, cfg.batchnorm = block_type, batchnorm
    _, _, d = _count_forward(cfg)
    assert d["block_node"] == 0


# ----------------------------------------------------------------------------------------------------- engines
def _run_engine(cfg, dtype, use_graph, steps, batch, side, node=True):
    import lvae_b200
    from lvae_b200 import ops
    from lvae_b200.engine import TrainEngine
    ops.set_whole_block(node)
    try:
        lvae_b200.manual_seed(7)
        model = _build(cfg, 31, dtype)
        eng = TrainEngine(model, batch, use_graph=use_graph, wgrad_side_stream=side)
        losses = []
        for i in range(steps):
            x, _, _ = make_inputs(cfg, batch, 40 + i, True)
            losses.append(float(eng.step(x.float().cuda())["loss"]))
        torch.cuda.synchronize()
        bufs = torch.cat([b.detach().double().flatten() for b in model.buffers()])
        return losses, eng.arena.flat.detach().clone(), bufs, eng.launches_per_step
    finally:
        ops.set_whole_block(True)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_ungated_graph_replay_equals_eager_steps(dtype):
    """As tests/test_engine_gpu.py::test_graph_replay_equals_eager_steps, for MNIST-3 with ungated blocks."""
    from lvae_b200 import ops
    cfg = _mnist3("bacdbacd", False, 0.2)
    le, pe, be, _ = _run_engine(cfg, dtype, False, 3, 8, side=False)
    lg, pg, bg, launches = _run_engine(cfg, dtype, True, 3, 8, side=True)
    tol_l, tol_p = (8e-6, 2e-6) if dtype == torch.float32 else (2e-4, 3e-5)
    for a, b in zip(le, lg):
        assert abs(a - b) <= tol_l * abs(a), (le, lg)
    d = (pe - pg).abs()
    assert float((d > tol_p).float().mean()) < 5e-3
    assert float(d.max()) <= 3 * 3e-4 * 2 + 1e-6
    assert rel_err(bg, be) < 1e-4
    assert not ops._pending_bn1
    _, _, _, launches_off = _run_engine(cfg, dtype, True, 2, 8, side=True, node=False)
    _record("launches per step, MNIST-3 ungated %s: node %d, op by op %d" % (str(dtype).split(".")[-1], launches, launches_off))
    assert 0 < launches < launches_off


def test_ungated_iw_graph_equals_eager_and_sharding_is_invariant():
    import lvae_b200
    from lvae_b200 import ops
    from lvae_b200.engine import IWEvaluator
    cfg = _mnist3("bacdbacd", False, 0.2)
    model = _build(cfg, 23, torch.float32)
    x, _, _ = make_inputs(cfg, 16, 2, False)
    xd = x.float().cuda()
    K = 11
    lvae_b200.manual_seed(6)
    bg = IWEvaluator(model, 16, use_graph=True).bound(xd, K)
    lvae_b200.manual_seed(6)
    be = IWEvaluator(model, 16, use_graph=False).bound(xd, K)
    assert float((bg - be).abs().max()) < 1e-5 * abs(float(be.mean())) + 1e-4, (bg, be)
    states = []
    for r in range(2):
        lvae_b200.manual_seed(6)
        ev = IWEvaluator(model, 16, use_graph=False)
        ev.rank, ev.world = r, 2
        states.append(ev.local_state(xd, K).clone())
    bs = ops.iw_lse_combine(torch.stack(states).contiguous(), K)
    assert float((bs - be).abs().max()) < 2e-4 * abs(float(be.mean())) + 1e-4
