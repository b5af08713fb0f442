"""GPU: the tensor-core path at 128 filters -- streamed-weight convolutions (csrc/conv_tcgen05.cu) and input-channel windows
of the weight gradient (csrc/wgrad_tcgen05.cu) -- against float64, then a 128-filter LadderVAE end to end.

Kernel cases use operands from the bf16 integers {-2, ..., 2} (and integer biases), so every fp32 accumulator is an exact
integer: each result must equal the float64 reference rounded ONCE to the output dtype, bit for bit.  Every y / dw / dbias
sits in a sentinel-filled buffer that must be untouched afterwards."""
import pytest
import torch
import torch.nn.functional as F

from oracle import lvae_oracle as O
from oracle.make_golden import make_inputs, small_cfg
from lvae_test_helpers import rel_err

pytestmark = pytest.mark.gpu

GUARD = 4096
NUM_SMS = 148


def _lib():
    import lvae_b200
    return lvae_b200._capi


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def ints(shape, gen, dtype=torch.bfloat16):
    return torch.randint(-2, 3, shape, generator=gen, device="cuda", dtype=torch.int32).to(dtype)


class Guarded:
    """A tensor of `shape` in the middle of a buffer filled with a sentinel that no kernel may overwrite."""

    def __init__(self, shape, dtype, zero=True):
        n = 1
        for s in shape:
            n *= s
        self.n, self.sent = n, 1000.0                     # representable in bf16 and fp32, never a result here
        self.buf = torch.full((n + 2 * GUARD,), self.sent, dtype=dtype, device="cuda")
        self.t = self.buf[GUARD:GUARD + n].view(shape)
        if zero:
            self.t.zero_()

    def intact(self):
        return bool((self.buf[:GUARD] == self.sent).all()) and bool((self.buf[GUARD + self.n:] == self.sent).all())


def exact(got, ref64, what):
    want = ref64.to(got.dtype)
    bad = got.float() != want.float()
    assert not bool(bad.any()), "%s: %d of %d entries differ (max |d| %.3g)" % (
        what, int(bad.sum()), bad.numel(), float((got.double() - ref64).abs().max()))


def pack(weight, mode):
    """lvae_pack_weights of a (O, I, k, k) fp32 weight: mode 2 forward operand, mode 3 dgrad operand."""
    from lvae_b200 import ops
    o, i, k, _ = weight.shape
    wp = ops.WeightPack(o, i, k * k, mode)
    return wp.get(weight, torch.bfloat16)


def tc_plan(cin, n, k, two, h, w, f32):
    return int(_lib().lib().lvae_conv2d_tc_plan(cin, n, k, int(two), h, w, int(f32)))


def n_tiles(B, H, W):
    return (B * H * W + 127) // 128


# (B, H, W): one CTA, an uneven last CTA, a capped grid at the benchmark size.  Non-halo tiles (Cin > 64 has no halo path):
# 128 pixels per tile, a grid of min(tiles, 148) persistent CTAs.
GRIDS = [(1, 8, 8), (3, 16, 16), (256, 16, 16), (256, 32, 32)]


def test_grid_table_covers_single_cta_uneven_and_capped_launches():
    t = [n_tiles(*g) for g in GRIDS]
    assert 1 in t                                                 # single-CTA launch
    assert any(x > NUM_SMS and x % NUM_SMS for x in t)            # capped grid whose CTAs do unequal numbers of tiles
    assert any(x > NUM_SMS for x in t) and max(t) == 256 * 32 * 32 // 128


# forward: (Cin, N, k, two inputs, fp32 output, residual, expected plan)
FWD = [
    (128, 128, 3, False, False, False, 2),      # streamed, TMA-store epilogue (N = 128)
    (128, 128, 3, False, False, True, 2),       # streamed, plain epilogue (residual)
    (128, 64, 3, False, False, False, 1),       # resident, TMA-store epilogue (N = 64)
    (128, 100, 3, False, True, False, 2),       # streamed, fp32 epilogue (the DMoL head)
    (128, 256, 1, False, False, False, 1),      # the 1x1 gate conv at 128 filters, N = 256 plain epilogue
    (128, 128, 1, True, False, False, 1),       # the merge 128 + 128 -> 128
    (128, 256, 3, False, False, False, 2),      # streamed, N = 256
]


@pytest.mark.parametrize("grid", GRIDS, ids=lambda g: "B%dx%dx%d" % g)
@pytest.mark.parametrize("case", FWD, ids=lambda c: "%d%s-%d-k%d%s%s" % (c[0], "x2" if c[3] else "", c[1], c[2],
                                                                         "-f32" if c[4] else "", "-res" if c[5] else ""))
def test_forward_exact(case, grid):
    cin, n, k, two, f32, res, plan = case
    B, H, W = grid
    if B == 256 and not (k == 3 and n in (128, 100)):
        pytest.skip("benchmark sizes: the 3x3 128 -> 128 convs and the head")
    assert tc_plan(cin, n, k, two, H, W, f32) == plan
    g = torch.Generator(device="cuda").manual_seed(cin * 7 + n + k + B)
    x = ints((B, H, W, cin), g)
    x2 = ints((B, H, W, cin), g) if two else None
    w = ints((n, cin * (2 if two else 1), k, k), g, torch.float32)
    bias = ints((n,), g, torch.float32)
    r = ints((B, H, W, n), g, torch.float32 if f32 else torch.bfloat16) if res else None
    odt = torch.float32 if f32 else torch.bfloat16
    y = Guarded((B, H, W, n), odt, zero=False)
    from lvae_b200 import ops
    s0 = ops.stats.get("tc_fwd_streamed", 0)
    _lib().call("lvae_conv2d_tc_ex", x.data_ptr(), _p(x2), pack(w, 2).data_ptr(), bias.data_ptr(), None, _p(r), y.t.data_ptr(),
                None, 0, B, H, W, cin, n, k, 0, int(f32), None, _stream())
    xin = torch.cat([x, x2], 3) if two else x
    ref = F.conv2d(xin.permute(0, 3, 1, 2).double(), w.double(), bias.double(), padding=k // 2).permute(0, 2, 3, 1)
    if r is not None:
        ref = ref + r.double()
    torch.cuda.synchronize()
    exact(y.t, ref, "forward")
    assert y.intact(), "write outside y"
    assert ops.stats.get("tc_fwd_streamed", 0) == s0          # a direct library call is not an ops route


# dgrad: (forward Cin, forward N, k, two inputs); the operand is dY (N channels, zero-padded to a multiple of 64), the output
# the forward's input gradient (split at Cin for the merge); last: the expected plan
DGRAD = [(128, 128, 3, False, 2), (128, 64, 3, False, 1), (128, 100, 3, False, 2), (128, 256, 1, False, 1),
         (128, 128, 1, True, 1)]


@pytest.mark.parametrize("grid", GRIDS, ids=lambda g: "B%dx%dx%d" % g)
@pytest.mark.parametrize("case", DGRAD, ids=lambda c: "%d%s-%d-k%d" % (c[0], "x2" if c[3] else "", c[1], c[2]))
def test_dgrad_exact(case, grid):
    cin_f, n_f, k, two, expect = case
    B, H, W = grid
    if B == 256 and not (n_f == 128 and k == 3):
        pytest.skip("benchmark sizes: the 3x3 128 -> 128 conv")
    cin_tot = cin_f * (2 if two else 1)
    gpad = (n_f + 63) // 64 * 64
    g = torch.Generator(device="cuda").manual_seed(cin_f + 3 * n_f + k + B)
    w = ints((n_f, cin_tot, k, k), g, torch.float32)
    gy = ints((B, H, W, gpad), g)
    gy[..., n_f:] = 0
    assert tc_plan(gpad, cin_tot, k, False, H, W, False) == expect
    if two:
        y = Guarded((B, H, W, cin_f), torch.bfloat16, zero=False)
        y2 = Guarded((B, H, W, cin_f), torch.bfloat16, zero=False)
    else:
        y, y2 = Guarded((B, H, W, cin_tot), torch.bfloat16, zero=False), None
    _lib().call("lvae_conv2d_tc_ex", gy.data_ptr(), None, pack(w, 3).data_ptr(), None, None, None, y.t.data_ptr(),
                y2.t.data_ptr() if two else None, cin_f if two else 0, B, H, W, gpad, cin_tot, k, 1, 0, None, _stream())
    ref = F.conv_transpose2d(gy[..., :n_f].permute(0, 3, 1, 2).double(), w.double(), padding=k // 2).permute(0, 2, 3, 1)
    torch.cuda.synchronize()
    if two:
        exact(y.t, ref[..., :cin_f], "dgrad (first input)")
        exact(y2.t, ref[..., cin_f:], "dgrad (second input)")
        assert y.intact() and y2.intact()
    else:
        exact(y.t, ref, "dgrad")
        assert y.intact()


# weight gradient: (xC per input, N, k, two inputs, dY channels): every (X window, dY window) launch the ops plan issues
WGRAD = [(128, 128, 3, False, 128), (128, 64, 3, False, 64), (128, 256, 1, False, 256), (128, 128, 1, True, 128),
         (128, 100, 3, False, 128)]
WGRIDS = [(1, 8, 8), (3, 16, 16), (256, 32, 32)]


@pytest.mark.parametrize("grid", WGRIDS, ids=lambda g: "B%dx%dx%d" % g)
@pytest.mark.parametrize("case", WGRAD, ids=lambda c: "%d%s-%d-k%d" % (c[0], "x2" if c[3] else "", c[1], c[2]))
def test_wgrad_windows_exact(case, grid):
    from lvae_b200 import ops
    xc, n, k, two, dyc = case
    B, H, W = grid
    if B == 256 and not (n == 128 and k == 3):
        pytest.skip("benchmark sizes: the 3x3 128 -> 128 conv")
    if n == 100:                                   # the DMoL head: dY zero-padded to 128, windows of 64 + 36 rows
        wins = [(x0, 64, c0) for x0 in (0, 64) for c0 in (0, 64)]
    else:
        wins = list(ops.wgrad_tc_windows(n, k, two, xc))
    assert len({x0 for x0, _, _ in wins}) == xc // 64 and wins
    g = torch.Generator(device="cuda").manual_seed(xc + n + k + B + two)
    x = ints((B, H, W, xc), g)
    x2 = ints((B, H, W, xc), g) if two else None
    gy = ints((B, H, W, dyc), g)
    gy[..., n:] = 0
    cin = xc * (2 if two else 1)
    dw = Guarded((n, cin, k, k), torch.float32)
    db = Guarded((n,), torch.float32)
    ws = torch.empty(512 * 128, dtype=torch.float32, device="cuda")
    row = cin * k * k
    for x0, nw, c0 in wins:
        _lib().call("lvae_conv2d_wgrad_tc_ex", x.data_ptr(), _p(x2), gy.data_ptr(), dw.t.data_ptr() + 4 * c0 * row,
                    None if x0 else db.t.data_ptr() + 4 * c0, ws.data_ptr(), B, H, W, nw, k, 0, min(nw, n - c0), dyc, c0,
                    xc, x0, _stream())
    xin = (torch.cat([x, x2], 3) if two else x).permute(0, 3, 1, 2).double()
    g64 = gy[..., :n].permute(0, 3, 1, 2).double()
    ref_w = torch.nn.grad.conv2d_weight(xin, (n, cin, k, k), g64, padding=k // 2)
    torch.cuda.synchronize()
    exact(dw.t, ref_w, "dw")
    exact(db.t, g64.sum((0, 2, 3)), "dbias (exactly once per dY window)")
    assert dw.intact() and db.intact()


# ------------------------------------------------------------------------------------------------ model and engine
def wide_cfg(lik):
    return small_cfg(n_filters=128, z_dims=[32, 64], img_shape=(16, 16), downsample=[0, 1], dropout=0.2,
                     color_ch=1 if lik == "bernoulli" else 3, likelihood_form=lik)


def _model(cfg, seed):
    import lvae_b200
    m = lvae_b200.LadderVAE(**cfg.kwargs())
    m.load_state_dict(O.make_params(cfg, seed), strict=True)
    return m.cuda().train()


def _step(model, cfg, x, eps, masks):
    import lvae_b200
    with lvae_b200.inject(eps=[e.float().cuda() for e in eps[0]], masks=[m.float().cuda() for m in masks]):
        out = model(x.float().cuda())
    loss = (-out["ll"]).mean() + out["kl_loss"]
    loss.backward()
    torch.cuda.synchronize()
    return out, loss


@pytest.mark.parametrize("lik", ["bernoulli", "discr_log_mix"])
def test_wide_model_fp32_matches_oracle_and_bf16_runs_on_tensor_cores(lik):
    from lvae_b200 import ops
    from lvae_b200.lib.nn import Conv2d, ConvTranspose2d
    cfg = wide_cfg(lik)
    B = 8
    x, eps, masks = make_inputs(cfg, B, 5, True)
    # fp32 parity mode against the float64 oracle
    m32 = _model(cfg, 3)
    out32, loss32 = _step(m32, cfg, x, eps, masks)
    st = O.TrainState(cfg, O.make_params(cfg, 3, torch.float64))
    o2, t2 = st.step(x, eps[0], masks, update=False)
    assert rel_err(loss32, t2["loss"]) < 1e-4
    assert rel_err(out32["kl_sep"], o2["kl_sep"]) < 1e-4 and rel_err(out32["ll"], o2["ll"]) < 1e-4
    gmax = max(float(st.P[n].grad.abs().max()) for n in st.names if st.P[n].grad is not None)
    for n, p in m32.named_parameters():
        gr = st.P[n].grad
        if gr is not None:
            err = float((p.grad.double().cpu() - gr).abs().max())
            assert err < 1e-3 * max(float(gr.abs().max()), 1e-3 * gmax), (n, err)
    # bf16 on the tensor cores, against the fp32 mode
    m16 = _model(cfg, 3)
    m16.set_compute_dtype(torch.bfloat16)
    for k in list(ops.stats):
        ops.stats[k] = 0
    out16, loss16 = _step(m16, cfg, x, eps, masks)
    e_ll, e_kl, e_loss = rel_err(out16["ll"], out32["ll"]), rel_err(out16["kl_sep"], out32["kl_sep"]), rel_err(loss16, loss32)
    p32 = dict(m32.named_parameters())
    names = [n for n, p in m16.named_parameters() if p.grad is not None]
    n16 = torch.tensor([float(dict(m16.named_parameters())[n].grad.double().norm()) for n in names])
    n32 = torch.tensor([float(p32[n].grad.double().norm()) for n in names])
    e_g = float((n16 - n32).abs().max() / n32.max())
    assert e_ll < 2e-2 and e_kl < 2e-2 and e_loss < 2e-2 and e_g < 5e-2, (e_ll, e_kl, e_loss, e_g)
    # routes: every stride-1 1x1 / 3x3 conv forward on tcgen05, only the stem and the stride-2 convs on the CUDA cores
    convs = [m for m in m16.modules() if isinstance(m, (Conv2d, ConvTranspose2d))]
    n_cc = sum(1 for m in convs if not m.spec.tc_shape)
    assert n_cc >= 3 and ops.stats["cc_fwd"] == n_cc, (ops.stats, n_cc)
    assert ops.stats.get("tc_fwd_streamed", 0) > 0 and ops.stats.get("tc_dgrad_streamed", 0) > 0
    assert ops.stats.get("tc_wgrad_xwin", 0) > 0
    # weight gradients: the CUDA-core ones are the stem, the stride-2 convs and the 128 -> 1 Bernoulli head (N = 1)
    assert ops.stats["cc_wgrad"] == n_cc + (1 if lik == "bernoulli" else 0), ops.stats


def test_64_filter_step_never_streams():
    from lvae_b200 import ops
    cfg = small_cfg(n_filters=64, z_dims=[32, 64], img_shape=(16, 16), downsample=[0, 1], dropout=0.2)
    x, eps, masks = make_inputs(cfg, 4, 5, True)
    m = _model(cfg, 3)
    m.set_compute_dtype(torch.bfloat16)
    for k in list(ops.stats):
        ops.stats[k] = 0
    _step(m, cfg, x, eps, masks)
    assert ops.stats["tc_fwd"] > 0 and ops.stats["tc_wgrad"] > 0
    assert ops.stats.get("tc_fwd_streamed", 0) == 0 and ops.stats.get("tc_dgrad_streamed", 0) == 0
    assert ops.stats.get("tc_wgrad_xwin", 0) == 0


def _engine_run(use_graph, side, steps=3, B=8):
    import lvae_b200
    from lvae_b200.engine import TrainEngine
    lvae_b200.manual_seed(7)
    cfg = wide_cfg("discr_log_mix")
    model = _model(cfg, 31)
    model.set_compute_dtype(torch.bfloat16)
    eng = TrainEngine(model, B, use_graph=use_graph, wgrad_side_stream=side)
    losses = []
    for i in range(steps):
        x, _, _ = make_inputs(cfg, B, 40 + i, True)
        losses.append(float(eng.step(x.float().cuda())["loss"]))
    torch.cuda.synchronize()
    return losses, eng.arena.flat.detach().clone()


def test_wide_engine_graph_replay_equals_eager():
    le, pe = _engine_run(False, False)
    lg, pg = _engine_run(True, True)
    for a, b in zip(le, lg):
        assert abs(a - b) <= 2e-4 * abs(a), (le, lg)
    d = (pe - pg).abs()
    assert float((d > 3e-5).float().mean()) < 5e-3, float(d.max())
    assert float(d.max()) <= 3 * 3e-4 * 2 + 1e-6


def test_wide_iw_evaluator_graph_equals_eager():
    import lvae_b200
    from lvae_b200.engine import IWEvaluator
    cfg = wide_cfg("discr_log_mix")
    model = _model(cfg, 23).eval()
    model.set_compute_dtype(torch.bfloat16)
    x, _, _ = make_inputs(cfg, 8, 2, False)
    xd = x.float().cuda()
    lvae_b200.manual_seed(6)
    bg = IWEvaluator(model, 8, use_graph=True).bound(xd, 5)
    lvae_b200.manual_seed(6)
    be = IWEvaluator(model, 8, use_graph=False).bound(xd, 5)
    assert bool(torch.isfinite(be).all())
    assert float((bg - be).abs().max()) < 1e-5 * abs(float(be.mean())) + 1e-4, (bg, be)
