"""GPU: every route of the tcgen05 weight gradient (csrc/wgrad_tcgen05.cu) against a float64 reference of the same operands.

With operands drawn from the bf16 integers {-2, ..., 2} every product is exact and every partial sum is an integer of at most
2^20 (the largest case reduces over 2^18 pixels), so the TMEM accumulation, the L2 reduce-adds of the CTAs and the unpack's
+= are exact in any order: the kernel must equal the float64 reference bit for bit, and a dropped or doubled tile, a wrong
tap, halo offset or channel fails outright instead of hiding inside a tolerance.  One Gaussian case per route at a benchmark
shape checks realistic data against fp32 accumulation error (relative 1e-5).  Every dw / dbias sits inside a larger buffer
filled with a sentinel that must survive the call.

Routes: the one-call form (lvae_conv2d_wgrad_tc: halo tiles, non-halo tiles, the 1x1 gate and the two-input merge, I_real
below 64, dY channel windows with N_real below N), the stride-2 resampling convs (Conv2d and ConvTranspose2d, one-call and
_acc), and the engine's packed route (_acc reduce-adds, then one batched unpack of mixed descriptors with the clear and
overwrite bits)."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from lvae_test_helpers import rel_err

pytestmark = pytest.mark.gpu

SENT = -12345.5          # fills the guard zones around every dw / dbias
GUARD = 2048             # floats of guard zone on each side
WG_TILES_PER_CTA = 8     # csrc/wgrad_tcgen05.cu


def _capi():
    import lvae_b200
    return lvae_b200._capi


def _call(name, *args):
    _capi().call(name, *args)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def operand(shape, gen, kind):
    """NHWC bf16 operand on the device: integers in {-2, ..., 2} ("int") or standard normal ("gauss")."""
    if kind == "int":
        t = torch.randint(-2, 3, shape, generator=gen, device="cuda", dtype=torch.int32).float()
    else:
        t = torch.randn(shape, generator=gen, device="cuda")
    return t.to(torch.bfloat16)


class Guarded:
    """A float32 tensor of n elements in the middle of a sentinel-filled buffer."""

    def __init__(self, shape, init=None):
        n = 1
        for s in shape:
            n *= s
        self.n = n
        self.buf = torch.full((n + 2 * GUARD,), SENT, dtype=torch.float32, device="cuda")
        self.t = self.buf[GUARD:GUARD + n].view(shape)
        if init is None:
            self.t.zero_()
        else:
            self.t.copy_(init)

    def ptr(self, offset_floats=0):
        return self.t.data_ptr() + 4 * offset_floats

    def assert_guard_intact(self):
        lo, hi = self.buf[:GUARD], self.buf[GUARD + self.n:]
        assert bool((lo == SENT).all()) and bool((hi == SENT).all()), "write outside the gradient buffer"


def check(got, ref, kind, what):
    got, ref = got.double(), ref.double().to(got.device)
    if kind == "int":
        bad = got != ref
        assert not bool(bad.any()), "%s: %d of %d entries differ, max |diff| %g" % (
            what, int(bad.sum()), bad.numel(), float((got - ref).abs().max()))
    else:
        assert rel_err(got, ref) < 1e-5, (what, rel_err(got, ref))


def nchw64(t):
    return t.double().permute(0, 3, 1, 2).contiguous()


def ref_wgrad(x, dy, k, x2=None, cin=None, cols=None, stride=1):
    """float64 (dw, dbias) of a k x k Conv2d with padding k // 2: x (and x2) NHWC input, dy NHWC output gradient; cin: the
    input channels of dw (the rest of x is padding), cols: the dY channels that are the conv's outputs."""
    xi = torch.cat([x, x2], 3) if x2 is not None else x
    xi = nchw64(xi)
    if cin is not None:
        xi = xi[:, :cin].contiguous()
    g = nchw64(dy)
    if cols is not None:
        g = g[:, cols].contiguous()
    dw = torch.nn.grad.conv2d_weight(xi, (g.shape[1], xi.shape[1], k, k), g, stride=stride, padding=k // 2)
    return dw, g.sum((0, 2, 3))


def ref_wgrad_transposed(c, dy):
    """float64 (dw, dbias) of ConvTranspose2d(64, 64, 3, stride 2, padding 1, output_padding 1): c the input, dy the gradient
    of its output (both NHWC)."""
    w = torch.zeros(64, 64, 3, 3, dtype=torch.float64, device="cuda", requires_grad=True)
    y = F.conv_transpose2d(nchw64(c), w, stride=2, padding=1, output_padding=1)
    y.backward(nchw64(dy))
    return w.grad, nchw64(dy).sum((0, 2, 3))


def packed_size(N, k, two):
    return int(_capi().lib().lvae_wgrad_tc_packed_size(N, k, int(two)))


def geometry(B, H, W, N, k, two, stride, n_sms):
    """Pixel tiles, tiles per CTA and grid of one launch, by the host's formula in wgrad_tc_acc_impl."""
    halo = stride == 1 and k == 3 and not two and N == 64 and W % 8 == 0 and H % 16 == 0
    n_tiles = B * (W // 8) * (H // 16) if halo else -(-B * H * W // 128)
    grid = max(1, min(-(-n_tiles // WG_TILES_PER_CTA), n_sms))
    tpc = -(-n_tiles // grid)
    grid = -(-n_tiles // tpc)
    return dict(halo=halo, n_tiles=n_tiles, tiles_per_cta=tpc, grid=grid, capped=-(-n_tiles // WG_TILES_PER_CTA) > n_sms,
                uneven=n_tiles % tpc != 0)


# ----------------------------------------------------------------------------------------------------- one-call routes
# (B, H, W, N, ksize, two inputs, I_real)
ONE_CALL = [
    # 3x3, N = 64, halo tiles (16 x 8 pixels)
    (256, 32, 32, 64, 3, False, 0),      # the CIFAR bench's last top-down rung: 2048 tiles, 147 CTAs of 14, the last of 4
    (256, 16, 16, 64, 3, False, 0),
    (3, 32, 32, 64, 3, False, 0),
    (2, 16, 128, 64, 3, False, 0),
    (5, 16, 8, 64, 3, False, 0),
    # 3x3, N = 64, 128-pixel tiles spanning images
    (256, 2, 2, 64, 3, False, 0),
    (40, 2, 2, 64, 3, False, 0),         # 160 pixels: partial second tile
    (3, 4, 4, 64, 3, False, 0),          # 48 pixels
    (2, 8, 8, 64, 3, False, 0),
    (7, 1, 1, 64, 3, False, 0),          # every tap but the centre reads padding
    (1, 1, 128, 64, 3, False, 0),
    # 1x1 gate, N = 128
    (256, 16, 16, 128, 1, False, 0),
    (3, 4, 4, 128, 1, False, 0),
    (40, 2, 2, 128, 1, False, 0),
    # 1x1 merge over two inputs, N = 64
    (256, 16, 16, 64, 1, True, 0),
    (3, 4, 4, 64, 1, True, 0),
    (40, 2, 2, 64, 1, True, 0),
    # 3x3 over the zero-padded 64-channel copy of a 32-channel z (conv_out of a stochastic block)
    (4, 16, 16, 64, 3, False, 32),
    (6, 4, 4, 64, 3, False, 32),
]
# dY 128 channels wide, 100 real (the DMoL head): two launches of 64 output channels
DY_WINDOW = [(4, 32, 32), (3, 4, 4)]
# stride-2 resampling convs: small grid (Hg, Wg, B)
S2_GRIDS = [(1, 1, 70), (2, 2, 40), (8, 8, 256), (16, 16, 64), (4, 64, 2)]


def _case_id(c):
    B, H, W, N, k, two, I_real = c
    return "%dx%dx%d_N%d_k%d%s%s" % (B, H, W, N, k, "_two" if two else "", "_I%d" % I_real if I_real else "")


def run_one_call(case, kind, seed):
    B, H, W, N, k, two, I_real = case
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = operand((B, H, W, 64), g, kind)
    if I_real:
        x[..., I_real:] = 0
    x2 = operand((B, H, W, 64), g, kind) if two else None
    dy = operand((B, H, W, N), g, kind)
    cin = I_real or (128 if two else 64)
    dw, db = Guarded((N, cin, k, k)), Guarded((N,))
    ws = torch.full((packed_size(N, k, two),), float("nan"), device="cuda")      # scratch: the call clears it
    _call("lvae_conv2d_wgrad_tc", x.data_ptr(), _p(x2), dy.data_ptr(), dw.ptr(), db.ptr(), ws.data_ptr(), B, H, W, N, k,
          I_real, 0, 0, 0, _stream())
    torch.cuda.synchronize()
    rw, rb = ref_wgrad(x, dy, k, x2, cin=cin)
    check(dw.t, rw, kind, "dw")
    check(db.t, rb, kind, "dbias")
    dw.assert_guard_intact()
    db.assert_guard_intact()


@pytest.mark.parametrize("case", ONE_CALL, ids=_case_id)
def test_one_call_exact(case):
    run_one_call(case, "int", 11 + sum(case[:5]))


def run_dy_window(shape, kind, seed):
    """DmolHeadFn's weight gradient: dY (B,H,W,128) with channels 100..127 zero, launches dy_c0 = 0 (N_real 64) and
    dy_c0 = 64 (N_real 36) into rows 0.. and 64.. of one (100, 64, 3, 3) gradient."""
    B, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = operand((B, H, W, 64), g, kind)
    dy = operand((B, H, W, 128), g, kind)
    dy[..., 100:] = 0
    dw, db = Guarded((100, 64, 3, 3)), Guarded((100,))
    ws = torch.empty((packed_size(64, 3, False),), device="cuda")
    for c0 in (0, 64):
        _call("lvae_conv2d_wgrad_tc", x.data_ptr(), None, dy.data_ptr(), dw.ptr(c0 * 64 * 9), db.ptr(c0), ws.data_ptr(),
              B, H, W, 64, 3, 0, min(64, 100 - c0), 128, c0, _stream())
    torch.cuda.synchronize()
    rw, rb = ref_wgrad(x, dy, 3, cols=slice(0, 100))
    check(dw.t, rw, kind, "dw")
    check(db.t, rb, kind, "dbias")
    dw.assert_guard_intact()
    db.assert_guard_intact()


@pytest.mark.parametrize("shape", DY_WINDOW)
def test_dy_window_exact(shape):
    run_dy_window(shape, "int", 5 + sum(shape))


# ----------------------------------------------------------------------------------------------------- stride 2
def _unpack_table(descs):
    """Device table of unpack descriptors: descs = [(gp, dw_ptr, dbias_ptr, N, k, two, I_real, N_real, clear)]."""
    lib = _capi().lib()
    dsz = int(lib.lvae_wgrad_unpack_desc_size())
    host = ctypes.create_string_buffer(dsz * len(descs))
    for i, (gp, dwp, dbp, N, k, two, I_real, N_real, clear) in enumerate(descs):
        _call("lvae_wgrad_unpack_desc", ctypes.addressof(host) + i * dsz, gp.data_ptr(), dwp, dbp, N, k, int(two), I_real,
              N_real, clear)
    return torch.frombuffer(bytearray(host.raw), dtype=torch.uint8).cuda()


def run_s2(grid, transposed, form, kind, seed):
    Hg, Wg, B = grid
    g = torch.Generator(device="cuda").manual_seed(seed)
    big = operand((B, 2 * Hg, 2 * Wg, 64), g, kind)
    small = operand((B, Hg, Wg, 64), g, kind)
    # Conv2d: xs = the input (big), c = dY (small).  ConvTranspose2d: xs = dY (big), c = the input (small).
    dw, db = Guarded((64, 64, 3, 3)), Guarded((64,))
    dbp = None if transposed else db.ptr()
    if form == "one_call":
        ws = torch.full((packed_size(64, 3, False),), float("nan"), device="cuda")
        _call("lvae_conv2d_wgrad_tc_s2", big.data_ptr(), small.data_ptr(), dw.ptr(), dbp, ws.data_ptr(), B, Hg, Wg, _stream())
        gp = None
    else:
        gp = torch.zeros((packed_size(64, 3, False),), device="cuda")
        _call("lvae_conv2d_wgrad_tc_s2_acc", big.data_ptr(), small.data_ptr(), gp.data_ptr(), B, Hg, Wg, _stream())
        tab = _unpack_table([(gp, dw.ptr(), dbp, 64, 3, False, 64, 64, 1)])
        _call("lvae_wgrad_unpack_batched", tab.data_ptr(), 1, 64, _stream())
    if transposed:       # the bias gradient of a ConvTranspose2d sums its (large) output grid
        _call("lvae_colsum", big.data_ptr(), None, db.ptr(), B, 4 * Hg * Wg, 64, 1, _stream())
    torch.cuda.synchronize()
    if transposed:
        rw, rb = ref_wgrad_transposed(small, big)
    else:
        rw, rb = ref_wgrad(big, small, 3, stride=2)
    check(dw.t, rw, kind, "dw")
    check(db.t, rb, kind, "dbias")
    dw.assert_guard_intact()
    db.assert_guard_intact()
    if gp is not None:
        assert not bool(gp.any()), "the unpack's clear bit left the packed gradient non-zero"


@pytest.mark.parametrize("form", ["one_call", "acc"])
@pytest.mark.parametrize("transposed", [False, True], ids=["conv", "convT"])
@pytest.mark.parametrize("grid", S2_GRIDS, ids=lambda g: "%dx%dx%d" % g)
def test_stride2_exact(grid, transposed, form):
    run_s2(grid, transposed, form, "int", 3 + sum(grid) + int(transposed))


# ----------------------------------------------------------------------------------------------------- packed route
def _packed_convs():
    """(name, B, H, W, N, k, two, I_real, N_real, dyC, dy_c0) of the mixed table: 3x3 N = 64, 1x1 N = 128, two-input 1x1,
    3x3 with I_real = 32, and the DMoL head's second window (dY channels 64..99 of 128: N_real = 36)."""
    return [("3x3", 8, 16, 16, 64, 3, False, 0, 0, 0, 0),
            ("gate", 40, 2, 2, 128, 1, False, 0, 0, 0, 0),
            ("merge", 4, 16, 16, 64, 1, True, 0, 0, 0, 0),
            ("zpad", 5, 16, 8, 64, 3, False, 32, 0, 0, 0),
            ("head", 2, 32, 32, 64, 3, False, 0, 36, 128, 64)]


def _packed_operands(conv, g, kind):
    name, B, H, W, N, k, two, I_real, N_real, dyC, dy_c0 = conv
    x = operand((B, H, W, 64), g, kind)
    x2 = operand((B, H, W, 64), g, kind) if two else None
    dy = operand((B, H, W, dyC or N), g, kind)
    if dyC:
        dy[..., dy_c0 + N_real:] = 0            # the head's zero padding channels 100..127
    # (I_real = 32: channels 32.. stay non-zero here; the unpack alone must drop their rows)
    cin = I_real or (128 if two else 64)
    rw, rb = ref_wgrad(x, dy, k, x2, cin=cin, cols=slice(dy_c0, dy_c0 + (N_real or N)))
    return (x, x2, dy), (rw, rb)


def _accumulate(conv, gp, ops_):
    name, B, H, W, N, k, two, I_real, N_real, dyC, dy_c0 = conv
    x, x2, dy = ops_
    _call("lvae_conv2d_wgrad_tc_acc", x.data_ptr(), _p(x2), dy.data_ptr(), gp.data_ptr(), B, H, W, N, k, dyC, dy_c0, _stream())


@pytest.mark.parametrize("kind", ["int", "gauss"])
def test_packed_route_as_the_engine_drives_it(kind):
    """Two _acc launches per conv into one packed buffer, then ONE batched unpack of a mixed descriptor table into preloaded
    gradients: dw == preload + g1 + g2, the clear bit leaves every packed buffer zero so that the next accumulate-and-unpack
    adds only the new gradient, and the overwrite bit replaces dw / dbias."""
    g = torch.Generator(device="cuda").manual_seed(77)
    convs = _packed_convs()
    sizes = [packed_size(c[4], c[5], c[6]) for c in convs]
    flat = torch.zeros(sum(sizes), device="cuda")
    gps = list(torch.split(flat, sizes))
    dws, dbs, refs = [], [], []
    for c in convs:
        name, B, H, W, N, k, two, I_real, N_real, dyC, dy_c0 = c
        rows, cin = N_real or N, I_real or (128 if two else 64)
        pre_w = torch.randint(-50, 51, (rows, cin, k, k), generator=g, device="cuda").float()
        pre_b = torch.randint(-50, 51, (rows,), generator=g, device="cuda").float()
        dws.append(Guarded((rows, cin, k, k), pre_w))
        dbs.append(Guarded((rows,), pre_b))
        refs.append([pre_w.double(), pre_b.double()])

    def table(clear):
        return _unpack_table([(gp, dw.ptr(), db.ptr(), c[4], c[5], c[6], c[7], c[8], clear)
                              for c, gp, dw, db in zip(convs, gps, dws, dbs)])

    def accumulate(times):
        for i, c in enumerate(convs):
            for _ in range(times):
                ops_, (rw, rb) = _packed_operands(c, g, kind)
                _accumulate(c, gps[i], ops_)
                refs[i][0] = refs[i][0] + rw
                refs[i][1] = refs[i][1] + rb

    def unpack_and_check(tab, what):
        _call("lvae_wgrad_unpack_batched", tab.data_ptr(), len(convs), 128, _stream())
        torch.cuda.synchronize()
        for c, dw, db, (rw, rb) in zip(convs, dws, dbs, refs):
            check(dw.t, rw, kind, "%s %s dw" % (what, c[0]))
            check(db.t, rb, kind, "%s %s dbias" % (what, c[0]))
            dw.assert_guard_intact()
            db.assert_guard_intact()
        assert not bool(flat.any()), "%s: the clear bit left packed gradients non-zero" % what

    tab = table(1)
    accumulate(2)
    unpack_and_check(tab, "preload + g1 + g2")
    accumulate(1)
    unpack_and_check(tab, "second step")
    for r in refs:                                   # overwrite: only the new gradient remains
        r[0], r[1] = torch.zeros_like(r[0]), torch.zeros_like(r[1])
    accumulate(1)
    unpack_and_check(table(3), "overwrite")


# ----------------------------------------------------------------------------------------------------- realistic data
GAUSS = [
    ("one_call", (256, 32, 32, 64, 3, False, 0)),
    ("one_call", (256, 2, 2, 64, 3, False, 0)),
    ("one_call", (256, 16, 16, 128, 1, False, 0)),
    ("one_call", (256, 16, 16, 64, 1, True, 0)),
    ("one_call", (64, 16, 16, 64, 3, False, 32)),
    ("dy_window", (64, 32, 32)),
    ("s2", ((8, 8, 256), False)),
    ("s2", ((8, 8, 256), True)),
]


@pytest.mark.parametrize("route,case", GAUSS, ids=lambda v: str(v).replace(" ", "") if not isinstance(v, str) else v)
def test_gaussian_operands_at_bench_shapes(route, case):
    if route == "one_call":
        run_one_call(case, "gauss", 101)
    elif route == "dy_window":
        run_dy_window(case, "gauss", 102)
    else:
        run_s2(case[0], case[1], "one_call", "gauss", 103)


# ----------------------------------------------------------------------------------------------------- tile counts
def test_case_tables_reach_the_benchmark_tile_counts():
    """The launches above include a grid capped at the SM count with more than WG_TILES_PER_CTA tiles per CTA, a last CTA
    with fewer tiles than the others, and a single-CTA launch (host formula, this device's SM count)."""
    n_sms = torch.cuda.get_device_properties(0).multi_processor_count
    geos = [geometry(B, H, W, N, k, two, 1, n_sms) for B, H, W, N, k, two, _ in ONE_CALL]
    geos += [geometry(B, H, W, 64, 3, False, 1, n_sms) for B, H, W in DY_WINDOW]
    geos += [geometry(B, Hg, Wg, 64, 3, False, 2, n_sms) for Hg, Wg, B in S2_GRIDS]
    assert any(g["capped"] and g["tiles_per_cta"] > WG_TILES_PER_CTA for g in geos)
    assert any(g["capped"] and g["uneven"] for g in geos)
    assert any(g["grid"] == 1 for g in geos)
    assert any(g["halo"] and g["capped"] for g in geos) and any(not g["halo"] and g["n_tiles"] > 1 for g in geos)
    bench = geometry(256, 32, 32, 64, 3, False, 1, n_sms)
    if n_sms == 148:
        assert (bench["n_tiles"], bench["grid"], bench["tiles_per_cta"]) == (2048, 147, 14)


# ----------------------------------------------------------------------------------------------------- modules
def test_conv2d_64_to_128_3x3_bf16_forward_backward_exact():
    """conv_in_q / conv_in_p of a 64-dimensional latent layer: Conv2d(64, 128, 3) in bf16.  Its weight gradient does not fit
    one launch (5 pairs x 128 TMEM columns); it runs as two N = 64 launches over dY channel windows."""
    import lvae_b200  # noqa: F401
    from lvae_b200 import ops
    from lvae_b200.lib.nn import Conv2d
    g = torch.Generator(device="cuda").manual_seed(64128)
    B, H, W = 6, 16, 16
    mod = Conv2d(64, 128, 3, padding=1).cuda()
    mod.spec.out_fp32 = True                  # as LadderVAE.set_compute_dtype sets it for conv_in_q / conv_in_p
    w = torch.randint(-2, 3, mod.weight.shape, generator=g, device="cuda").float()
    b = torch.randint(-2, 3, (128,), generator=g, device="cuda").float()
    with torch.no_grad():
        mod.weight.copy_(w)
        mod.bias.copy_(b)
    x = operand((B, H, W, 64), g, "int")
    gy = operand((B, H, W, 128), g, "int")
    xr = nchw64(x).requires_grad_(True)
    wr, br = w.double().requires_grad_(True), b.double().requires_grad_(True)
    yr = F.conv2d(xr, wr, br, padding=1)
    yr.backward(nchw64(gy))
    xd = x.permute(0, 3, 1, 2).requires_grad_(True)          # logical NCHW view of the NHWC tensor
    before = dict(ops.stats)
    y = mod(xd)
    assert y.dtype == torch.float32
    check(y, yr.detach(), "int", "forward")
    y.backward(gy.permute(0, 3, 1, 2).float())
    torch.cuda.synchronize()
    assert ops.stats["tc_wgrad"] == before["tc_wgrad"] + 1 and ops.stats["cc_wgrad"] == before["cc_wgrad"]
    check(mod.weight.grad, wr.grad, "int", "dw")
    check(mod.bias.grad, br.grad, "int", "dbias")
    # the data gradient is rounded to bf16 once: within half a bf16 unit of the exact value
    gx, gxr = xd.grad.double(), xr.grad
    assert bool(((gx - gxr).abs() <= gxr.abs() * 2.0 ** -8).all())


def _small_bf16_model(z_dims, seed):
    import lvae_b200
    from oracle import lvae_oracle as O
    from oracle.make_golden import small_cfg
    cfg = small_cfg(n_filters=64, z_dims=z_dims, downsample=[0] + [1] * (len(z_dims) - 1), dropout=0.2)
    model = lvae_b200.LadderVAE(**cfg.kwargs())
    model.load_state_dict(O.make_params(cfg, seed))
    return cfg, model.cuda().train().set_compute_dtype(torch.bfloat16)


def test_engine_step_packed_gradients_match_the_one_call_route(monkeypatch):
    """One eager TrainEngine step of a small bf16 model with side streams: every packed gradient the backward issues is
    unpacked, every conv that owns one issues it, the packed buffers are clear afterwards, and the gradients that reach the
    arena match the same forward and backward run without the engine (one-call route).  The forward kernels are the same;
    only the order of the double-precision BatchNorm atomics can flip a bf16 rounding, hence 1e-3 relative L2."""
    import lvae_b200
    from lvae_b200 import ops
    from lvae_b200.engine import TrainEngine
    from lvae_b200.lib.nn import Conv2d, ConvTranspose2d
    from oracle.make_golden import make_inputs
    cfg, model = _small_bf16_model([32, 32, 32], 41)
    _, ref_model = _small_bf16_model([32, 32, 32], 41)
    B = 8
    x, eps, masks = make_inputs(cfg, B, 9, True)
    noise = lambda: dict(eps=[e.float().cuda() for e in eps[0]], masks=[m.float().cuda() for m in masks])

    eng = TrainEngine(model, B, use_graph=False, wgrad_side_stream=True)
    owners = {n: m for n, m in model.named_modules()
              if isinstance(m, (Conv2d, ConvTranspose2d)) and hasattr(m.weight, "_lvae_gp")}
    assert eng.gpacks.n == len(owners) > 10
    logged, unpacked = [], []
    join = ops.join_side_stream
    monkeypatch.setattr(ops, "join_side_stream",
                        lambda: (logged.extend(i for ids in ops.packed_grad_log().values() for i in ids), join())[1])
    unpack = eng.gpacks.unpack
    monkeypatch.setattr(eng.gpacks, "unpack", lambda ids=None: (unpacked.extend(ids), unpack(ids))[1])
    with lvae_b200.inject(**noise()):
        out = eng.step(x.float().cuda())
    torch.cuda.synchronize()
    assert torch.isfinite(out["loss"]).all()
    assert len(logged) == len(set(logged)) and sorted(unpacked) == sorted(logged)     # each issued id unpacked once
    assert set(logged) == {m.weight._lvae_gp_id for m in owners.values()}
    assert not bool(eng.gpacks.flat.any()), "packed gradients not cleared by the unpack"

    with lvae_b200.inject(**noise()):
        o = ref_model(x.float().cuda())
    ((-o["ll"]).mean() + o["kl_loss"]).backward()
    torch.cuda.synchronize()
    ref_mods = dict(ref_model.named_modules())
    l2 = lambda t: float(t.double().norm())
    for name, m in owners.items():
        r = ref_mods[name]
        gw, rw = m.weight._lvae_grad_sink, r.weight.grad
        assert l2(gw - rw) <= 1e-3 * l2(rw), (name, l2(gw - rw) / l2(rw))
        if m.bias is not None:
            # a conv bias in front of a train-mode BatchNorm has a true gradient of zero: bound it by the weight's scale
            gb, rb = m.bias._lvae_grad_sink, r.bias.grad
            assert l2(gb - rb) <= 1e-3 * max(l2(rb), l2(rw)), (name, l2(gb - rb), l2(rb))


def test_engine_step_with_a_64_dimensional_latent_layer(monkeypatch):
    """bf16 training of a model with a 64-dimensional latent layer: its conv_in_q is Conv2d(64, 128, 3), whose weight gradient
    takes the tensor cores as two launches over dY channel windows into the gradient arena."""
    import lvae_b200
    from lvae_b200 import ops
    from lvae_b200.engine import TrainEngine
    from oracle.make_golden import make_inputs
    cfg, model = _small_bf16_model([32, 64], 43)
    eng = TrainEngine(model, 4, use_graph=False, wgrad_side_stream=True)
    conv = [m for n, m in model.named_modules() if n.endswith("conv_in_q") and m.spec.cout == 128]
    assert len(conv) == 1
    sink = conv[0].weight._lvae_grad_sink.data_ptr()
    seen = []
    call = ops.call
    monkeypatch.setattr(ops, "call", lambda name, *a: (seen.append((name, a)) if name == "lvae_conv2d_wgrad_tc" else None,
                                                       call(name, *a))[1])
    x, eps, masks = make_inputs(cfg, 4, 3, True)
    with lvae_b200.inject(eps=[e.float().cuda() for e in eps[0]], masks=[m.float().cuda() for m in masks]):
        out = eng.step(x.float().cuda())
    torch.cuda.synchronize()
    assert torch.isfinite(out["loss"]).all()
    mine = [(a[3] - sink, a[9], a[13], a[14]) for _, a in seen if sink <= a[3] < sink + conv[0].weight.numel() * 4]
    assert sorted(mine) == [(0, 64, 128, 0), (64 * 64 * 9 * 4, 64, 128, 64)]
    assert float(conv[0].weight._lvae_grad_sink.abs().max()) > 0
