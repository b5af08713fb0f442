"""CPU: routing of LadderVAE convolutions of every width onto the tensor-core kernels, and the argument checks of the wide
entry points.

For each width, every stride-1 conv of a LadderVAE is driven through ops.conv_forward_raw / conv_backward_raw with the
library calls recorded instead of issued: every lvae_conv2d_tc_ex launch must be a shape the library's own plan
(lvae_conv2d_tc_plan) accepts, resident at 64 filters; every weight-gradient launch must be a shape the kernel takes, its
X windows must tile the input channels and each dY window must add the bias gradient exactly once."""
import ctypes
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMMY = 0x1000          # non-null pointer that no check dereferences
WIDTHS = [16, 32, 64, 96, 128, 192, 256]


@pytest.fixture(scope="module")
def lib():
    import importlib.util
    spec = importlib.util.spec_from_file_location("lvae_build", os.path.join(ROOT, "ladder-vae-pytorch_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()
    import lvae_b200
    return lvae_b200._capi.lib()


def _model(width, lik):
    from oracle.make_golden import small_cfg
    import lvae_b200
    cfg = small_cfg(n_filters=width, z_dims=[32, 64], img_shape=(16, 16), downsample=[0, 1],
                    color_ch=1 if lik == "bernoulli" else 3, likelihood_form=lik)
    return lvae_b200.LadderVAE(**cfg.kwargs())


def _convs(model):
    """(module, two inputs) for every stride-1 1x1 / 3x3 conv; the merge convs read two equal halves."""
    from lvae_b200.lib.nn import Conv2d
    from lvae_b200.models.lvae_layers import MergeLayer
    merges = set()
    for m in model.modules():
        if isinstance(m, MergeLayer):
            merges.add(id(m.layer[0] if isinstance(m.layer, torch.nn.Sequential) else m.layer))
    return [(m, id(m) in merges) for m in model.modules() if isinstance(m, Conv2d) and m.spec.tc_shape]


def _drive(monkeypatch, spec, weight, bias, cin, two, out_f32=False):
    from lvae_b200 import ops
    calls = []
    monkeypatch.setattr(ops, "call", lambda name, *a: calls.append((name, a)))
    monkeypatch.setattr(ops, "_stream", lambda: None)
    ws = torch.empty(512 * 128)
    monkeypatch.setattr(ops, "_wgrad_workspace", lambda dev: ws)
    B, H, W = 2, 8, 8
    bf = lambda c: torch.zeros(B, H, W, c, dtype=torch.bfloat16)
    c1 = cin // 2 if two else cin
    xn, x2n = bf(c1), (bf(c1) if two else None)
    gw, gb = torch.zeros(weight.shape), torch.zeros(spec.cout)
    weight._lvae_grad_sink, bias._lvae_grad_sink = gw, gb
    try:
        ops.conv_forward_raw(spec, xn, x2n, weight, bias, None, None)
        ops.conv_backward_raw(spec, xn, x2n, weight, bias, None, bf(spec.cout), need_x=True)
    finally:
        del weight._lvae_grad_sink, bias._lvae_grad_sink
    return calls, gw, gb


@pytest.mark.parametrize("lik", ["bernoulli", "discr_log_mix"])
@pytest.mark.parametrize("width", WIDTHS)
def test_every_conv_takes_a_route_the_library_accepts(lib, monkeypatch, width, lik):
    from lvae_b200 import ops
    model = _model(width, lik)
    for m, two in _convs(model):
        sp = m.spec
        calls, gw, gb = _drive(monkeypatch, sp, m.weight, m.bias, sp.cin, two)
        tc = [a for n, a in calls if n == "lvae_conv2d_tc_ex"]
        for a in tc:
            Cin, N, k, out_f32 = a[12], a[13], a[14], a[16]
            plan = lib.lvae_conv2d_tc_plan(Cin, N, k, int(a[1] is not None), a[10], a[11], out_f32)
            assert plan in (ops.TC_RESIDENT, ops.TC_STREAMED), (width, sp.cin, sp.cout, sp.k, a[12:17])
            if width == 64:
                assert plan == ops.TC_RESIDENT
        if sp.cin % 64 == 0 and sp.cout % 64 == 0 and max(sp.cin, sp.cout) <= 256:
            assert len(tc) == 2, (width, sp.cin, sp.cout, sp.k)            # forward and dgrad on the tensor cores
        elif sp.cin % 64:
            assert all(a[15] == 1 for a in tc)                            # CUDA-core forward for other widths
        wins = [a for n, a in calls if n == "lvae_conv2d_wgrad_tc_ex"]
        ones = [a for n, a in calls if n == "lvae_conv2d_wgrad_tc"]
        for a in ones:
            assert lib.lvae_wgrad_tc_packed_size(a[9], a[10], int(a[1] is not None)) > 0
        if wins:
            xC = wins[0][15]
            row = sp.cin * sp.k * sp.k * 4
            bias_per_dy = {}
            for a in wins:
                N, k, dy_c0, x0 = a[9], a[10], a[14], a[16]
                assert lib.lvae_wgrad_tc_packed_size(N, k, int(a[1] is not None)) > 0
                assert a[15] == xC and x0 % 64 == 0 and x0 + 64 <= xC and xC == sp.cin // (2 if two else 1)
                assert a[3] == gw.data_ptr() + dy_c0 * row
                if a[4] is not None:
                    assert a[4] == gb.data_ptr() + dy_c0 * 4
                    bias_per_dy[dy_c0] = bias_per_dy.get(dy_c0, 0) + 1
            pairs = sorted((a[16], a[14]) for a in wins)
            dys = sorted({a[14] for a in wins})
            assert pairs == sorted((x0, c) for x0 in range(0, xC, 64) for c in dys)      # every (X, dY) window once
            assert sum(a[9] for a in wins if a[16] == 0) == sp.cout                      # dY windows tile N
            assert bias_per_dy == {c: 1 for c in dys}
        if width == 64:
            assert not wins


@pytest.mark.parametrize("width", WIDTHS)
def test_dmol_head_plans(lib, width):
    """The fused DMoL head takes 64 and 128 input channels; both of its tensor-core launches must be accepted."""
    from lvae_b200 import ops
    if width not in (64, 128):
        return
    H = W = 16
    assert ops.conv_tc_plan(width, 100, 3, False, H, W, True) != ops.TC_REJECTED
    assert ops.conv_tc_plan(128, width, 3, False, H, W, False) != ops.TC_REJECTED
    expect = ops.TC_RESIDENT if width == 64 else ops.TC_STREAMED
    assert ops.conv_tc_plan(width, 100, 3, False, H, W, True) == expect


@pytest.mark.parametrize("args,plan", [
    ((64, 64, 3, 0, 32, 32, 0), 1), ((64, 128, 1, 0, 32, 32, 0), 1), ((64, 64, 1, 1, 32, 32, 0), 1),
    ((64, 100, 3, 0, 32, 32, 1), 1), ((64, 128, 3, 0, 32, 32, 0), 1),
    ((128, 128, 3, 0, 16, 16, 0), 2), ((128, 100, 3, 0, 16, 16, 1), 2), ((128, 64, 3, 0, 16, 16, 0), 1),
    ((128, 256, 1, 0, 16, 16, 0), 1), ((128, 128, 1, 1, 16, 16, 0), 1), ((256, 256, 3, 0, 16, 16, 0), 2),
    ((96, 64, 3, 0, 16, 16, 0), 0), ((320, 64, 1, 0, 16, 16, 0), 0), ((128, 128, 3, 1, 16, 16, 0), 2),
    ((256, 64, 3, 1, 16, 16, 0), 0), ((64, 64, 5, 0, 16, 16, 0), 0), ((64, 64, 3, 0, 16, 12, 0), 0),
    ((64, 64, 3, 0, 16, 256, 0), 0), ((64, 300, 3, 0, 16, 16, 0), 0)])
def test_conv_plan(lib, args, plan):
    assert lib.lvae_conv2d_tc_plan(*args) == plan


def test_fused_epilogue_on_streamed_weights_is_rejected(lib):
    import lvae_b200
    f = lvae_b200._capi.ConvFuse()
    f.stats_acc = DUMMY
    rc = lib.lvae_conv2d_tc_ex(DUMMY, None, DUMMY, None, None, None, DUMMY, None, 0, 2, 16, 16, 128, 128, 3, 0, 0,
                               ctypes.addressof(f), None)
    assert rc != 0 and "fused epilogues need resident weights" in lib.lvae_last_error().decode()


@pytest.mark.parametrize("xC,x_c0,what", [
    (128, -64, "negative X channel window"),
    (128, 32, "X channel window not 64-aligned"),
    (128, 128, "X channel window past the 128 input channels"),
    (64, 64, "X channel window past the 64 input channels"),
    (96, 0, "X channel window past the 96 input channels"),
])
def test_windowed_wgrad_rejects_bad_windows_before_any_device_call(lib, xC, x_c0, what):
    rc = lib.lvae_conv2d_wgrad_tc_ex(DUMMY, None, DUMMY, DUMMY, DUMMY, DUMMY, 2, 8, 8, 64, 3, 0, 0, 0, 0, xC, x_c0, None)
    assert rc != 0
    assert what in lib.lvae_last_error().decode(), lib.lvae_last_error().decode()


def test_windowed_wgrad_checks_input_rows_against_the_full_width(lib):
    rc = lib.lvae_conv2d_wgrad_tc_ex(DUMMY, None, DUMMY, DUMMY, DUMMY, DUMMY, 2, 8, 8, 64, 3, 129, 0, 0, 0, 128, 64, None)
    assert rc != 0 and lib.lvae_last_error().decode().startswith("conv2d_wgrad_tc: I_real 129")


@pytest.mark.parametrize("N,k,two,xC,expect", [
    (128, 3, False, 128, [(0, 64, 0), (0, 64, 64), (64, 64, 0), (64, 64, 64)]),
    (256, 1, False, 128, [(0, 128, 0), (0, 128, 128), (64, 128, 0), (64, 128, 128)]),
    (128, 1, True, 128, [(0, 128, 0), (64, 128, 0)]),
    (64, 3, False, 128, [(0, 64, 0), (64, 64, 0)]),
    (100, 3, False, 128, []),
    (128, 3, True, 128, []),
])
def test_wgrad_windows(lib, N, k, two, xC, expect):
    from lvae_b200 import ops
    assert list(ops.wgrad_tc_windows(N, k, two, xC)) == expect
