"""CPU: argument checks of the tensor-core weight-gradient entry points and the routing that feeds them.

The checks run on the host and return before any CUDA call, so a bad I_real / N_real / dY window is refused here without a
device.  The routing tests drive ops.conv_backward_raw with the library calls recorded instead of issued: every shape it
sends to lvae_conv2d_wgrad_tc[_acc] must be one the kernel accepts (lvae_wgrad_tc_packed_size > 0), and the engine's
PackedGradArena must give a packed gradient to exactly the single-launch shapes."""
import ctypes
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMMY = 0x1000          # non-null pointer that no check dereferences


@pytest.fixture(scope="module")
def libpath():
    import importlib.util
    spec = importlib.util.spec_from_file_location("lvae_build", os.path.join(ROOT, "ladder-vae-pytorch_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.build()


@pytest.fixture(scope="module")
def lib(libpath):
    import lvae_b200
    return lvae_b200._capi.lib()


def _desc(lib, N, k, two, I_real, N_real):
    buf = ctypes.create_string_buffer(int(lib.lvae_wgrad_unpack_desc_size()))
    return lib.lvae_wgrad_unpack_desc(ctypes.addressof(buf), DUMMY, DUMMY, DUMMY, N, k, two, I_real, N_real, 1)


@pytest.mark.parametrize("N,k,two,I_real,N_real", [
    (64, 3, 0, 65, 0),          # more input channels than one 64-channel operand holds
    (64, 1, 1, 129, 0),         # ... than two
    (64, 3, 0, 0, 65),          # more output channels than the packed gradient's N columns
    (128, 1, 0, 0, 129),
    (64, 3, 0, -1, 0),
    (64, 3, 0, 0, -36),
])
def test_unpack_desc_rejects_rows_and_columns_outside_the_packed_gradient(lib, N, k, two, I_real, N_real):
    assert _desc(lib, N, k, two, I_real, N_real) != 0
    msg = lib.lvae_last_error().decode()
    assert "wgrad_unpack_desc" in msg and "I_real" in msg and "N_real" in msg, msg


@pytest.mark.parametrize("N,k,two,I_real,N_real", [
    (64, 3, 0, 0, 0), (64, 3, 0, 32, 36), (64, 3, 0, 64, 64), (128, 1, 0, 64, 128), (64, 1, 1, 128, 64), (64, 1, 1, 100, 1)])
def test_unpack_desc_accepts_every_window_inside_the_packed_gradient(lib, N, k, two, I_real, N_real):
    assert _desc(lib, N, k, two, I_real, N_real) == 0, lib.lvae_last_error().decode()


@pytest.mark.parametrize("N,k,two,I_real,N_real", [(64, 3, 0, 65, 0), (64, 1, 1, 129, 0), (64, 3, 0, 0, 100),
                                                   (128, 1, 0, 0, 129), (64, 3, 0, -1, 0), (128, 1, 0, 0, -1)])
def test_one_call_wgrad_rejects_rows_and_columns_outside_the_packed_gradient(lib, N, k, two, I_real, N_real):
    rc = lib.lvae_conv2d_wgrad_tc(DUMMY, DUMMY if two else None, DUMMY, DUMMY, DUMMY, DUMMY, 2, 8, 8, N, k, I_real, N_real,
                                  0, 0, None)
    assert rc != 0
    msg = lib.lvae_last_error().decode()
    assert msg.startswith("conv2d_wgrad_tc: I_real"), msg


def test_one_call_wgrad_rejects_the_shape_that_does_not_fit_tmem(lib):
    """3x3 with N = 128 needs five accumulator pairs of 128 columns (> 512): the kernel refuses it; ops splits it instead."""
    assert lib.lvae_wgrad_tc_packed_size(128, 3, 0) == 0
    assert lib.lvae_conv2d_wgrad_tc(DUMMY, None, DUMMY, DUMMY, DUMMY, DUMMY, 2, 8, 8, 128, 3, 0, 0, 0, 0, None) != 0
    assert "unsupported shape" in lib.lvae_last_error().decode()


@pytest.mark.parametrize("B,H,W,N,dyC,dy_c0,what", [
    (2, 8, 8, 64, 128, -64, "dY channel window"),
    (2, 8, 8, 64, 128, 32, "dY channel window"),
    (2, 8, 8, 64, 100, 64, "dY channel window"),
    (2, 8, 8, 128, 128, 64, "dY channel window"),
    (0, 8, 8, 64, 0, 0, "B positive"),
    (2, 0, 8, 64, 0, 0, "powers of two"),
    (2, 8, 256, 64, 0, 0, "powers of two"),
])
def test_accumulate_wgrad_rejects_bad_geometry_before_any_device_call(lib, B, H, W, N, dyC, dy_c0, what):
    assert lib.lvae_conv2d_wgrad_tc_acc(DUMMY, None, DUMMY, DUMMY, B, H, W, N, 1, dyC, dy_c0, None) != 0
    assert what in lib.lvae_last_error().decode()


EXPECTED_PLAN = {
    # (N, k, inputs): launches (width, first dY channel) of the tensor-core weight gradient
    (64, 1, 1): ((64, 0),), (64, 1, 2): ((64, 0),), (64, 3, 1): ((64, 0),), (64, 3, 2): (),
    (100, 1, 1): (), (100, 1, 2): (), (100, 3, 1): (), (100, 3, 2): (),
    (128, 1, 1): ((128, 0),), (128, 1, 2): ((128, 0),), (128, 3, 1): ((64, 0), (64, 64)), (128, 3, 2): (),
}


@pytest.mark.parametrize("N,k,inputs", sorted(EXPECTED_PLAN))
def test_route_plan_sends_only_shapes_the_kernel_takes(lib, N, k, inputs):
    from lvae_b200 import ops
    plan = ops.wgrad_tc_plan(N, k, inputs == 2)
    assert plan == EXPECTED_PLAN[(N, k, inputs)]
    for n, c0 in plan:
        assert lib.lvae_wgrad_tc_packed_size(n, k, int(inputs == 2)) > 0
    # the windows tile the N output channels exactly, in order
    assert [c0 for _, c0 in plan] == [sum(n for n, _ in plan[:i]) for i in range(len(plan))]
    assert sum(n for n, _ in plan) in (0, N)


def _record_backward(monkeypatch, N, k, inputs, padded=False):
    """ops.conv_backward_raw of a bf16 Conv2d with the library calls recorded (no device): [(name, args)]."""
    from lvae_b200 import ops
    from lvae_b200.lib.nn import Conv2d
    calls = []
    monkeypatch.setattr(ops, "call", lambda name, *a: calls.append((name, a)))
    monkeypatch.setattr(ops, "_stream", lambda: None)
    ws = torch.empty(512 * 128)
    monkeypatch.setattr(ops, "_wgrad_workspace", lambda dev: ws)
    cin = 32 if padded else 64 * inputs
    mod = Conv2d(cin, N, k, padding=k // 2)
    B, H, W = 2, 8, 8
    bf = lambda c: torch.zeros(B, H, W, c, dtype=torch.bfloat16)
    x2n = bf(64) if inputs == 2 else None
    gwbuf = torch.zeros(mod.weight.shape)
    gbbuf = torch.zeros(N)
    mod.weight._lvae_grad_sink, mod.bias._lvae_grad_sink = gwbuf, gbbuf
    try:
        ops.conv_backward_raw(mod.spec, bf(64), x2n, mod.weight, mod.bias, None, bf(N), need_x=False)
    finally:
        del mod.weight._lvae_grad_sink, mod.bias._lvae_grad_sink
    return calls, gwbuf, gbbuf


@pytest.mark.parametrize("N,k,inputs", sorted(EXPECTED_PLAN))
def test_conv_backward_issues_the_planned_launches(lib, monkeypatch, N, k, inputs):
    calls, gwbuf, gbbuf = _record_backward(monkeypatch, N, k, inputs)
    tc = [a for name, a in calls if name == "lvae_conv2d_wgrad_tc"]
    plan = EXPECTED_PLAN[(N, k, inputs)]
    assert len(tc) == len(plan)
    if not plan:
        assert [name for name, _ in calls] == ["lvae_conv2d_wgrad"]          # CUDA-core weight gradient
        return
    row = gwbuf[0].numel() * 4
    for a, (n, c0) in zip(tc, plan):
        x, x2, dy, dw, db, ws, B, H, W, Nl, kl, I_real, N_real, dyC, dy_c0, _ = a
        assert lib.lvae_wgrad_tc_packed_size(Nl, kl, int(x2 is not None)) > 0
        assert (Nl, kl, dy_c0) == (n, k, c0) and dyC == N and I_real == 0 and N_real in (0, n)
        assert dw == gwbuf.data_ptr() + c0 * row and db == gbbuf.data_ptr() + c0 * 4
        assert (x2 is not None) == (inputs == 2)


def test_conv_backward_passes_the_real_input_channels_of_a_padded_operand(lib, monkeypatch):
    """conv_out of a stochastic block reads the 64-channel bf16 copy of a 32-channel z: the unpack must stop at I_real = 32."""
    calls, gwbuf, _ = _record_backward(monkeypatch, 64, 3, 1, padded=True)
    (a,) = [a for name, a in calls if name == "lvae_conv2d_wgrad_tc"]
    assert a[11] == 32 and a[3] == gwbuf.data_ptr()


@pytest.mark.parametrize("N,k,inputs", sorted(EXPECTED_PLAN))
def test_packed_grad_arena_agrees_with_the_route_plan(lib, N, k, inputs):
    """The engine gives a packed gradient (lvae_conv2d_wgrad_tc_acc + batched unpack) exactly to the convs whose weight
    gradient is ONE launch of the full width; a split conv takes the one-call route and must own none."""
    from lvae_b200.engine import PackedGradArena
    from lvae_b200.lib.nn import Conv2d
    mod = Conv2d(64 * inputs, N, k, padding=k // 2)
    for p in mod.parameters():
        p._lvae_grad_sink = torch.zeros_like(p)
    arena = PackedGradArena(torch.nn.Sequential(mod))
    single = EXPECTED_PLAN[(N, k, inputs)] == ((N, 0),)
    assert hasattr(mod.weight, "_lvae_gp") == single and arena.n == int(single)
    if single:
        assert mod.weight._lvae_gp.numel() == lib.lvae_wgrad_tc_packed_size(N, k, int(inputs == 2))
