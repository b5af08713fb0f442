"""CPU: which residual-block layouts run as one block node, and the host checks of the residual + statistics epilogue."""
import ctypes
import itertools
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMMY = 0x1000          # non-null pointer that no check dereferences


@pytest.fixture(scope="module")
def lib():
    import importlib.util
    spec = importlib.util.spec_from_file_location("lvae_build", os.path.join(ROOT, "ladder-vae-pytorch_b200", "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.build()
    import lvae_b200
    return lvae_b200._capi.lib()


def _takes_node(block_type, gated, dropout, batchnorm):
    """True / False, or None when the reference constructor itself rejects the layout."""
    from lvae_b200.lib.nn import ResidualBlock
    try:
        blk = ResidualBlock(64, "elu", block_type=block_type, dropout=dropout, gated=gated, batchnorm=batchnorm)
    except TypeError:
        return None
    return blk._whole_block


CASES = list(itertools.product(["bacdbacd", "bacdbac", "cabdcabd"], [False, True], [None, 0.0, 0.2], [True, False]))


def _expected(block_type, gated, dropout, batchnorm):
    if block_type == "bacdbacd" and dropout is None:
        return None                               # nn.Dropout2d(None) raises (lib/nn.py:89)
    return block_type in ("bacdbacd", "bacdbac") and batchnorm


@pytest.mark.parametrize("block_type,gated,dropout,batchnorm", CASES)
def test_block_node_classification(lib, block_type, gated, dropout, batchnorm):
    assert _takes_node(block_type, gated, dropout, batchnorm) == _expected(block_type, gated, dropout, batchnorm)


def test_node_gets_the_dropout_modules_behind_each_conv(lib):
    """bacdbacd: a Dropout2d behind both convs; bacdbac: behind conv1 only, or none without dropout."""
    from lvae_b200.lib.nn import Dropout2d, ResidualBlock
    for bt, p, expect in [("bacdbacd", 0.2, (True, True)), ("bacdbac", 0.2, (True, False)), ("bacdbac", None, (False, False))]:
        for gated in (False, True):
            plan = ResidualBlock(64, "elu", block_type=bt, dropout=p, gated=gated)._plan
            assert (isinstance(plan[1][2], Dropout2d), isinstance(plan[3][2], Dropout2d)) == expect
            assert (plan[-1][0] == "gate") == gated


def _fuse(**kw):
    import lvae_b200
    f = lvae_b200._capi.ConvFuse()
    f.stats_acc = DUMMY
    for k, v in kw.items():
        setattr(f, k, v)
    return f


@pytest.mark.parametrize("N,k,Cin,H,out_f32,what", [
    (128, 1, 64, 16, 0, "residual + fused output statistics need N == 64"),     # N != 64
    (64, 3, 64, 16, 1, "residual + fused output statistics need N == 64"),      # fp32 output
    (128, 3, 128, 16, 0, "residual + fused output statistics need N == 64"),    # streamed weights (3x3 128 -> 128)
])
def test_residual_with_statistics_is_rejected_before_any_device_call(lib, N, k, Cin, H, out_f32, what):
    f = _fuse()
    rc = lib.lvae_conv2d_tc_ex(DUMMY, None, DUMMY, None, None, DUMMY, DUMMY, None, 0, 2, H, H, Cin, N, k, 0, out_f32,
                               ctypes.addressof(f), None)
    assert rc != 0 and what in lib.lvae_last_error().decode(), lib.lvae_last_error().decode()


def test_residual_with_split_output_is_rejected(lib):
    f = _fuse()
    rc = lib.lvae_conv2d_tc_ex(DUMMY, None, DUMMY, None, None, DUMMY, DUMMY, DUMMY, 64, 2, 16, 16, 64, 128, 1, 0, 0,
                               ctypes.addressof(f), None)
    assert rc != 0 and "residual and split output are exclusive" in lib.lvae_last_error().decode()


def test_residual_with_batchnorm_backward_sums_is_rejected(lib):
    f = _fuse(stats_acc=None, bnb_x=DUMMY, bnb_save=DUMMY, bnb_gamma=DUMMY, bnb_beta=DUMMY, bnb_acc=DUMMY)
    rc = lib.lvae_conv2d_tc_ex(DUMMY, None, DUMMY, None, None, DUMMY, DUMMY, None, 0, 2, 16, 16, 64, 64, 3, 1, 0,
                               ctypes.addressof(f), None)
    assert rc != 0 and "residual cannot be combined with the fused BatchNorm-backward sums" in lib.lvae_last_error().decode()


def test_statistics_fusion_accepts_a_residual(lib):
    from lvae_b200 import ops
    assert ops._tc_fusable(64, False)
    assert not ops._tc_fusable(64, True) and not ops._tc_fusable(128, False) and not ops._tc_fusable(64, False, nsplit=32)
