"""CPU parity of the likelihood heads that stay on tensor ops (SURVEY.md 8f rank 4): the Gaussian and the single
discretized-logistic head of lib/likelihoods.py:81-180 and their densities (:233-288, :391-411), against golden vectors
written from the unmodified reference by oracle/make_golden_heads.py (and against the live reference when it is mounted)."""
import os

import numpy as np
import pytest
import torch

from oracle.make_golden_heads import OUT, make_inputs
from oracle.make_golden_refchecks import OUT as REFCHECKS, bernoulli_inputs, logistic_inputs
from oracle import ref_loader


@pytest.fixture(scope="module")
def gold():
    return np.load(OUT)


def _ours():
    from lvae_b200.lib import likelihoods as L
    return L


def _head(L):
    head = L.DiscretizedLogisticLikelihood.__new__(L.DiscretizedLogisticLikelihood)
    torch.nn.Module.__init__(head)
    head.n_bins, head.double_precision = 256, False
    head.parameter_net = torch.nn.Identity()         # the conv is covered by the GPU tests; here: everything after it
    return head


def test_log_normal_matches_reference(gold):
    L = _ours()
    x, raw = make_inputs(int(gold["seed"]))
    for name, dt, tol in (("f32", torch.float32, 1e-6), ("f64", torch.float64, 1e-13)):
        mean, lv = raw.to(dt).chunk(2, dim=1)
        ours = L.log_normal(x.to(dt), mean, lv, reduce="none").double().numpy()
        np.testing.assert_allclose(ours, gold["log_normal_" + name], rtol=tol)


def test_discretized_logistic_head_matches_reference(gold):
    L = _ours()
    x, raw = make_inputs(int(gold["seed"]))
    head = _head(L)
    params = head.distr_params(raw.float())
    np.testing.assert_array_equal(params["mean"].double().numpy(), gold["dl_mean_f32"])
    np.testing.assert_array_equal(params["logscale"].double().numpy(), gold["dl_logscale_f32"])
    assert float(params["logscale"].min()) == -7.0                      # the clamp is exercised
    ll = head.log_likelihood(x.float(), params).double().numpy()
    np.testing.assert_allclose(ll, gold["dl_ll_f32"], rtol=2e-6)
    head.double_precision = True
    lld = head.log_likelihood(x.float(), params)
    assert lld.dtype == torch.float32                                   # double=True computes in fp64, returns fp32 (:284-287)
    np.testing.assert_allclose(lld.double().numpy(), gold["dl_ll_double_f32"], rtol=1e-6)
    red = L.log_discretized_logistic(x.float() * (255 / 256) + 1 / 512, params["mean"], params["logscale"], n_bins=256,
                                     reduce="mean")
    np.testing.assert_allclose(float(red), float(gold["dl_mean_reduce_f32"]), rtol=2e-6)
    # float64 inputs through the density itself (the head casts its conv output to fp32, the function does not)
    p64 = {"mean": torch.from_numpy(gold["dl_mean_f64"]), "logscale": torch.from_numpy(gold["dl_logscale_f64"])}
    ll64 = L.log_discretized_logistic(x * (255 / 256) + 1 / 512, p64["mean"], p64["logscale"], n_bins=256, reduce="none")
    np.testing.assert_allclose(ll64.numpy(), gold["dl_ll_f64"], rtol=1e-12)


def test_density_argument_checks():
    L = _ours()
    x = torch.zeros(2, 1, 3, 3)
    with pytest.raises(RuntimeError):
        L.log_normal(x, x, x, reduce="median")                         # likelihoods.py:426-428
    with pytest.raises(AssertionError):
        L.log_normal(x, torch.zeros(2, 1, 3, 4), x)                    # :421
    # a scalar scale parameter is broadcast (:422-423)
    a = L.log_normal(x, x, torch.zeros(()), reduce="none")
    assert tuple(a.shape) == (2,) and torch.allclose(a, torch.full((2,), -0.5 * 9 * float(np.log(2 * np.pi))))


def test_head_samplers_shape_and_range():
    L = _ours()
    torch.manual_seed(0)
    _, raw = make_inputs()
    mean, lv = raw.float().chunk(2, dim=1)
    s = L.GaussianLikelihood.sample({"mean": mean, "logvar": lv})
    assert s.shape == mean.shape and torch.isfinite(s).all()
    assert L.GaussianLikelihood.mode({"mean": mean, "logvar": lv}) is mean
    head = _head(L)
    p = head.distr_params(raw.float())
    s = head.sample(p)
    assert s.shape == mean.shape and float(s.min()) >= 0.0 and float(s.max()) <= 1.0


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference tree not mounted")
def test_golden_heads_are_current(gold):
    """The committed fixture equals what the live reference computes now (guards against a stale fixture)."""
    ref = ref_loader.load_reference()["likelihoods"]
    x, raw = make_inputs(int(gold["seed"]))
    mean, lv = raw.chunk(2, dim=1)
    np.testing.assert_allclose(ref.log_normal(x, mean, lv, reduce="none").numpy(), gold["log_normal_f64"], rtol=1e-14)


@pytest.fixture(scope="module")
def refchecks():
    return np.load(REFCHECKS)


def test_logistic_rsample_is_bit_identical_to_reference(refchecks):
    """Same torch generator state -> same logistic draw as lib/stochastic.py:115-138 (tensor and tuple inputs): against
    the stored draws, and against the live reference when it is mounted."""
    from lvae_b200.lib.stochastic import logistic_rsample
    ref = ref_loader.load_reference()["stochastic"] if ref_loader.reference_available() else None
    for name, arg in logistic_inputs():
        torch.manual_seed(123)
        a = logistic_rsample(arg)
        want = refchecks["logistic_" + name]
        assert a.numpy().dtype == want.dtype
        np.testing.assert_array_equal(a.numpy(), want)
        if ref is not None:
            torch.manual_seed(123)
            b = ref.logistic_rsample(arg)
            assert a.dtype == b.dtype and torch.equal(a, b)


def test_base_model_checkpoint_roundtrip(tmp_path):
    """The boilr stand-in keeps `checkpoint` / `load` / `global_step` working for the reference's experiment code."""
    import lvae_b200
    from lvae_b200.configs import baseline_kwargs
    kw = baseline_kwargs("mnist3")
    m1, m2 = lvae_b200.LadderVAE(**kw), lvae_b200.LadderVAE(**kw)
    with torch.no_grad():
        for p in m1.parameters():
            p.add_(0.01)
    for step in (10, 20, 30):
        m1.global_step = step
        m1.checkpoint(str(tmp_path), max_ckpt=2)
    assert sorted(os.listdir(tmp_path)) == ["model_20.pt", "model_30.pt"]
    m2.load(str(tmp_path), device="cpu")
    assert m2.global_step == 30
    for (k1, v1), (k2, v2) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)
    m2.increment_global_step()
    assert m2.global_step == 31


def test_log_bernoulli_tensor_form_is_bit_identical_to_reference(refchecks):
    """The probability-form Bernoulli log-likelihood used outside the fused forward (likelihoods.py:385-388), including
    the saturated probabilities where BCE clamps the logs at -100: against the stored outputs, and against the live
    reference when it is mounted."""
    L = _ours()
    ref = ref_loader.load_reference()["likelihoods"] if ref_loader.reference_available() else None
    for name, p, x, soft in bernoulli_inputs():
        for reduce, target in (("none", x), ("mean", soft), ("sum", soft)):
            a = L.log_bernoulli(target, p, reduce=reduce)
            want = refchecks["bern_%s_%s" % (name, reduce)]
            assert a.numpy().dtype == want.dtype
            np.testing.assert_array_equal(a.numpy(), want)
            if ref is not None:
                assert torch.equal(a, ref.log_bernoulli(target, p, reduce=reduce))
