"""TEST INFRASTRUCTURE ONLY -- stored outputs of the original project for the CPU checks that compare with it bit for bit.

    LVAE_REFERENCE_ROOT=<checkout of addtt/ladder-vae-pytorch> python -m oracle.make_golden_refchecks
    python -m oracle.make_golden_refchecks --restatement

Writes tests/golden/reference_checks.npz, which tests/test_heads_cpu.py and tests/test_dropin_cpu.py compare with on
every machine (and, where the original is mounted, with the original itself as well):
  * logistic_rsample (lib/stochastic.py:115-138) after torch.manual_seed(123) on a tensor, a (mean, log-scale) tuple
    and a float64 tensor,
  * the probability-form log_bernoulli (lib/likelihoods.py:385-388) in float32 and float64 with reduce none / mean /
    sum, including saturated probabilities where BCE clamps the logs at -100,
  * LVAEExperiment.forward_pass (experiment/experiment_manager.py:322-367) on a fixed model output, beta_anneal 0
    and 1000,
  * the state-dict layout and parameter count of the LadderVAE the drop-in test builds from its command line.

Without --restatement the functions are the original's and the layout is that of the original's LadderVAE.  With
--restatement they are this repository's restatements (lvae_b200.lib, tests/dropin_experiment.py, the oracle's
param_shapes), which the live checks in those tests pin bit for bit to the original wherever it is mounted; the
file records which of the two produced it (`source`).
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

from . import ref_loader
from .make_golden_heads import make_inputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "reference_checks.npz")

# LadderVAE arguments the reference's experiment layer derives from tests/test_dropin_cpu.py's ARGV
DROPIN_KWARGS = dict(color_ch=1, z_dims=[32, 32, 32], blocks_per_layer=4, downsample=[1, 1, 1], merge_type="residual",
                     batchnorm=True, nonlin="elu", stochastic_skip=True, n_filters=64, dropout=0.2,
                     res_block_type="bacdbacd", free_bits=0.5, learn_top_prior=True, img_shape=(28, 28),
                     likelihood_form="bernoulli", gated=True, no_initial_downscaling=False, analytical_kl=False)
FORWARD_PASS_ANNEALS = (0, 1000)


def logistic_inputs():
    """(name, argument) pairs for logistic_rsample."""
    _, raw = make_inputs()
    return [("f32_tensor", raw.float()), ("f32_tuple", tuple(raw.float().chunk(2, dim=1))), ("f64_tensor", raw)]


def bernoulli_inputs():
    """(dtype name, p, x, soft): binary and soft targets, probabilities with 0, 1 and near-saturated entries."""
    g = torch.Generator().manual_seed(0)
    res = []
    for name, dt in (("f32", torch.float32), ("f64", torch.float64)):
        p = torch.rand(4, 1, 28, 28, generator=g).to(dt)
        p[0, 0, 0, :4] = torch.tensor([0.0, 1.0, 1e-30, 1 - 1e-7]).to(dt)
        x = (torch.rand(4, 1, 28, 28, generator=g) < 0.15).to(dt)
        soft = torch.rand(4, 1, 28, 28, generator=g).to(dt)
        res.append((name, p, x, soft))
    return res


def forward_pass_model():
    """A stand-in model: a fixed output dict, global_step 250 and two parameters (what forward_pass reads)."""
    g = torch.Generator().manual_seed(0)
    B, L = 5, 3
    out = {"ll": -torch.rand(B, generator=g) * 100, "kl_sep": torch.rand(B, generator=g) * 10, "kl": torch.rand((), generator=g),
           "kl_loss": torch.rand((), generator=g) * 10, "out_mean": None, "out_mode": None, "out_sample": None,
           "likelihood_params": None, "kl_avg_layerwise": torch.rand(L, generator=g)}
    params = [torch.nn.Parameter(torch.randn(3, 4, generator=g)), torch.nn.Parameter(torch.randn(7, generator=g))]
    model = lambda x, _o=out: _o      # noqa: E731
    model.global_step = 250
    model.parameters = lambda: iter(params)
    return model


def main():
    restatement = "--restatement" in sys.argv
    if restatement:
        import lvae_b200.lib.likelihoods as likelihoods
        import lvae_b200.lib.stochastic as stochastic
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from dropin_experiment import forward_pass

        def run_forward_pass(model, x, anneal):
            return forward_pass(model, x, torch.device("cpu"), anneal)

        from . import lvae_oracle as O
        cfg = O.LVAEConfig(**DROPIN_KWARGS)
        layout = [[k, list(s)] for k, s in O.param_shapes(cfg).items()]
        n_params = len(O.trainable_names(cfg))
    else:
        import importlib
        import types
        mods = ref_loader.load_reference()
        likelihoods, stochastic = mods["likelihoods"], mods["stochastic"]
        # as tests/test_dropin_cpu.py imports it: boilr stand-in, then the mirror, then the original
        for p in (ref_loader.REFERENCE_ROOT, os.path.join(ROOT, "ladder-vae-pytorch_b200"), os.path.join(ROOT, "tests", "dropin")):
            sys.path.insert(0, p)
        em = importlib.import_module("experiment.experiment_manager")

        def run_forward_pass(model, x, anneal):
            exp = em.LVAEExperiment.__new__(em.LVAEExperiment)
            exp.args = types.SimpleNamespace(beta_anneal=anneal)
            exp.device = torch.device("cpu")
            exp.model = model
            return exp.forward_pass(x)

        kw = dict(DROPIN_KWARGS)
        refm = mods["lvae"].LadderVAE(kw.pop("color_ch"), **kw)
        layout = [[k, list(v.shape)] for k, v in refm.state_dict().items()]
        n_params = len(list(refm.parameters()))
    out = {"source": np.array("restatement" if restatement else "reference")}
    for name, arg in logistic_inputs():
        torch.manual_seed(123)
        out["logistic_" + name] = stochastic.logistic_rsample(arg).numpy()
    for name, p, x, soft in bernoulli_inputs():
        out["bern_%s_none" % name] = likelihoods.log_bernoulli(x, p, reduce="none").numpy()
        out["bern_%s_mean" % name] = likelihoods.log_bernoulli(soft, p, reduce="mean").numpy()
        out["bern_%s_sum" % name] = likelihoods.log_bernoulli(soft, p, reduce="sum").numpy()
    for anneal in FORWARD_PASS_ANNEALS:
        res = run_forward_pass(forward_pass_model(), torch.zeros(5, 1, 2, 2), anneal)
        out["fp%d_keys" % anneal] = np.array(sorted(res))
        for k, v in res.items():
            if v is not None:
                out["fp%d_%s" % (anneal, k)] = v.detach().numpy()
    out["dropin_state_layout"] = np.array(json.dumps(layout))
    out["dropin_n_params"] = np.int64(n_params)
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, "from the", out["source"], {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
