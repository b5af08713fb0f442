"""The drop-in route of INTEGRATION.md section 1, exercised: the reference's experiment layer
(experiment/experiment_manager.py, evaluate.py) is imported UNCHANGED from /root/reference with the kernel-backed mirror
(`ladder-vae-pytorch_b200/{models,lib}`) ahead of it on sys.path and a boilr stand-in (tests/dropin) for the un-vendored
dependency.  `LVAEExperiment._make_model` (experiment_manager.py:38-74) then builds OUR LadderVAE from the reference's own
argparse defaults; its state_dict must have the keys and shapes of the model the reference builds from the same args.

CPU-only (constructing the modules needs no GPU; running them does).  Importing the reference's experiment layer needs
the reference tree; the model layout and forward_pass are checked everywhere against tests/golden/reference_checks.npz
(oracle/make_golden_refchecks.py)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import ref_loader
from oracle.make_golden_refchecks import DROPIN_KWARGS, FORWARD_PASS_ANNEALS, OUT as REFCHECKS, forward_pass_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_reference = pytest.mark.skipif(not ref_loader.reference_available(), reason="reference tree not present")

SCRIPT = r'''
import json, sys, types, argparse
import torch
import lvae_b200.dropin
lvae_b200.dropin.install()                            # what `python -m lvae_b200.dropin main.py ...` does first
import experiment.experiment_manager as em            # the reference's file, unchanged
import models.lvae, lib.nn, lib.datasets              # mirror, mirror, reference (data loading is not replaced)
out = {"em_file": em.__file__, "lvae_file": models.lvae.__file__, "nn_file": lib.nn.__file__, "datasets_file": lib.datasets.__file__}
import boilr
out["boilr_file"] = boilr.__file__

class Exp(em.LVAEExperiment):
    def _make_datamanager(self):                       # no dataset download: a synthetic stand-in with the same attributes
        ds = [(torch.rand(1, 28, 28).round(), 0) for _ in range(8)]
        return types.SimpleNamespace(color_ch=1, img_size=(28, 28), data_shape=(1, 28, 28),
                                     train=types.SimpleNamespace(dataset=ds), test=[(torch.stack([d[0] for d in ds]), None)])

exp = Exp.__new__(Exp)
parser = argparse.ArgumentParser(allow_abbrev=False)
exp._add_args(parser)                                  # boilr stand-in base flags + the reference's own flags
args = exp._check_args(parser.parse_args(ARGV))
exp.args = args
exp.setup("cpu")
m = exp.model
out["model_class"] = type(m).__module__ + "." + type(m).__name__
out["model_file"] = sys.modules[type(m).__module__].__file__
out["state"] = {k: list(v.shape) for k, v in m.state_dict().items()}
out["optimizer"] = type(exp.optimizer).__name__
out["n_opt_params"] = sum(len(g["params"]) for g in exp.optimizer.param_groups)
out["run_description"] = exp._make_run_description(args)
out["beta_mid"] = em.linear_anneal(500, 0.0, 1.0, 1000)
import evaluate                                        # evaluate.py imports too (boilr.eval / torchvision.utils)
out["evaluate_file"] = evaluate.__file__
# the launcher itself on a two-line script placed in the reference's position on sys.path
import subprocess, tempfile, os
with tempfile.TemporaryDirectory() as d:
    open(os.path.join(d, "probe.py"), "w").write("from models.lvae import LadderVAE\nimport sys\nprint('launcher ok' if 'ladder-vae-pytorch_b200' in sys.modules[LadderVAE.__module__].__file__ else 'WRONG', sys.argv[1:])\n")
    r = subprocess.run([sys.executable, "-m", "lvae_b200.dropin", os.path.join(d, "probe.py"), "--flag"], capture_output=True, text=True)
    out["via_launcher"] = r.stdout.strip().split(" [")[0] if r.returncode == 0 else r.stderr[-500:]
print("RESULT" + json.dumps(out))
'''

ARGV = ["--dataset", "static_mnist", "--zdims", "32", "32", "32", "--downsample", "1", "1", "1", "--nonlin", "elu", "--skip",
        "--blocks-per-layer", "4", "--gated", "--freebits", "0.5", "--learn-top-prior", "--batch-size", "4"]


def run_dropin():
    env = dict(os.environ)
    # cwd = the reference checkout (first on sys.path, as for `python main.py`); the repo root makes `lvae_b200` importable
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "tests", "dropin")])
    r = subprocess.run([sys.executable, "-c", SCRIPT.replace("ARGV", repr(ARGV))], capture_output=True, text=True, env=env,
                       cwd=ref_loader.REFERENCE_ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT")][-1]
    return json.loads(line[len("RESULT"):])


@needs_reference
def test_reference_experiment_layer_builds_the_kernel_backed_model():
    out = run_dropin()
    ref = ref_loader.REFERENCE_ROOT
    ours = os.path.join(ROOT, "ladder-vae-pytorch_b200")
    assert out["em_file"].startswith(ref) and out["evaluate_file"].startswith(ref)        # reference code, unchanged
    assert out["datasets_file"].startswith(ref)                                           # not replaced by the mirror
    assert out["lvae_file"].startswith(ours) and out["nn_file"].startswith(ours) and out["model_file"].startswith(ours)
    assert out["via_launcher"] == "launcher ok"
    assert out["boilr_file"].startswith(os.path.join(ROOT, "tests", "dropin"))
    assert out["model_class"].endswith("LadderVAE") and out["optimizer"] == "Adamax"
    assert out["beta_mid"] == 0.5
    assert "static_mnist,3ly,4bpl,64ch,skip,gate,block=bacdbacd,elu,freeb=0.5,drop=0.2,learnp" in out["run_description"]
    # same model from the same arguments, built by the reference's own classes
    mods = ref_loader.load_reference()
    refm = mods["lvae"].LadderVAE(1, z_dims=[32, 32, 32], blocks_per_layer=4, downsample=[1, 1, 1], merge_type="residual",
                                  batchnorm=True, nonlin="elu", stochastic_skip=True, n_filters=64, dropout=0.2,
                                  res_block_type="bacdbacd", free_bits=0.5, learn_top_prior=True, img_shape=(28, 28),
                                  likelihood_form="bernoulli", gated=True, no_initial_downscaling=False, analytical_kl=False)
    want = {k: list(v.shape) for k, v in refm.state_dict().items()}
    assert out["state"] == want
    assert out["n_opt_params"] == len(list(refm.parameters()))


def test_kernel_backed_model_has_the_reference_state_dict_layout():
    """The LadderVAE the drop-in route builds from ARGV has the state-dict keys, order and shapes, and the parameter
    count, stored for the reference model built from the same arguments (tests/golden/reference_checks.npz; see
    oracle/make_golden_refchecks.py for where the stored values come from)."""
    import lvae_b200
    g = np.load(REFCHECKS)
    m = lvae_b200.LadderVAE(**DROPIN_KWARGS)
    assert [[k, list(v.shape)] for k, v in m.state_dict().items()] == json.loads(str(g["dropin_state_layout"]))
    assert len(list(m.parameters())) == int(g["dropin_n_params"])


def test_restated_forward_pass_matches_the_reference():
    """tests/dropin_experiment.py restates LVAEExperiment.forward_pass (experiment_manager.py:322-367) for machines without
    the reference tree: against the outputs stored in tests/golden/reference_checks.npz, and, where the reference is
    present, against the live forward_pass fed the same model output."""
    from dropin_experiment import forward_pass as restated
    g = np.load(REFCHECKS)
    for anneal in FORWARD_PASS_ANNEALS:
        b = restated(forward_pass_model(), torch.zeros(5, 1, 2, 2), torch.device("cpu"), anneal)
        assert sorted(b) == list(g["fp%d_keys" % anneal])
        for k, v in b.items():
            assert (v is None) == ("fp%d_%s" % (anneal, k) not in g.files), k
            if v is not None:
                np.testing.assert_array_equal(v.detach().numpy(), g["fp%d_%s" % (anneal, k)], err_msg=k)
    if ref_loader.reference_available():
        _restated_forward_pass_matches_the_live_reference()


def _restated_forward_pass_matches_the_live_reference():
    import importlib
    import types
    saved = {k: sys.modules.get(k) for k in ("boilr", "boilr.data", "boilr.nn", "boilr.nn.init", "boilr.utils", "boilr.models",
                                             "experiment", "experiment.experiment_manager", "experiment.data", "models",
                                             "models.lvae", "lib", "lib.datasets", "multiobject", "multiobject.pytorch")}
    paths = [os.path.join(ROOT, "tests", "dropin"), os.path.join(ROOT, "ladder-vae-pytorch_b200"), ref_loader.REFERENCE_ROOT]
    for k in saved:
        sys.modules.pop(k, None)
    for p in reversed(paths):
        sys.path.insert(0, p)
    try:
        em = importlib.import_module("experiment.experiment_manager")
        from dropin_experiment import forward_pass as restated
        g = torch.Generator().manual_seed(0)
        B, L = 5, 3
        out = {"ll": -torch.rand(B, generator=g) * 100, "kl_sep": torch.rand(B, generator=g) * 10, "kl": torch.rand((), generator=g),
               "kl_loss": torch.rand((), generator=g) * 10, "out_mean": None, "out_mode": None, "out_sample": None,
               "likelihood_params": None, "kl_avg_layerwise": torch.rand(L, generator=g)}
        params = [torch.nn.Parameter(torch.randn(3, 4, generator=g)), torch.nn.Parameter(torch.randn(7, generator=g))]
        model = types.SimpleNamespace(global_step=250, parameters=lambda: iter(params), __call__=None)
        for anneal in (0, 1000):
            exp = em.LVAEExperiment.__new__(em.LVAEExperiment)
            exp.args = types.SimpleNamespace(beta_anneal=anneal)
            exp.device = torch.device("cpu")
            exp.model = lambda x, _o=out: _o
            exp.model.global_step = 250
            exp.model.parameters = lambda: iter(params)
            a = exp.forward_pass(torch.zeros(B, 1, 2, 2))
            b = restated(exp.model, torch.zeros(B, 1, 2, 2), exp.device, anneal)
            assert set(a) == set(b)
            for k in a:
                if a[k] is not None:
                    assert torch.equal(a[k], b[k]), k
    finally:
        for p in paths:
            sys.path.remove(p)
        for k, v in saved.items():
            sys.modules.pop(k, None)
            if v is not None:
                sys.modules[k] = v
