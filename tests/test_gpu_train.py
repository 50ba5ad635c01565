"""Training step on the GPU against the gradient / optimizer oracle (oracle/lvsr_oracle_grad.py):
gradients of every parameter (1e-4 of the parameter's largest gradient entry + a small absolute floor),
the cost, and parameters after updates with the step-rule chain of lvsr/main.py:480-519."""
from collections import OrderedDict

import numpy as np
import pytest

from helpers import O, PYRAMID, WSJ, make_recognizer, package
from oracle import lvsr_oracle_grad as G

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _grad_errors(got, want):
    errs = {}
    for k, w in want.items():
        scale = max(np.abs(w).max(), 1e-30)
        errs[k] = float(np.abs(got[k].astype(np.float64) - w).max() / scale)
    return errs


def _check_grads(cfg, params, batch, tol=1e-4, atol_frac=1e-6):
    pkg = package()
    rec = make_recognizer(cfg, params)
    algo = pkg.GradientDescent(recognizer=rec, step_rule=pkg.CompositeRule([pkg.RemoveNotFinite(0.0)]))
    cost, grads = algo.cost_and_gradients(dict(zip(algo.SOURCES, batch)))
    want_cost, want = G.cost_and_grads(cfg, params, *batch)
    assert abs(cost - want_cost) <= 1e-4 * abs(want_cost), (cost, want_cost)
    gmax = max(np.abs(w).max() for w in want.values())
    errs = _grad_errors(grads, want)
    bad = {}
    for k, e in errs.items():
        # relative to the parameter's own largest gradient entry, with a floor relative to the model's largest
        floor = atol_frac * gmax / max(np.abs(want[k]).max(), 1e-30)
        if e > tol + floor:
            bad[k] = (e, float(np.abs(want[k]).max()))
    worst = max(errs.values())
    print("cost", cost, "worst rel grad err %.2e" % worst, "of", len(errs), "parameters")
    assert not bad, bad
    return algo, rec


PRIORS = [None, dict(type="window_around_median", before=5, after=7),
          dict(type="expanding", initial_begin=0, initial_end=6, min_speed=0.7, max_speed=2.2)]


@pytest.mark.parametrize("prior", PRIORS, ids=lambda p: "default" if p is None else p["type"])
def test_gradients_match_oracle_pyramid(prior):
    _torch()
    cfg = O.make_config(prior=prior, **PYRAMID)
    params = O.init_params(cfg, seed=5, scale=10.0)
    batch = O.synthetic_batch(cfg, B=6, T=56, seed=21)
    _check_grads(cfg, params, batch)


def test_gradients_match_oracle_wsj_architecture():
    """4-layer pyramidal BiGRU(256) (8-CTA clusters in the BPTT kernel), M=512, n=100, 2 label-masked rows."""
    _torch()
    cfg = O.make_config(**WSJ)
    params = O.init_params(cfg, seed=1, scale=10.0)
    batch = O.synthetic_batch(cfg, B=5, T=48, seed=3)
    _check_grads(cfg, params, batch)


def test_gradients_island_batch_no_masks():
    _torch()
    cfg = O.make_config(**PYRAMID)
    params = O.init_params(cfg, seed=7, scale=10.0)
    x, m, labels, lm = O.synthetic_batch(cfg, B=18, T=40, seed=12)
    _check_grads(cfg, params, (x, None, labels, None))


@pytest.mark.parametrize("rules,max_norm", [(("momentum", "adadelta"), 1.0), (("momentum",), 0.0), (("adadelta",), 0.5)])
def test_training_steps_match_oracle(rules, max_norm):
    """Two process_batch calls == two oracle train_steps (float64) on the same batches."""
    _torch()
    pkg = package()
    cfg = O.make_config(**PYRAMID)
    params = O.init_params(cfg, seed=5, scale=10.0)
    tc = G.make_train_config(gradient_threshold=2.0, rules=rules, scale=0.05, momentum=0.5, decay_rate=0.95,
                             epsilon=1e-6, max_norm=max_norm)
    rec = make_recognizer(cfg, params)
    algo = pkg.GradientDescent(recognizer=rec, step_rule=pkg.step_rule_from_config(tc, dict(max_norm=max_norm)))
    algo.initialize()
    ref = OrderedDict((k, v.copy()) for k, v in params.items())
    state = {}
    for step in range(2):
        batch = O.synthetic_batch(cfg, B=4, T=40, seed=100 + step)
        ref, ref_cost, ref_grads = G.train_step(cfg, ref, state, batch, tc)
        algo.process_batch(dict(zip(algo.SOURCES, batch)))
        assert abs(float(algo.last_cost.item()) - ref_cost) <= 1e-4 * abs(ref_cost)
        assert abs(algo.total_gradient_norm() - G.l2_norm(ref_grads.values())) <= 1e-4 * G.l2_norm(ref_grads.values())
        got = rec.get_parameter_values()
        for k, v in ref.items():
            # compare the UPDATE (new - old would cancel; the parameters themselves are O(0.1..1))
            assert np.abs(got[k] - v).max() <= 2e-5 * max(1.0, np.abs(v).max()) + 1e-6, (step, k, np.abs(got[k] - v).max())
    if max_norm > 0:
        for k, v in rec.get_parameter_values().items():
            if G.is_weight(k):
                assert (np.sqrt((v.astype(np.float64) ** 2).sum(axis=0)) <= max_norm * (1 + 1e-5)).all(), k
    # the forward pass uses the updated (re-packed) weights
    x, m, labels, lm = O.synthetic_batch(cfg, B=3, T=32, seed=5)
    want = O.recognizer_cost(cfg, ref, x, m, labels, lm)
    got = rec.cost(x, m, labels, lm)
    assert np.abs(got - want).max() <= 1e-3 * np.abs(want).max()


def test_non_finite_gradient_zeroes_the_parameter_and_burn_in_delays_updates():
    torch = _torch()
    pkg = package()
    cfg = O.make_config(**PYRAMID)
    params = O.init_params(cfg, seed=5, scale=10.0)
    batch = O.synthetic_batch(cfg, B=3, T=32, seed=1)
    rec = make_recognizer(cfg, params)
    algo = pkg.GradientDescent(recognizer=rec, step_rule=pkg.CompositeRule(
        [pkg.StepClipping(10.0), pkg.Momentum(0.1, 0.0), pkg.RemoveNotFinite(0.0), pkg.BurnIn(num_steps=2)]))
    algo.initialize()
    before = rec.get_parameter_values()
    for i in range(3):
        algo.process_batch(dict(zip(algo.SOURCES, batch)))
        after = rec.get_parameter_values()
        changed = any(np.abs(after[k] - before[k]).max() > 0 for k in before)
        assert changed == (i == 2), i              # lvsr/algorithms.py:35-43: the first num_steps updates are zeroed
    # poison one gradient: RemoveNotFinite(0.0) zeroes that parameter, the others still move (B/algorithms/__init__.py:855-861)
    x = batch[0].copy()
    algo2 = pkg.GradientDescent(recognizer=rec, step_rule=pkg.CompositeRule([pkg.Momentum(0.1, 0.0), pkg.RemoveNotFinite(0.0)]))
    algo2.initialize()
    algo2._forward_backward(dict(zip(algo2.SOURCES, (x,) + tuple(batch[1:]))), None)
    name = "/recognizer/generator/readout/post_merge/bias.b"
    import ctypes as C
    lib, h = pkg._lib.load(), rec._require_ready()
    idx = list(rec.parameter_shapes()).index(name)
    off, cnt = C.c_int64(), C.c_int64()
    pkg._lib.check(lib.lvsr_model_param_offset(h, idx, C.byref(off), C.byref(cnt)))
    algo2._buf[off.value] = float("nan")
    pkg._lib.check(lib.lvsr_train_apply_updates(h, algo2._buf.data_ptr(), 1.0, C.byref(algo2._tc), rec._stream()))
    torch.cuda.synchronize()
    now = rec.get_parameter_values()
    assert np.all(now[name] == 0)
    other = "/recognizer/generator/readout/post_merge/mlp/linear_0.W"
    assert np.abs(now[other] - after[other]).max() > 0 and np.isfinite(now[other]).all()


def test_two_gpu_step_equals_single_gpu_step_on_the_concatenated_batch():
    """SURVEY.md 8e: batch sharded over ranks + ONE NCCL all-reduce of the flat gradient buffer."""
    torch = _torch()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    port = 29600 + os.getpid() % 300
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(root, "tests", "dist_train_worker.py")], capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:], r.stderr[-2000:])
    assert r.returncode == 0 and "DIST_TRAIN_OK" in r.stdout


def test_gradients_with_tensor_core_backward_gemms(monkeypatch):
    """T*B >= 2048 rows switches the encoder's weight-gradient (X^T dY, split-K) and input-gradient (dY W^T) GEMMs to
    the tcgen05 3xTF32 kernel; same bar as the FFMA path, and the two paths agree with each other."""
    _torch()
    cfg = O.make_config(**PYRAMID)
    params = O.init_params(cfg, seed=5, scale=10.0)
    batch = O.synthetic_batch(cfg, B=32, T=64, seed=77)
    algo, rec = _check_grads(cfg, params, batch)
    _, g_tc = algo.cost_and_gradients(dict(zip(algo.SOURCES, batch)))
    monkeypatch.setenv("LVSR_NO_TC_GEMM", "1")
    pkg = package()
    rec2 = make_recognizer(cfg, params)
    algo2 = pkg.GradientDescent(recognizer=rec2, step_rule=pkg.CompositeRule([pkg.RemoveNotFinite(0.0)]))
    _, g_ff = algo2.cost_and_gradients(dict(zip(algo2.SOURCES, batch)))
    for k in g_tc:
        scale = max(np.abs(g_ff[k]).max(), 1e-30)
        assert np.abs(g_tc[k] - g_ff[k]).max() / scale < 2e-4, k


def test_one_of_n_feedback_cost_and_gradients():
    """embed_outputs=False (the WSJ configs): no lookup table, fork weights indexed by the label."""
    _torch()
    cfg = O.make_config(embed_outputs=False, **PYRAMID)
    params = O.init_params(cfg, seed=5, scale=10.0)
    assert "/recognizer/generator/fork/fork_inputs.W" in params and params["/recognizer/generator/fork/fork_inputs.W"].shape == (33, 128)
    batch = O.synthetic_batch(cfg, B=5, T=48, seed=9)
    algo, rec = _check_grads(cfg, params, batch)
    want = O.recognizer_cost(cfg, params, *batch)
    got = rec.cost(*batch)
    assert np.abs(got - want).max() <= 1e-4 * np.abs(want).max()


def test_wsj_training_batch_matches_golden_gradients():
    """WSJ architecture, B = 16 (island-mode persistent decoder), T*B = 5120 rows (tcgen05 backward GEMMs), against the
    committed float64 gradient oracle (tests/golden/make_train_golden.py): per parameter sum, sum |.|, max |.| and a random
    projection of the gradient."""
    _torch()
    import os
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "train_golden.npz"))
    cfg = O.make_config(**WSJ)
    params = O.init_params(cfg, seed=1, scale=10.0)
    batch = O.synthetic_batch(cfg, B=16, T=320, seed=17)
    pkg = package()
    rec = make_recognizer(cfg, params)
    algo = pkg.GradientDescent(recognizer=rec, step_rule=pkg.CompositeRule([pkg.RemoveNotFinite(0.0)]))
    cost, grads = algo.cost_and_gradients(dict(zip(algo.SOURCES, batch)))
    assert abs(cost - float(gold["cost"])) <= 1e-4 * abs(float(gold["cost"]))
    names, stats = [str(n) for n in gold["names"]], gold["stats"]
    assert names == list(grads)
    rng = np.random.RandomState(7)
    gmax = stats[:, 2].max()
    worst = 0.0
    for k, want in zip(names, stats):
        g = grads[k].astype(np.float64)
        r = rng.normal(size=g.shape)
        got = np.array([g.sum(), np.abs(g).sum(), np.abs(g).max(), (g * r).sum()])
        # sums of n entries of size <= max|g| carry rounding of order sqrt(n) * eps * max|g|; 1e-4 of the natural scale of each statistic
        scale = np.array([want[1], want[1], want[2], want[2] * np.sqrt(g.size)]) + 1e-6 * gmax
        err = np.abs(got - want) / scale
        worst = max(worst, err.max())
        assert (err < 2e-4).all(), (k, err)
    print("worst relative error over %d parameters: %.2e" % (len(names), worst))


def test_single_utterance_single_label_and_determinism():
    """Edge shapes (B = 1, L = 2) and run-to-run determinism: every reduction of the backward pass has a fixed order
    (split-K partials, per-CTA partial sums, no floating-point atomics), so two calls give bit-identical gradients."""
    _torch()
    cfg = O.make_config(**PYRAMID)
    params = O.init_params(cfg, seed=5, scale=10.0)
    x, m, labels, lm = O.synthetic_batch(cfg, B=1, T=24, seed=2, label_div=24)
    assert labels.shape[0] == 2
    algo, rec = _check_grads(cfg, params, (x, m, labels, lm))
    batch = O.synthetic_batch(cfg, B=32, T=64, seed=3)            # tensor-core split-K path
    pkg = package()
    rec2 = make_recognizer(cfg, params)
    algo2 = pkg.GradientDescent(recognizer=rec2, step_rule=pkg.CompositeRule([pkg.RemoveNotFinite(0.0)]))
    c1, g1 = algo2.cost_and_gradients(dict(zip(algo2.SOURCES, batch)))
    c2, g2 = algo2.cost_and_gradients(dict(zip(algo2.SOURCES, batch)))
    assert c1 == c2
    for k in g1:
        assert np.array_equal(g1[k], g2[k]), k
