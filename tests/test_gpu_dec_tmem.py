"""P resident in tensor memory (dec_scan.cu, LVSR_DEC_TMEM_P): at the benchmarked shapes the persistent decoder keeps each
CTA's slice of P in TMEM and must produce bit for bit what the L2 path produces; windowed priors never take it."""
import ctypes as C

import numpy as np
import pytest

import bench
from helpers import O, PYRAMID, make_recognizer, package

pytestmark = pytest.mark.gpu
KEYS = ("costs", "weights", "energies", "states", "weighted_averages")


def _torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _plan():
    lib = package()._lib.load()
    cs, isl, tm = C.c_int(-1), C.c_int(-1), C.c_int(-1)
    package()._lib.check(lib.lvsr_dec_scan_plan(C.byref(cs), C.byref(isl), C.byref(tm)))
    return cs.value, isl.value, tm.value


def _run(rec, monkeypatch, switch, *args):
    monkeypatch.setenv("LVSR_DEC_TMEM_P", switch)
    r = rec.cost_matrix(*args, return_all=True)
    out = {k: r[k].detach().cpu().numpy().copy() for k in KEYS}
    assert rec.launch_status() == (0, 0)
    return out, _plan()


def _assert_bitwise(a, b):
    for k in KEYS:
        assert a[k].shape == b[k].shape, k
        assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), k


@pytest.mark.parametrize("name,B,T,L", [("metric", 64, 1000, 125), ("config2", 32, 800, 100)])
def test_benchmarked_shapes_bitwise_equal_with_p_in_tmem(name, B, T, L, monkeypatch):
    _torch()
    monkeypatch.setenv("LVSR_DEC_CHECK", "1")
    cfg = O.make_config(**bench.NET)
    rec = make_recognizer(cfg)
    rec.set_parameter_values(bench.init_values(rec.parameter_shapes()))
    x, m, labels, lm = bench.synthetic_batch(B, T, 40, L, 32, seed=1234)
    att, attm = rec.encode(x, m)
    off, plan_off = _run(rec, monkeypatch, "0", labels, lm, att, attm)
    on, plan_on = _run(rec, monkeypatch, "1", labels, lm, att, attm)
    print(name, "plan (cs, islands, p_in_tmem): off", plan_off, "on", plan_on)
    assert plan_off[0] > 0 and plan_off[2] == 0
    assert plan_on[0] == plan_off[0] and plan_on[1] == plan_off[1] and plan_on[2] == 1
    _assert_bitwise(on, off)


@pytest.mark.parametrize("prior", [dict(type="window_around_median", before=7, after=9),
                                   dict(type="expanding", initial_begin=0, initial_end=8, min_speed=0.6, max_speed=1.9)],
                         ids=lambda p: p["type"])
def test_windowed_prior_keeps_the_l2_path(prior, monkeypatch):
    _torch()
    monkeypatch.setenv("LVSR_DEC_CHECK", "1")
    cfg = O.make_config(prior=prior, **PYRAMID)
    params = O.init_params(cfg, seed=8, scale=10.0)
    x, m, labels, lm = O.synthetic_batch(cfg, B=64, T=96, seed=95)     # 4 islands of 16 rows
    att, attm = O.encoder(cfg, params, x, m)
    rec = make_recognizer(cfg, params)
    args = (labels, lm, att.astype(np.float32), attm.astype(np.float32))
    on, plan_on = _run(rec, monkeypatch, "1", *args)
    off, plan_off = _run(rec, monkeypatch, "0", *args)
    assert plan_on[0] > 0 and plan_on[1] == 1 and plan_on[2] == 0      # island mode, P streamed from L2
    assert plan_off == plan_on
    _assert_bitwise(on, off)
