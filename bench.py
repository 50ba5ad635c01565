#!/usr/bin/env python
"""bench.py -- frames/sec of the attention-lvcsr hot path (encoder + teacher-forced
attention decoder) at the BASELINE.json metric configuration.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one synthetic batch per GPU:
B=64 utterances x T=1000 frames x F=40 filterbanks, 4x pyramidal BiGRU(256)
(subsample [1,1,2,2] -> T'=250), content+location attention (M=512, K=10, n=100),
GRU(256) decoder, L=125 teacher-forced steps, Maxout(2) readout over V=32 symbols.
Multi-GPU: utterance batches shard across ranks (weak scaling, no data-path collective).

Prints ONE JSON line on rank 0 (see the task contract): `value` = frames/s with inputs
resident in HBM; `e2e` = same metric through the host-buffer C-ABI call
(lvsr_recognizer_cost_host: pinned host inputs, H2D + D2H inside the timed region);
`roofline` = attention-step kernel, algorithmic bytes / CUDA-event time vs the measured
HBM peak; `cpu_baseline` = float32 twin of the oracle on a bounded sample of the workload.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(B=64, T=1000, F=40, L=125, V=32)
NET = dict(num_features=40, dims_bidir=[256, 256, 256, 256], subsample=[1, 1, 2, 2], dim_dec=256,
           dim_matcher=512, conv_n=100, conv_num_filters=10, num_phonemes=32, post_merge_dims=[256],
           maxout_pieces=2)
METRIC = "encoder+decoder frames/sec at batch64x1000frx40fb"


def synthetic_batch(B, T, F, L, V, seed):
    """Synthetic utterances of the BASELINE shape: lengths U{0.6T..T} (max == T), N(0,1)
    features, right-padded 0/1 masks, labels U{0..V-2} + eos of length ~T_b/8 (max == L)."""
    rng = np.random.RandomState(seed)
    lens = rng.randint(int(math.ceil(0.6 * T)), T + 1, size=B)
    lens[rng.randint(B)] = T
    x = rng.normal(size=(T, B, F)).astype(np.float32)
    m = (np.arange(T)[:, None] < lens[None, :]).astype(np.float32)
    x *= m[:, :, None]
    lab_lens = np.minimum(L, np.ceil(lens / 8.0).astype(int))
    lab_lens[lens == T] = L
    labels = np.zeros((L, B), dtype=np.int64)
    lm = np.zeros((L, B), dtype=np.float32)
    for b in range(B):
        n = int(lab_lens[b])
        labels[:n - 1, b] = rng.randint(0, V - 1, size=n - 1)
        labels[n - 1, b] = V - 1
        lm[:n, b] = 1
    return x, m, labels, lm


def init_values(shapes, seed=1, scale=10.0):
    """Random-init weights of the architecture (WSJ scheme x10 'trained-like', SURVEY.md 8d)."""
    rng = np.random.RandomState(seed)
    out = {}
    for name, shape in shapes.items():
        leaf = name.rsplit(".", 1)[1]
        if leaf == "b":
            v = np.zeros(shape)
        elif leaf in ("state_to_state", "state_to_gates"):
            d = shape[0]
            blocks = []
            for _ in range(shape[1] // d):
                q, r = np.linalg.qr(rng.randn(d, d))
                blocks.append(q * np.sign(np.diag(r)))
            v = np.hstack(blocks)
        elif leaf == "initial_state":
            v = rng.normal(0, 0.001, size=shape) * scale
        else:
            v = rng.normal(0, 0.01, size=shape) * scale
        out[name] = v.astype(np.float32)
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if out.returncode == 0 and out.stdout.strip():
                    self.rows.append([c.strip() for c in out.stdout.strip().split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def max_over_ranks(value, world, device=None, dist=None):
    """Step time of a sharded job = the slowest rank's (barrier-bracketed) device time."""
    if world == 1:
        return float(value)
    import torch
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def shard_seed(rank, base=1234):
    """Every rank draws its own utterance shard (weak scaling: the global batch is world x B)."""
    return base + rank


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


# DRAM traffic of ONE dec_scan_kernel launch at the metric configuration (dram__bytes_read.sum +
# dram__bytes_write.sum of the `ncu --set full` capture summarised in profiles/r2a_summary.md /
# profiles/r2a_dec_scan_metrics.csv), and the L2->SM bytes of the same capture.
NCU_DEC_SCAN = {"config": (64, 1000, 125), "dram_bytes": 2.672282e9 + 1.510394e9, "l2_to_sm_bytes": 13.303018e9,
                "l2_hit_pct": 70.18, "source": "profiles/r2a_dec_scan_metrics.csv"}


def attention_step_bytes(B, Tw, M, E):
    """ALGORITHMIC bytes of one attention+decoder step (SURVEY.md 8d): read P_cut and H_cut
    once, read alpha_prev + mask, write alpha + energies."""
    return 4 * Tw * B * (M + E) + 4 * B * Tw * 4


def cpu_reference_run(steps, warmup, sample_B=64):
    """The reference's CPU path cannot run here (Python-2 Theano, SURVEY.md 8c): time its
    restatement (oracle, float32 twin, numpy+BLAS on all host cores) on the SAME workload: `sample_B` = 64 utterances
    of T=1000 frames, L=125 teacher-forced steps (bounded by the number of steps, not by a smaller batch)."""
    from oracle import lvsr_oracle as O
    W = WORKLOAD
    cfg = O.make_config(**NET)
    params = O.cast_params(O.init_params(cfg, seed=1, scale=10.0), np.float32)
    x, m, labels, lm = synthetic_batch(sample_B, W["T"], W["F"], W["L"], W["V"], seed=1234)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.recognizer_cost(cfg, params, x, m, labels, lm)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    fps = sample_B * W["T"] / float(np.mean(times))
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count()
    return fps, float(np.mean(times)) * 1e3, dict(
        value=fps, unit="frames/s", cores=cores, kind="port",
        sample="%d utterances x %d frames x %d fbank, %d decoder steps, float32 numpy+BLAS restatement of the "
               "Theano CPU path (Theano itself cannot run: SURVEY.md 8c)" % (sample_B, W["T"], W["F"], W["L"]))


def dump_outputs(arrays, path, limit=64 * 10 ** 6):
    """Write each float32 array (utterances on axis 1) as path/<name>.npy, at most `limit` bytes in all: past
    that, every array keeps the same leading utterances, as many as fit, so that runs stay comparable."""
    B = next(iter(arrays.values())).shape[1]
    per_utt = sum(a.nbytes for a in arrays.values()) / B
    keep = min(B, int((limit - 1024 * len(arrays)) // per_utt))       # 1 KiB per .npy header, generously
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a[:, :keep]))


TRAIN_WORKLOAD = dict(B=64, T=1500, F=40, L=190, V=32)       # BASELINE.json configs[3]
TRAIN_CONF = dict(gradient_threshold=10.0, rules=["momentum", "adadelta"], scale=1.0, momentum=0.0, decay_rate=0.95,
                  epsilon=1e-8)                              # exp/wsj/configs/wsj_jan_new.yaml:75-85
TRAIN_METRIC = "training-step frames/sec at batch64x1500frx40fb (configs[3]: forward + backward + grad all-reduce + update)"


def train_bench(pkg, torch, dev, rank, world, steps, warmup, dist_mod, flush, barrier):
    """One training step = GradientDescent.process_batch on a synthetic config-4 batch per GPU: forward with tape,
    BPTT, ONE NCCL all-reduce of the flat gradient buffer (N > 1), step rules + update.  Device time per step
    (CUDA events, max over ranks), the all-reduce alone, and the same step from pinned host buffers."""
    import ctypes as C
    W = TRAIN_WORKLOAD
    rec = pkg.SpeechRecognizer(
        input_dims={"recordings": W["F"]}, input_num_chars={}, eos_label=W["V"] - 1, num_phonemes=W["V"],
        dim_dec=NET["dim_dec"], dims_bidir=NET["dims_bidir"], subsample=NET["subsample"], conv_n=NET["conv_n"],
        conv_num_filters=NET["conv_num_filters"], dim_matcher=NET["dim_matcher"],
        post_merge_dims=NET["post_merge_dims"], post_merge_activation=pkg.Maxout(2),
        enc_transition=pkg.GatedRecurrent, dec_transition=pkg.GatedRecurrent, device=dev)
    rec.set_parameter_values(init_values(rec.parameter_shapes()))
    algo = pkg.GradientDescent(recognizer=rec, step_rule=pkg.step_rule_from_config(TRAIN_CONF, dict(max_norm=1.0)))
    algo.initialize()
    lib = pkg._lib.load()
    x, m, labels, lm = synthetic_batch(W["B"], W["T"], W["F"], W["L"], W["V"], seed=shard_seed(rank, base=4321))
    names = ("recordings", "recordings_mask", "labels", "labels_mask")
    dbatch = dict(zip(names, (torch.as_tensor(a, device=dev) for a in (x, m, labels, lm))))
    hbatch = dict(zip(names, (torch.as_tensor(a).pin_memory() for a in (x, m, labels, lm))))
    for _ in range(max(2, warmup)):
        algo.process_batch(dbatch)
    barrier()
    lib.lvsr_launch_count(1)
    total_ms = 0.0
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        algo.process_batch(dbatch)
        b.record()
        torch.cuda.synchronize(dev)
        total_ms += a.elapsed_time(b)
    launches = int(lib.lvsr_launch_count(1))
    ms_dev = max_over_ranks(total_ms, world, dev, dist_mod) / steps
    cost = float(algo.last_cost.item())
    # the collective alone
    ar_ms = 0.0
    if world > 1:
        buf = torch.zeros_like(algo._buf)
        for _ in range(2):
            dist_mod.all_reduce(buf)
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            dist_mod.all_reduce(buf)
        b.record()
        torch.cuda.synchronize(dev)
        ar_ms = max_over_ranks(a.elapsed_time(b), world, dev, dist_mod) / steps
    # end to end from pinned host buffers, cost read back every step
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        algo.process_batch({k: v.to(dev, non_blocking=True) for k, v in hbatch.items()})
        cost = float(algo.last_cost.item())
    ms_host = max_over_ranks((time.perf_counter() - t0) * 1e3, world, dev, dist_mod) / steps
    barrier()
    prof = {}
    lib.lvsr_profile_enable(1)
    algo.process_batch(dbatch)
    torch.cuda.synchronize(dev)
    for cls in ("gemm", "gemm_tn", "bigru", "bigru_bwd", "dec_scan", "dec_bwd_step", "att_bwd", "skinny", "window", "readout"):
        tot, cnt = C.c_double(), C.c_int64()
        lib.lvsr_profile_read(cls.encode(), C.byref(tot), C.byref(cnt))
        prof[cls] = {"ms": round(tot.value, 3), "launches": cnt.value}
    lib.lvsr_profile_enable(0)
    frames = W["B"] * W["T"] * world
    return {
        "metric": TRAIN_METRIC, "value": frames / (ms_dev * 1e-3), "unit": "frames/s", "ms_per_step": ms_dev,
        "n_gpus": world, "steps": steps, "scaling": "weak", "dtype": "f32",
        "config": {"workload": "configs[3]: batch %d x %d frames x %d fbank per GPU, WSJ architecture, %d label steps, "
                               "StepClipping(10) + Momentum(1, 0) + AdaDelta(0.95, 1e-8) + max-norm 1 (wsj_jan_new.yaml)"
                               % (W["B"], W["T"], W["F"], W["L"]),
                   "global_batch": W["B"] * world, "parallelism": "dp%d, one all-reduce(sum) of the flat gradient buffer per step" % world},
        "e2e": {"value": frames / (ms_host * 1e-3), "unit": "frames/s",
                "h2d_bytes_per_step": int(x.nbytes + m.nbytes + labels.nbytes + lm.nbytes), "d2h_bytes_per_step": 4},
        "collective": {"kind": "NCCL all-reduce(sum), fp32" if world > 1 else "none (1 GPU)",
                       "bytes": int(algo._buf.numel() * 4), "ms_alone": ar_ms,
                       "share_of_step": (ar_ms / ms_dev) if ms_dev > 0 else None},
        "gpu_launches_per_step": launches // max(1, steps),
        "kernel_ms_per_step": prof, "cost": cost,
    }


SEARCH_CASES = {
    # BASELINE.json configs[0]: 8 utterances x 200 frames, 1-layer BiGRU(128), greedy decode
    "config1_greedy": dict(U=8, T=200, beam=1, scale=8.0,
                           net=dict(num_features=40, dims_bidir=[128], subsample=[1], dim_dec=128, conv_n=100,
                                    conv_num_filters=10, num_phonemes=32, post_merge_dims=[128], maxout_pieces=2)),
    # configs[2]: WSJ-shaped, 32 utterances x 800 frames, beam_size = 10, char-level output
    "config3_beam10": dict(U=32, T=800, beam=10, scale=8.0, net=NET),
}
SEARCH_METRIC = "beam-search utterances/sec at 32x800frx40fb, WSJ architecture, beam_size=10 (configs[2])"


def search_values(shapes, seed=1):
    """'Trained-like' weights (init_values) with a sharper readout so that hypotheses of many lengths finish."""
    v = init_values(shapes, seed=seed)
    v["/recognizer/generator/readout/post_merge/mlp/linear_0.W"] *= 10.0
    v["/recognizer/generator/readout/post_merge/mlp/linear_0.b"][-1] = 1.0        # eos = V - 1
    return v


def search_bench(pkg, torch, dev, rank, world, steps, warmup, dist_mod, barrier, cpu_baseline=True):
    """Decode U utterances per GPU with BeamSearch.search_many (device-resident hypotheses, k-best on the GPU);
    wall clock around the call (recordings start in HOST memory: the encoder H2D copy is inside), max over ranks."""
    out = {}
    lib = pkg._lib.load()
    for name, case in SEARCH_CASES.items():
        net = case["net"]
        rec = pkg.SpeechRecognizer(
            input_dims={"recordings": 40}, input_num_chars={}, eos_label=31, num_phonemes=32, dim_dec=net["dim_dec"],
            dims_bidir=net["dims_bidir"], subsample=net["subsample"], conv_n=net["conv_n"],
            conv_num_filters=net["conv_num_filters"], dim_matcher=net.get("dim_matcher"),
            post_merge_dims=net["post_merge_dims"], post_merge_activation=pkg.Maxout(2),
            max_decoded_length_scale=case["scale"], data_prepend_eos=False,
            enc_transition=pkg.GatedRecurrent, dec_transition=pkg.GatedRecurrent, device=dev)
        values = search_values(rec.parameter_shapes())
        rec.set_parameter_values(values)
        rec.init_beam_search(case["beam"])
        rng = np.random.RandomState(99 + rank)
        lens = rng.randint(int(0.6 * case["T"]), case["T"] + 1, size=case["U"])
        lens[0] = case["T"]
        utts = [rng.normal(size=(int(t), 40)).astype(np.float32) for t in lens]
        inputs = [{"recordings": u} for u in utts]
        res = None
        for _ in range(max(1, warmup)):
            res = rec.beam_search_many(inputs, raise_on_failure=False)
        barrier()
        lib.lvsr_launch_count(1)
        t0 = time.perf_counter()
        for _ in range(steps):
            res = rec.beam_search_many(inputs, raise_on_failure=False)
        torch.cuda.synchronize(dev)
        ms = max_over_ranks((time.perf_counter() - t0) * 1e3, world, dev, dist_mod) / steps
        launches = int(lib.lvsr_launch_count(1)) // max(1, steps)
        found = [r for r in res if r is not None]
        tok = [len(r[0][0]) for r in found]
        entry = {"utterances_per_s": case["U"] * world / (ms * 1e-3), "frames_per_s": float(lens.sum()) * world / (ms * 1e-3),
                 "ms_per_batch": ms, "utterances_per_gpu": case["U"], "beam_size": case["beam"], "max_frames": case["T"],
                 "decoded": len(found), "mean_best_length": float(np.mean(tok)) if tok else 0.0,
                 "gpu_launches_per_batch": launches}
        if cpu_baseline and rank == 0:
            from oracle import lvsr_oracle as O
            cfg = O.make_config(max_decoded_length_scale=case["scale"], **net)
            p32 = {k: v.astype(np.float32) for k, v in values.items()}
            n = 1 if case["beam"] > 1 else 2
            t0 = time.perf_counter()
            same = 0
            for u, r in list(zip(utts, res))[:n]:
                try:
                    o = O.beam_search(cfg, p32, u, case["beam"])
                    same += int(r is not None and o[0][0] == r[0][0])
                except O.CandidateNotFoundError:
                    same += int(r is None)
            dt = time.perf_counter() - t0
            entry["cpu_oracle_utterances_per_s"] = n / dt
            entry["cpu_oracle_sample"] = "%d utterance(s), float32 numpy restatement of BeamSearch.search" % n
            entry["best_hypothesis_identical_to_cpu_oracle"] = "%d/%d" % (same, n)
        out[name] = entry
        del rec
    return out


STRESS_NET = dict(num_features=40, dims_bidir=[256, 256, 256], subsample=[1, 1, 1], dim_dec=256, dim_matcher=512, conv_n=100,
                  conv_num_filters=10, num_phonemes=63, post_merge_dims=[256], maxout_pieces=2)
STRESS_WORKLOAD = dict(B=16, T=2000, F=40, L=60, V=63)       # BASELINE.json configs[4]: 128 utterances over 8 GPUs
STRESS_METRIC = "encoder+decoder frames/sec, TIMIT-shaped long utterances: batch 128 x 2000fr x 40fb over 8 GPUs (configs[4])"


def stress_bench(pkg, torch, dev, rank, world, steps, warmup, dist_mod, flush, barrier):
    """configs[4]: 16 utterances x 2000 frames per GPU, 3 x BiGRU(256) without subsampling (T' = 2000), 63 symbols,
    window_around_median(100, 100): teacher-forced cost; HBM GB/s of the decoder kernel and the tensor-core rate of the
    fork GEMMs against the measured peaks."""
    import ctypes as C
    W = STRESS_WORKLOAD
    rec = pkg.SpeechRecognizer(
        input_dims={"recordings": W["F"]}, input_num_chars={}, eos_label=W["V"] - 1, num_phonemes=W["V"],
        dim_dec=STRESS_NET["dim_dec"], dims_bidir=STRESS_NET["dims_bidir"], subsample=STRESS_NET["subsample"],
        conv_n=STRESS_NET["conv_n"], conv_num_filters=STRESS_NET["conv_num_filters"], dim_matcher=STRESS_NET["dim_matcher"],
        post_merge_dims=STRESS_NET["post_merge_dims"], post_merge_activation=pkg.Maxout(2),
        prior=dict(type="window_around_median", before=100, after=100),
        enc_transition=pkg.GatedRecurrent, dec_transition=pkg.GatedRecurrent, device=dev)
    rec.set_parameter_values(init_values(rec.parameter_shapes()))
    lib = pkg._lib.load()
    x, m, labels, lm = synthetic_batch(W["B"], W["T"], W["F"], W["L"], W["V"], seed=shard_seed(rank, base=777))
    xd, md = torch.as_tensor(x, device=dev), torch.as_tensor(m, device=dev)
    yd, ymd = torch.as_tensor(labels, device=dev), torch.as_tensor(lm, device=dev)

    def step():
        att, attm = rec.encode(xd, md)
        return rec.cost_matrix(yd, ymd, att, attm, return_all=True)
    for _ in range(max(3, warmup)):
        r = step()
    barrier()
    total = 0.0
    for _ in range(steps):
        flush.fill_(1)
        torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = step()
        b.record()
        torch.cuda.synchronize(dev)
        total += a.elapsed_time(b)
    ms = max_over_ranks(total, world, dev, dist_mod) / steps
    t0 = time.perf_counter()
    for _ in range(steps):
        rec.cost(x, m, labels, lm)
    ms_host = max_over_ranks((time.perf_counter() - t0) * 1e3, world, dev, dist_mod) / steps
    prof = {}
    lib.lvsr_profile_enable(1)
    r = step()
    torch.cuda.synchronize(dev)
    for cls in ("gemm", "bigru", "dec_scan", "attention", "window", "dense", "readout"):
        tot, cnt = C.c_double(), C.c_int64()
        lib.lvsr_profile_read(cls.encode(), C.byref(tot), C.byref(cnt))
        prof[cls] = {"ms": round(tot.value, 3), "launches": cnt.value}
    lib.lvsr_profile_enable(0)
    # the window actually attended: positions with non-zero alignment or inside the cut -> algorithmic bytes of the decoder
    w = r["weights"]                                  # [L, B, T']
    Tp = w.shape[2]
    nz = (w > 0).any(dim=1)                           # [L, T'] union over the batch = the batch-global cut, at least
    first = torch.where(nz.any(dim=1), nz.float().argmax(dim=1), torch.zeros_like(nz[:, 0], dtype=torch.long))
    last = torch.where(nz.any(dim=1), Tp - 1 - nz.flip(1).float().argmax(dim=1), torch.zeros_like(first))
    tw = (last - first + 1).float().mean().item()
    peaks, peak_src = measured_peaks()
    M, E = STRESS_NET["dim_matcher"], 2 * STRESS_NET["dims_bidir"][-1]
    persistent = prof["attention"]["launches"] == 0          # the class is recorded even when the planner declines the shape
    dec_ms = prof["dec_scan"]["ms"] if persistent else (prof["attention"]["ms"] + prof["dense"]["ms"] + prof["window"]["ms"])
    step_bytes = attention_step_bytes(W["B"], tw, M, E)
    hbm = step_bytes * W["L"] / (dec_ms * 1e-3) / 1e9 if dec_ms > 0 else 0.0
    gemm_flops, t_l, din = 0.0, W["T"], W["F"]
    for D in STRESS_NET["dims_bidir"]:
        gemm_flops += 2.0 * t_l * W["B"] * din * 6 * D
        din = 2 * D
    gemm_flops += 2.0 * Tp * W["B"] * E * M
    tf = gemm_flops / (prof["gemm"]["ms"] * 1e-3) / 1e12 if prof["gemm"]["ms"] > 0 else 0.0
    frames = W["B"] * W["T"] * world
    return {
        "metric": STRESS_METRIC, "value": frames / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms, "n_gpus": world,
        "steps": steps, "scaling": "weak", "dtype": "f32",
        "config": {"workload": "configs[4]: %d utterances x %d frames x %d fbank per GPU, 3 x BiGRU(256), no subsampling (T' = %d), "
                               "%d symbols, window_around_median(100,100), %d teacher-forced steps" % (W["B"], W["T"], W["F"], Tp, W["V"], W["L"]),
                   "global_batch": W["B"] * world, "parallelism": "dp%d (utterance shards, no data-path collective)" % world},
        "e2e": {"value": frames / (ms_host * 1e-3), "unit": "frames/s",
                "h2d_bytes_per_step": int(x.nbytes + m.nbytes + labels.nbytes + lm.nbytes), "d2h_bytes_per_step": int(W["L"] * W["B"] * 4)},
        "decoder": {"path": "persistent dec_scan_kernel" if persistent else
                            "step-wise kernels (window / att_step / dense): 16 rows x T' = 2000 needs 16 co-resident 8-CTA clusters "
                            "or 500-position chunks, neither fits (dec_scan.cu planner)",
                    "mean_window_positions": tw, "algorithmic_bytes_per_step": step_bytes, "us_per_step": dec_ms * 1e3 / W["L"],
                    "hbm_GBps": hbm, "hbm_frac_of_measured_peak": hbm / peaks["hbm_gbs"], "peak_source": peak_src},
        "fork_gemms": {"useful_tflops": tf, "tensor_pipe_frac_3xtf32": 3.0 * tf / (peaks["bf16_tflops"] / 2.0),
                       "note": "3 tf32 products per useful product (exact hi/lo split); tf32 dense peak taken as half the measured bf16 peak; "
                               "the time includes the hi/lo split passes and the readout-merge FFMA GEMMs"},
        "kernel_ms_per_step": prof,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mode", default="metric", choices=["metric", "train", "search", "stress"],
                    help="metric: the BASELINE headline (forward cost, teacher forcing) with a `train` block for the "
                         "training step; train: the training step (configs[3]) as the main line")
    ap.add_argument("--no-train", action="store_true", help="metric mode: skip the training-step block")
    ap.add_argument("--batch", type=int, default=WORKLOAD["B"],
                    help="diagnostic only: utterances per GPU (the metric is quoted on the default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="metric mode: write what the last timed step returned (costs [L,B], attended [T',B,E], "
                         "attended_mask [T',B]) for rank 0's shard as DIR/<name>.npy in float32, at most 64 MB "
                         "(the default batch takes 33 MB; a larger --batch keeps its first utterances)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.mode != "metric" or args.impl != "ours"):
        ap.error("--dump-outputs is only supported with --mode metric --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    W = dict(WORKLOAD, B=args.batch)
    config = {"workload": "configs[metric]: WSJ-shaped synthetic, batch %d x %d frames x %d fbank per GPU, "
                          "4-layer pyramidal BiGRU(256) + content+location attention + GRU(256) decoder, "
                          "%d teacher-forced steps" % (W["B"], W["T"], W["F"], W["L"]),
              "global_batch": W["B"] * world, "frames": W["T"], "parallelism": "dp%d (utterance shards)" % world,
              "l2": "L2 flushed (256 MiB write) between timed iterations"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        fps, ms, cb = cpu_reference_run(args.steps, 0)
        config["reference_sample_B"] = 64
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": 0, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": cb,
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    import torch
    import __graft_entry__ as graft
    pkg = graft.load_package()
    assert torch.cuda.is_available(), "bench.py needs a GPU"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    rec = pkg.SpeechRecognizer(
        input_dims={"recordings": W["F"]}, input_num_chars={}, eos_label=W["V"] - 1, num_phonemes=W["V"],
        dim_dec=NET["dim_dec"], dims_bidir=NET["dims_bidir"], subsample=NET["subsample"], conv_n=NET["conv_n"],
        conv_num_filters=NET["conv_num_filters"], dim_matcher=NET["dim_matcher"],
        post_merge_dims=NET["post_merge_dims"], post_merge_activation=pkg.Maxout(2),
        enc_transition=pkg.GatedRecurrent, dec_transition=pkg.GatedRecurrent, device=dev)
    rec.set_parameter_values(init_values(rec.parameter_shapes()))
    lib = pkg._lib.load()

    x, m, labels, lm = synthetic_batch(W["B"], W["T"], W["F"], W["L"], W["V"], seed=shard_seed(rank))
    xd, md = torch.as_tensor(x, device=dev), torch.as_tensor(m, device=dev)
    yd, ymd = torch.as_tensor(labels, device=dev), torch.as_tensor(lm, device=dev)
    xh, mh = torch.as_tensor(x).pin_memory(), torch.as_tensor(m).pin_memory()
    yh, ymh = torch.as_tensor(labels).pin_memory(), torch.as_tensor(lm).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step_device():
        att, attm = rec.encode(xd, md)
        return {"costs": rec.cost_matrix(yd, ymd, att, attm), "attended": att, "attended_mask": attm}

    def step_host():
        return rec.cost(xh.numpy(), mh.numpy(), yh.numpy(), ymh.numpy())

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        """Device time of `steps` calls and what the last call returned."""
        total_ms = 0.0
        for i in range(steps):
            flush.fill_(1)                       # evict L2 between timed iterations
            torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = fn()
            b.record()
            torch.cuda.synchronize(dev)
            total_ms += a.elapsed_time(b)
            if i < steps - 1:
                out = None                       # free it so that the next step reuses its memory
        return total_ms, out

    dist_mod = None
    if world > 1:
        import torch.distributed as dist_mod

    if args.mode in ("search", "stress"):
        sampler = ClockSampler(local_rank)
        sampler.start()
        if args.mode == "search":
            sr = search_bench(pkg, torch, dev, rank, world, args.steps, 1, dist_mod, barrier,
                              cpu_baseline=not args.no_cpu_baseline)
            main_case = sr["config3_beam10"]
            line = {"metric": SEARCH_METRIC, "value": main_case["utterances_per_s"], "unit": "utterances/s", "n_gpus": world,
                    "steps": args.steps, "warmup": 1, "ms_per_step": main_case["ms_per_batch"],
                    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "config": {"workload": "configs[2]: 32 utterances x <=800 frames per GPU, beam_size 10; configs[0] in `search`",
                               "parallelism": "dp%d (utterances sharded, no cross-device traffic)" % world},
                    "e2e": {"value": main_case["utterances_per_s"], "unit": "utterances/s",
                            "h2d_bytes_per_step": int(main_case["frames_per_s"] * main_case["ms_per_batch"] * 1e-3 / world * 40 * 4),
                            "d2h_bytes_per_step": 0, "note": "recordings start in host memory; value == e2e for this mode"},
                    "gpu_launches": main_case["gpu_launches_per_batch"], "search": sr}
        else:
            line = stress_bench(pkg, torch, dev, rank, world, args.steps, args.warmup, dist_mod, flush, barrier)
            line.update({"warmup": args.warmup, "higher_is_better": True, "vs_baseline": None, "data": "synthetic"})
        sampler.stop_flag.set()
        sampler.join(timeout=2)
        if rank == 0:
            line["clocks"] = sampler.summary()
            print(json.dumps(line))
        if world > 1:
            dist_mod.destroy_process_group()
        return 0

    if args.mode == "train":
        sampler = ClockSampler(local_rank)
        sampler.start()
        tr = train_bench(pkg, torch, dev, rank, world, args.steps, args.warmup, dist_mod, flush, barrier)
        sampler.stop_flag.set()
        sampler.join(timeout=2)
        if rank == 0:
            tr.update({"warmup": args.warmup, "higher_is_better": True, "vs_baseline": None, "data": "synthetic",
                       "gpu_launches": tr["gpu_launches_per_step"] * args.steps, "clocks": sampler.summary()})
            print(json.dumps(tr))
        if world > 1:
            dist_mod.destroy_process_group()
        return 0

    for _ in range(args.warmup):
        step_device()
    step_host()
    barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    lib.lvsr_launch_count(1)
    barrier()
    ms_dev, last = timed(step_device, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs({k: v.float().cpu().numpy() for k, v in last.items()}, args.dump_outputs)
    del last
    barrier()
    launches = int(lib.lvsr_launch_count(1))
    ms_dev = max_over_ranks(ms_dev, world, dev, dist_mod)

    # end to end through the host-buffer C-ABI call (wall clock around a synchronising call)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    torch.cuda.synchronize(dev)
    ms_host = max_over_ranks((time.perf_counter() - t0) * 1e3, world, dev, dist_mod)
    barrier()
    sampler.stop_flag.set()
    sampler.join(timeout=2)

    # per-kernel-class device time (second pass with CUDA events around every launch)
    prof = {}
    lib.lvsr_profile_enable(1)
    step_device()
    torch.cuda.synchronize(dev)
    import ctypes as C
    for cls in ("gemm", "bigru", "attention", "window", "dense", "dec_scan", "readout"):
        tot, cnt = C.c_double(), C.c_int64()
        lib.lvsr_profile_read(cls.encode(), C.byref(tot), C.byref(cnt))
        prof[cls] = {"ms": tot.value, "launches": cnt.value}
    lib.lvsr_profile_enable(0)

    train_block = None
    if not args.no_train and args.batch == WORKLOAD["B"]:
        try:
            train_block = train_bench(pkg, torch, dev, rank, world, args.steps, 2, dist_mod, flush, barrier)
        except Exception as e:          # the headline must survive a failure of the secondary measurement
            train_block = {"error": "%s: %s" % (type(e).__name__, e)}

    if rank != 0:
        if world > 1:
            dist_mod.destroy_process_group()
        return 0

    frames = W["B"] * W["T"] * world
    ms_step = ms_dev / args.steps
    value = frames / (ms_step * 1e-3)
    e2e_value = frames / (ms_host / args.steps * 1e-3)
    peaks, peak_src = measured_peaks()
    Tp = rec.encoded_length(W["T"])
    step_bytes = attention_step_bytes(W["B"], Tp, NET["dim_matcher"], 2 * NET["dims_bidir"][-1])
    if prof["dec_scan"]["launches"] > 0:
        # persistent decoder: one launch runs all L attention+GRU steps
        kern = "dec_scan_kernel (persistent attention+decoder scan, %d steps per launch)" % W["L"]
        launch_bytes = step_bytes * W["L"]
        k_us = prof["dec_scan"]["ms"] * 1e3 / prof["dec_scan"]["launches"]
        dec_us = k_us / W["L"]
    else:
        att = prof["attention"]
        kern = "att_step_kernel (attention step of the decoder)"
        launch_bytes = step_bytes
        k_us = att["ms"] * 1e3 / max(1, att["launches"])
        dec_us = (prof["attention"]["ms"] + prof["window"]["ms"] + prof["dense"]["ms"]) * 1e3 / max(1, att["launches"])
    achieved = launch_bytes / (k_us * 1e-6) / 1e9 if k_us > 0 else 0.0
    # the encoder recurrence has no bandwidth or tensor roofline (SURVEY.md 8d): report time per
    # sequential step next to the fp32 FMA time of its two dependent products
    enc_steps, t_l = 0, W["T"]
    for k in NET["subsample"]:
        enc_steps += t_l
        t_l = -(-t_l // k)
    D = NET["dims_bidir"][0]
    fma_per_step = 2 * W["B"] * 3 * D * D
    # D = 256: bigru_mma_kernel -- mma.sync m16n8k16 on fp16 head/tail splits (fp32-equivalent, DESIGN.md section 2);
    # per CTA and step 12 weight tiles x 16 k-steps x 2 MMAs at the measured 2.0 cycles per MMA and SM
    # (tools/micro/mma_rate.cu) = 768 cycles of tensor pipe
    recurrence = {"kernel": "bigru_mma_kernel" if D == 256 else "bigru_kernel", "sequential_steps": enc_steps,
                  "us_per_step": prof["bigru"]["ms"] * 1e3 / enc_steps if enc_steps else None,
                  "fp32_fma_floor_us": fma_per_step / (148 * 128 * 1.965e9) * 1e6,
                  "mma_sync_floor_us": (12 * (D // 16) * 2 * 2.0) / 1.965e9 * 1e6 if D == 256 else None}
    out = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
        "e2e": {"value": e2e_value, "unit": "frames/s",
                "h2d_bytes_per_step": int(x.nbytes + m.nbytes + labels.nbytes + lm.nbytes),
                "d2h_bytes_per_step": int(W["L"] * W["B"] * 4)},
        "gpu_launches": launches,
        "clocks": sampler.summary(),
        "roofline": {"bound": "hbm", "kernel": kern,
                     "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / peaks["hbm_gbs"],
                     "traffic": (NCU_DEC_SCAN["dram_bytes"] if (prof["dec_scan"]["launches"] > 0 and
                                 (W["B"], W["T"], W["L"]) == NCU_DEC_SCAN["config"]) else None),
                     "traffic_source": NCU_DEC_SCAN["source"],
                     "l2_to_sm_GBps": (NCU_DEC_SCAN["l2_to_sm_bytes"] / (k_us * 1e-6) / 1e9
                                       if (prof["dec_scan"]["launches"] > 0 and k_us > 0 and
                                           (W["B"], W["T"], W["L"]) == NCU_DEC_SCAN["config"]) else None),
                     "binds": "latency (dependent phases at 25 % occupancy); P and H are L2-resident (hit rate 70 %), "
                              "HBM moves about half the algorithmic bytes",
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": launch_bytes, "us_per_launch": k_us,
                     "decoder_step_us": dec_us,
                     "decoder_step_frac": (step_bytes / (dec_us * 1e-6) / 1e9 / peaks["hbm_gbs"]) if dec_us > 0 else 0.0,
                     "how": "CUDA events around every launch of the class in a separate profiled pass",
                     "encoder_recurrence": recurrence},
        "kernel_ms_per_step": {k: round(v["ms"], 3) for k, v in prof.items()},
        "kernel_launches_per_step": {k: v["launches"] for k, v in prof.items()},
    }
    if train_block is not None:
        out["train"] = train_block
    if not args.no_cpu_baseline:
        _, _, cb = cpu_reference_run(1, 0, sample_B=16)
        out["cpu_baseline"] = cb
    print(json.dumps(out))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
