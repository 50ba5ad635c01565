"""compat/: the reference's import names over the engine (SURVEY.md 8b b1) -- host-only checks."""
import os
import subprocess
import sys

from compat_helpers import COMPAT, ROOT, write_experiment


def _import_compat():
    if COMPAT not in sys.path:
        sys.path.insert(0, COMPAT)
    import lvsr.config as C
    return C


def test_configuration_parent_changes_and_stages(tmp_path):
    """lvsr/config.py:9-92: parent links are merged recursively, command-line changes are parsed as YAML,
    stages are ordered by `number` and each stage is the base configuration plus its changes."""
    C = _import_compat()
    exp = write_experiment(tmp_path)
    cfg = C.Configuration(exp["child"], "$LVSR/lvsr/configs/schema.yaml",
                          [("net.conv_n", "6"), ("monitoring.search.beam_size", "5")])
    assert cfg["net"]["dims_bidir"] == [128] and cfg["net"]["conv_n"] == 6          # parent + change
    assert cfg["monitoring"]["search"]["beam_size"] == 5
    assert cfg["training"]["num_batches"] == 3 and cfg["training"]["gradient_threshold"] == 10.0
    assert cfg.multi_stage and list(cfg.ordered_stages) == ["pretraining", "main"]
    assert cfg.ordered_stages["pretraining"]["training"]["num_batches"] == 2
    assert cfg.ordered_stages["main"]["training"]["scale"] == 0.5 and "stages" not in cfg.ordered_stages["main"]
    # YAML python tags resolve to the engine's configuration tokens
    import _engine
    assert isinstance(cfg["net"]["post_merge_activation"], _engine.pkg.Maxout)
    assert cfg["net"]["post_merge_activation"].num_pieces == 2
    assert cfg["net"]["enc_transition"] is _engine.pkg.GatedRecurrent
    assert isinstance(cfg["initialization"]["/recognizer"]["rec_weights_init"], _engine.pkg.Orthogonal)


def test_dataset_batches_are_time_major_padded_and_masked(tmp_path):
    _import_compat()
    from lvsr.datasets import Data
    exp = write_experiment(tmp_path)
    data = Data(path=exp["npz"], batch_size=4, sort_k_batches=2)
    assert data.num_labels == 12 and data.eos_label == 11 and data.num_features == 40
    n = 0
    for b in data.batches("train"):
        T, B, F = b["recordings"].shape
        assert b["recordings_mask"].shape == (T, B) and b["labels"].shape[1] == B and b["labels"].dtype.kind == "i"
        last = b["labels_mask"].sum(axis=0).astype(int) - 1
        assert (b["labels"][last, range(B)] == data.eos_label).all()            # eos appended (datasets/__init__.py:267-270)
        assert (b["recordings"][b["recordings_mask"] == 0] == 0).all()
        n += B
    assert n == 10


# Replays a call recorded from the reference's bin/run.py (tests/golden/make_run_py_golden.py): its imports, then
# Configuration(...) and lvsr.main.<func>(config, **kwargs) with exactly the arguments run.py passed.
RUN_PY_REPLAY = r"""
import importlib, json, logging, sys
call = json.loads(open(sys.argv[1]).read().replace("<tmp>", sys.argv[2]))
for module, name in call["imports"]:
    if name:
        getattr(importlib.import_module(module), name)
logging.basicConfig(level=call["logging_level"], format="%(asctime)s: %(name)s: %(levelname)s: %(message)s")
from lvsr.config import Configuration
import lvsr.main
path, schema, changes = call["configuration_args"]
config = Configuration(path, schema, [tuple(c) for c in changes])
config["cmd_args"] = call["cmd_args"]
getattr(lvsr.main, call["func"])(config, **call["kwargs"])
"""


def test_reference_run_py_runs_unchanged_up_to_the_device(tmp_path):
    """The call the reference's UNMODIFIED bin/run.py makes for `run.py search <tmp>/missing.tar <tmp>/base.yaml
    monitoring.search.beam_size 2` with PYTHONPATH=compat (recorded in tests/golden/run_py_search_call.json):
    its imports resolve, Configuration and lvsr.main.search accept its arguments; without a GPU the first device
    call fails loudly (no CPU fallback)."""
    write_experiment(tmp_path)
    env = dict(os.environ, PYTHONPATH=COMPAT, CUDA_VISIBLE_DEVICES="")
    call = os.path.join(ROOT, "tests", "golden", "run_py_search_call.json")
    r = subprocess.run([sys.executable, "-c", RUN_PY_REPLAY, call, str(tmp_path)], env=env, capture_output=True,
                       text=True, timeout=300)
    out = r.stdout + r.stderr
    assert "Recognizer initialization started" in out, out[-2000:]
    assert r.returncode != 0 and ("CUDA" in out or "cuda" in out), out[-2000:]
    assert ROOT in out or "attention-lvcsr_b200" in out or "lvsr_b200" in out
