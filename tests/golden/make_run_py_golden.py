"""Generate tests/golden/run_py_search_call.json: the call that the original project's unmodified bin/run.py makes
into compat/ for `run.py search <tmp>/missing.tar <tmp>/base.yaml monitoring.search.beam_size 2` on the toy
experiment of tests/compat_helpers.py:

    imports             the (module, name) pairs run.py imports at its top level and before dispatching
    logging_level       the level run.py hands to logging.basicConfig
    configuration_args  the positional arguments of its lvsr.config.Configuration(...) call
    cmd_args            config['cmd_args'] as run.py sets it
    func, kwargs        the lvsr.main function it dispatches to and the keyword arguments it passes

The temporary directory is stored as "<tmp>".  Needs a checkout of rizar/attention-lvcsr (Python-3 readable
bin/run.py); nothing else of it is imported.  Run from the repo root:

    python tests/golden/make_run_py_golden.py <attention-lvcsr checkout>
"""
import ast
import json
import logging
import os
import runpy
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from compat_helpers import COMPAT, write_experiment  # noqa: E402

sys.path.insert(0, COMPAT)
OUT = os.path.join(ROOT, "tests", "golden", "run_py_search_call.json")


class Dispatched(Exception):
    pass


def imports_of(path):
    pairs = []
    for node in ast.walk(ast.parse(open(path).read())):
        if isinstance(node, ast.ImportFrom):
            pairs += [[node.module, a.name] for a in node.names]
        elif isinstance(node, ast.Import):
            pairs += [[a.name, None] for a in node.names]
    return sorted(p for p in pairs if p[0].split(".")[0] in ("lvsr", "blocks", "picklable_itertools"))


def main():
    run_py = os.path.join(sys.argv[1], "bin", "run.py")
    tmp = tempfile.mkdtemp()
    exp = write_experiment(tmp)
    import lvsr.config
    import lvsr.main
    rec = {}
    real_init = lvsr.config.Configuration.__init__

    def init(self, *args):
        rec["configuration_args"] = [args[0], args[1], [list(c) for c in args[2]]]
        real_init(self, *args)

    def search(config, **kwargs):
        rec.update(cmd_args=config["cmd_args"], func="search", kwargs=kwargs)
        raise Dispatched()

    lvsr.config.Configuration.__init__, lvsr.main.search = init, search
    argv = ["search", os.path.join(tmp, "missing.tar"), exp["base"], "monitoring.search.beam_size", "2"]
    sys.argv = [run_py] + argv
    try:
        runpy.run_path(run_py, run_name="__main__")
    except Dispatched:
        pass
    rec["logging_level"] = logging.getLevelName(logging.getLogger().level)
    rec["argv"] = argv
    rec["imports"] = imports_of(run_py)
    text = json.dumps(rec, indent=1, sort_keys=True, default=list).replace(tmp, "<tmp>")
    with open(OUT, "w") as f:
        f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
