"""Regenerate ``tests/golden/reference/``: what the tests that compare with the original fms-fsdp compare against.

    python scripts/make_reference_golden.py --reference PATH/TO/fms-fsdp

The original project is only needed here, once; the tests read the stored results.  Every file written is data: names and
parameter names of the public API, file hashes, model-zoo numbers, token streams and loader checkpoints.  Modules of the
original that import ``fms`` run against the stand-ins in ``baseline/fms_shim`` (as ``bench.py --impl reference`` does).
"""
import argparse
import ast
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tarfile
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "reference")
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

API_MODULES = [
    "fms_fsdp/config/training.py", "fms_fsdp/utils/config_utils.py", "fms_fsdp/utils/train_utils.py",
    "fms_fsdp/utils/checkpointing_utils.py", "fms_fsdp/utils/dataloader_utils.py", "fms_fsdp/utils/dataset_utils.py",
    "fms_fsdp/policies/ac_handler.py", "fms_fsdp/policies/mixed_precision.py", "fms_fsdp/policies/wrapping.py",
    "fms_fsdp/policies/param_init.py", "speculator/train_speculator_utils.py", "speculator/train_speculator.py",
    "fms_to_hf_llama.py", "fms_to_hf_mamba.py", "main_training_llama.py", "main_training_mamba.py",
]
AC_FRACTIONS = ["1/7", "1/4", "1/3", "2/5", "1/2", "3/5", "2/3", "3/4", "9/10", "1"]
AC_DEPTHS = [10, 24, 32, 40, 48, 80]


def _dump(name, obj):
    """One top-level key per line: small files, readable diffs."""
    with open(os.path.join(OUT, name), "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v, sort_keys=True)}" for k, v in sorted(obj.items()))
                + "\n}\n")


def _run_reference(ref, code):
    """Run ``code`` in a fresh interpreter that imports ``fms_fsdp`` from the original, not this repository."""
    head = (f"import sys\nsys.path = [{ref!r}, {os.path.join(ROOT, 'baseline', 'fms_shim')!r}] + "
            f"[p for p in sys.path if p not in ('', {ROOT!r})]\n")
    r = subprocess.run([sys.executable, "-c", head + code], capture_output=True, text=True, cwd="/", timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.split("OUT", 1)[1])


def _signature(fn):
    a = fn.args
    return {"pos": [x.arg for x in a.posonlyargs + a.args if x.arg not in ("self", "cls")], "kwonly": [x.arg for x in a.kwonlyargs]}


def api(ref):
    """Public functions, classes (with ``__init__`` and public methods) and module-level names, with parameter names."""
    out = {}
    for path in API_MODULES:
        tree = ast.parse(open(os.path.join(ref, path)).read())
        mod = {"functions": {}, "classes": {}, "names": []}
        for node in tree.body:
            if isinstance(node, ast.FunctionDef) and not node.name.startswith("_"):
                mod["functions"][node.name] = _signature(node)
            elif isinstance(node, ast.ClassDef):
                mod["classes"][node.name] = {b.name: _signature(b) for b in node.body if isinstance(b, ast.FunctionDef)
                                             and (b.name == "__init__" or not b.name.startswith("_"))}
            elif isinstance(node, ast.Assign):
                mod["names"] += [t.id for t in node.targets if isinstance(t, ast.Name) and not t.id.startswith("_")]
        out[path] = mod
    _dump("api.json", out)


def sources(ref):
    """SHA-256 of every Python file of the original ``fms_fsdp`` package (what ``baseline/_ref`` must hold)."""
    src = os.path.join(ref, "fms_fsdp")
    out = {}
    for dirpath, _, files in os.walk(src):
        for f in files:
            if f.endswith(".py"):
                p = os.path.join(dirpath, f)
                out[os.path.relpath(p, src)] = hashlib.sha256(open(p, "rb").read()).hexdigest()
    _dump("fms_fsdp_sources.json", out)


def ac_selection(ref):
    """Which blocks the original ``apply_fsdp_checkpointing`` wraps, per depth and fraction ("1" = wrapped)."""
    code = (
        "import json, torch.nn as nn\n"
        "from fms_fsdp.policies import ac_handler as ac\n"
        "from torch.distributed.algorithms._checkpoint.checkpoint_wrapper import CheckpointWrapper\n"
        "class Blk(nn.Linear):\n    pass\n"
        "out = {}\n"
        f"for n in {AC_DEPTHS!r}:\n"
        f"    for p in {AC_FRACTIONS!r}:\n"
        "        m = nn.Sequential(*[Blk(2, 2) for _ in range(n)])\n"
        "        ac.apply_fsdp_checkpointing(m, Blk, p)\n"
        "        out[f'{n}:{p}'] = ''.join('1' if isinstance(c, CheckpointWrapper) else '0' for c in m)\n"
        "print('OUT' + json.dumps(out))\n")
    _dump("ac_selection.json", _run_reference(ref, code))


def model_zoo(ref):
    """Every variant the original ``get_model_config`` knows, as a dict of its fields."""
    import re
    src = os.path.join(ref, "fms_fsdp", "utils", "config_utils.py")
    variants = sorted(set(re.findall(r'model_variant == "([a-z0-9_.]+)"', open(src).read())))
    code = (
        "import json, dataclasses\n"
        "from fms_fsdp.utils.config_utils import get_model_config\n"
        "out = {}\n"
        f"for v in {variants!r}:\n"
        "    c = get_model_config(v)\n"
        "    out[v] = c if isinstance(c, dict) else dataclasses.asdict(c)\n"
        "print('OUT' + json.dumps(out))\n")
    _dump("model_zoo.json", _run_reference(ref, code))


def train_config(ref):
    """The original ``train_config`` defaults and five batches of its ``get_dummy_loader`` (rank 1 of 4)."""
    code = (
        "import json, dataclasses\n"
        "from fms_fsdp.config import train_config\n"
        "from fms_fsdp.utils.dataloader_utils import get_dummy_loader\n"
        "c = train_config(); c.seq_length, c.batch_size, c.vocab_size = 16, 2, 50\n"
        "it = iter(get_dummy_loader(c, 1, 4))\n"
        "batches = [[t.tolist() for t in next(it)] for _ in range(5)]\n"
        "print('OUT' + json.dumps({'cfg': dataclasses.asdict(train_config()), 'batches': batches}))\n")
    _dump("train_config.json", _run_reference(ref, code))


def datasets(ref):
    """What the original's ``dataset_utils`` yields in each ``test_datasets`` comparison, as line digests, and the loader
    checkpoints crossing between the two implementations: for one written here, its digest (the test checks it is still
    written the same) and the original's continuation from it; those written by the original are stored whole, in
    ``loader_checkpoints.tar.xz``."""
    import importlib.util

    import fms_fsdp_b200.utils.dataset_utils as OURS
    import test_datasets as T

    spec = importlib.util.spec_from_file_location("_reference_dataset_utils",
                                                  os.path.join(ref, "fms_fsdp", "utils", "dataset_utils.py"))
    REF = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(REF)
    corpus, text = T.make_corpus(), T.make_text_corpus()[0]
    stored = tempfile.mkdtemp()
    g = {"stream": T._line_digests(iter(T._full_stack(REF, corpus, 0, 1)), 300),
         "text_reader": T._line_digests(iter(T._text_reader(REF, text)), 200)}
    for kw in T.PACKER_KW:
        g[f"packer {kw!r}"] = T._line_digests(iter(T._packer_stack(REF, corpus, kw)), 250)
    for case in T.PARTITION_CASES:
        if case[3] < 60:
            g[f"partition {case!r}"] = T._line_digests(iter(T._partition_stack(REF, corpus, *case)), 150)
    with tempfile.TemporaryDirectory() as tmp:
        ck = os.path.join(tmp, "ours_to_ref")
        T._write_checkpoint(OURS, corpus, ck)
        g["ours_to_ref checkpoint"] = T._checkpoint_digests(ck)
        g["ours_to_ref"] = T._resume(REF, corpus, 2, ck)
        ck = os.path.join(stored, "ref_to_ours")
        T._write_checkpoint(REF, corpus, ck)
        g["ref_to_ours"] = T._resume(REF, corpus, 4, ck)
        for writer_is_ours, old_world, new_world in T.RESCALE_CASES:
            key = f"rescale {(writer_is_ours, old_world, new_world)!r}"
            if writer_is_ours:
                ck = os.path.join(tmp, key)
                T._rescale_write(OURS, corpus, old_world, ck)
                g[key + " checkpoint"] = T._checkpoint_digests(ck)
            else:
                ck = os.path.join(stored, f"rescale_{old_world}_to_{new_world}")
                T._rescale_write(REF, corpus, old_world, ck)
            g[key] = T._rescale_resume(REF, corpus, new_world, ck)
        g["multi_worker"] = T._worker_run(REF, corpus, os.path.join(tmp, "multi_worker"))
    with tarfile.open(os.path.join(OUT, "loader_checkpoints.tar.xz"), "w:xz") as tar:
        for name in sorted(os.listdir(stored)):
            tar.add(os.path.join(stored, name), arcname=name)
    for d in (corpus, text, stored):
        shutil.rmtree(d)
    _dump("datasets.json", g)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reference", required=True, help="checkout of foundation-model-stack/fms-fsdp")
    ref = os.path.abspath(ap.parse_args().reference)
    os.makedirs(OUT, exist_ok=True)
    for make in (api, sources, ac_selection, model_zoo, train_config, datasets):
        make(ref)
        print("wrote", make.__name__)


if __name__ == "__main__":
    main()
