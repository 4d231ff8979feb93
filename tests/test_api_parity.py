"""Every public top-level name (and public method) of the original fms-fsdp's modules must exist under the same import path
(`fms_fsdp.*` aliases to `fms_fsdp_b200.*`) and take the same parameters.  The original's names and parameter names are
stored in tests/golden/reference/api.json (scripts/make_reference_golden.py regenerates it from a checkout)."""
import importlib
import json
import os

import pytest

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "api.json")) as _f:
    API = json.load(_f)
MODULES = {
    "fms_fsdp/config/training.py": "fms_fsdp.config.training",
    "fms_fsdp/utils/config_utils.py": "fms_fsdp.utils.config_utils",
    "fms_fsdp/utils/train_utils.py": "fms_fsdp.utils.train_utils",
    "fms_fsdp/utils/checkpointing_utils.py": "fms_fsdp.utils.checkpointing_utils",
    "fms_fsdp/utils/dataloader_utils.py": "fms_fsdp.utils.dataloader_utils",
    "fms_fsdp/utils/dataset_utils.py": "fms_fsdp.utils.dataset_utils",
    "fms_fsdp/policies/ac_handler.py": "fms_fsdp.policies.ac_handler",
    "fms_fsdp/policies/mixed_precision.py": "fms_fsdp.policies.mixed_precision",
    "fms_fsdp/policies/wrapping.py": "fms_fsdp.policies.wrapping",
    "fms_fsdp/policies/param_init.py": "fms_fsdp.policies.param_init",
    "speculator/train_speculator_utils.py": "speculator.train_speculator_utils",
    "speculator/train_speculator.py": "speculator.train_speculator",
    "fms_to_hf_llama.py": "fms_to_hf_llama",
    "fms_to_hf_mamba.py": "fms_to_hf_mamba",
    "main_training_llama.py": "main_training_llama",
    "main_training_mamba.py": "main_training_mamba",
}


@pytest.mark.parametrize("path,mod", sorted(MODULES.items()))
def test_public_names_of_reference_module_exist(path, mod):
    ref = API[path]
    ours = importlib.import_module(mod)
    missing = [name for name in ref["functions"] if not hasattr(ours, name)]
    for name, methods in ref["classes"].items():
        if name.startswith("_"):
            continue
        if not hasattr(ours, name):
            missing.append(name)
            continue
        cls = getattr(ours, name)
        missing += [f"{name}.{m}" for m in methods if not m.startswith("_") and not hasattr(cls, m)]
    missing += [name for name in ref["names"] if not hasattr(ours, name)]
    assert not missing, f"{mod} lacks {missing}"


@pytest.mark.parametrize("path,mod", sorted(MODULES.items()))
def test_signatures_accept_the_reference_call_forms(path, mod):
    """Every public function / method (and ``__init__``) takes the original's parameters under the same names and, unless it
    takes ``*args``, at the same positions -- so both keyword and positional call sites of existing users keep working."""
    import inspect
    ref = API[path]
    ours = importlib.import_module(mod)
    problems = []

    def check(sig, obj, label):
        try:
            params = list(inspect.signature(obj).parameters.values())
        except (TypeError, ValueError):
            return
        names = [p.name for p in params if p.name not in ("self", "cls")]
        var_kw = any(p.kind == p.VAR_KEYWORD for p in params)
        var_pos = any(p.kind == p.VAR_POSITIONAL for p in params)
        for i, n in enumerate(sig["pos"]):
            if n not in names:
                if not var_kw:
                    problems.append(f"{label}: no parameter {n}")
            elif names.index(n) != i and not var_pos:
                problems.append(f"{label}: {n} is parameter {names.index(n)}, reference has it at {i}")
        problems.extend(f"{label}: no keyword {n}" for n in sig["kwonly"] if n not in names and not var_kw)

    for name, sig in ref["functions"].items():
        if hasattr(ours, name):
            check(sig, getattr(ours, name), name)
    for name, methods in ref["classes"].items():
        if hasattr(ours, name):
            cls = getattr(ours, name)
            for m, sig in methods.items():
                if hasattr(cls, m):
                    check(sig, getattr(cls, m), f"{name}.{m}")
    assert not problems, f"{mod}: {problems}"
