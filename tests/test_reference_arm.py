"""Fairness of the reference arm of ``bench.py`` (``baseline/run_reference.py``): ``ibm-fms`` cannot be installed offline, so
the unmodified reference trains a plain-PyTorch stand-in of the few ``fms`` classes it imports (``baseline/fms_shim``).  The
stand-in must be the SAME model as this repo's LLaMA: same state-dict keys, same logits, same gradients."""
import os
import sys

import pytest
import torch

from fms_fsdp_b200.models.llama import LLaMA, LLaMAConfig

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("kv,theta", [(0, 10000.0), (2, 500000.0)])
def test_stand_in_fms_llama_equals_this_repos_llama(kv, theta):
    sys.path.insert(0, os.path.join(ROOT, "baseline", "fms_shim"))
    try:
        from fms.models.llama import LLaMA as ShimLLaMA, LLaMAConfig as ShimConfig
    finally:
        sys.path.pop(0)
    kw = dict(src_vocab_size=128, emb_dim=64, nheads=4, kvheads=kv, nlayers=2, multiple_of=16, max_expected_seq_len=64,
              rope_theta=theta)
    torch.manual_seed(0)
    ours = LLaMA(LLaMAConfig(**kw)); ours.reset_parameters()
    shim = ShimLLaMA(ShimConfig(**kw))
    sd = ours.state_dict()
    assert set(shim.state_dict().keys()) == set(sd.keys())
    shim.load_state_dict(sd)
    x = torch.randint(0, 128, (2, 24))
    lo, ls = ours(x), shim(x)
    assert torch.allclose(lo, ls, atol=1e-5, rtol=1e-4), (lo - ls).abs().max()
    w = torch.randn_like(lo)
    (lo * w).sum().backward()
    (ls * w).sum().backward()
    go = dict(ours.named_parameters())
    for n, p in shim.named_parameters():
        assert torch.allclose(go[n].grad, p.grad, atol=1e-5, rtol=1e-3), (n, (go[n].grad - p.grad).abs().max())


def test_reference_arm_runs_the_unmodified_reference():
    """The install the reference arm imports (``baseline/_ref``, when present) holds the original ``fms_fsdp`` package byte
    for byte: every file's SHA-256 is in tests/golden/reference/fms_fsdp_sources.json."""
    import hashlib
    import json
    inst = os.path.join(ROOT, "baseline", "_ref", "fms_fsdp")
    if not os.path.isdir(inst):
        pytest.skip("the reference arm's install baseline/_ref is not present")
    with open(os.path.join(ROOT, "tests", "golden", "reference", "fms_fsdp_sources.json")) as f:
        want = json.load(f)
    assert len(want) >= 12
    for rel, digest in want.items():
        path = os.path.join(inst, rel)
        assert os.path.exists(path), path
        with open(path, "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == digest, path
