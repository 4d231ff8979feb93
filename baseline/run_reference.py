"""`bench.py --impl reference`: drive the UNMODIFIED reference (pip --target baseline/_ref) on the headline
config through its own public API and stock code path -- its `train_config`, `get_model_config`,
`get_policies`, `get_dummy_loader`, torch FSDP wrap exactly as its `main_training_llama.py:82-115`, its
`train()` loop (torch.compile as in its defaults).  None of the B200 engine is imported.

Outcome of the offline install (also recorded in DESIGN.md): `pip install --no-index ... /root/reference` fails
on the missing `ibm-fms` requirement; `--no-deps` installs `fms_fsdp` + `speculator`.  `ibm-fms` and `fire` cannot
be installed (no index), so `baseline/fms_shim/` provides plain-PyTorch stand-ins for the handful of fms classes
the reference imports.  Timing: the K timed steps are ONE call of the reference's `train()` (which moves each
batch host->device and reads the loss back every step, i.e. it is inherently end-to-end), bracketed by
barrier + synchronize and CUDA events, max over ranks.
"""
import argparse
import contextlib
import io
import json
import math
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
# reference first, shim second; the repo root (our own fms_fsdp alias) must NOT shadow the reference
sys.path = [os.path.join(HERE, "_ref"), os.path.join(HERE, "fms_shim")] + [
    p for p in sys.path if os.path.abspath(p or ".") != os.path.dirname(HERE)]
for k in [k for k in sys.modules if k == "fms_fsdp" or k.startswith("fms_fsdp.")]:
    del sys.modules[k]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--model", default="llama2_7b")
    ap.add_argument("--seq", type=int, default=4096)
    ap.add_argument("--batch", type=int, default=2)
    ap.add_argument("--no_compile", action="store_true")
    ap.add_argument("--ac", default="0", help="selective activation checkpointing fraction (reference --selective_checkpointing)")
    a = ap.parse_args()

    import torch
    import torch.distributed as dist
    import torch.optim as optim
    from torch.distributed.fsdp import FullyShardedDataParallel as FSDP
    from torch.optim.lr_scheduler import LambdaLR

    os.environ.setdefault("RANK", "0"); os.environ.setdefault("WORLD_SIZE", "1"); os.environ.setdefault("LOCAL_RANK", "0")
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1"); os.environ.setdefault("MASTER_PORT", "29533")
    local_rank, rank, world = int(os.environ["LOCAL_RANK"]), int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])

    try:
        from fms.models.llama import LLaMA, LLaMABlock
        from fms_fsdp import config
        from fms_fsdp.utils.config_utils import get_model_config, update_config
        from fms_fsdp.utils.dataloader_utils import get_dummy_loader
        from fms_fsdp.utils.train_utils import get_policies, setup, setup_environ_flags, train
        import fms_fsdp
        assert os.path.join("baseline", "_ref") in fms_fsdp.__file__, fms_fsdp.__file__
    except Exception as e:  # reference not importable at all
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": f"reference import failed: {e!r}"[:300]}))
        return

    if a.model.startswith("mamba"):
        # the reference's Mamba entry point needs mamba_ssm (CUDA extension package; not in the image, no index access)
        try:
            import mamba_ssm  # noqa: F401
            why = "baseline/run_reference.py drives the reference's Llama entry point only"
        except Exception as e:
            why = f"mamba_ssm is not installed ({e!r})"
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": why[:300]}))
        return

    if a.model.startswith("qwen"):
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "the reference model zoo has no Qwen2 (q/k/v-bias) variant"}))
        return

    cfg = config.train_config()
    update_config(cfg, model_variant=a.model, use_dummy_dataset=True, sharding_strategy="fsdp", seq_length=a.seq,
                  batch_size=a.batch, low_cpu_fsdp=True, use_torch_compile=not a.no_compile,
                  report_interval=max(a.steps, a.warmup),   # one report per train() call, never per step
                  num_steps=a.warmup, vocab_size=32000, fsdp_activation_checkpointing=(a.ac not in ("0", "0.0", "")),
                  selective_checkpointing=a.ac, checkpoint_interval=10 ** 9)
    torch.cuda.manual_seed(cfg.seed); torch.manual_seed(cfg.seed)
    setup()
    torch.cuda.set_device(local_rank); torch.cuda.empty_cache()
    setup_environ_flags()
    mp_policy, wrapping_policy, sharding, apply_ac, param_init_fn = get_policies(cfg, rank, LLaMABlock)
    llama_config = get_model_config(cfg.model_variant)
    with torch.device("meta"):
        model = LLaMA(llama_config)
    train_loader = get_dummy_loader(cfg, rank, world)
    model = FSDP(model, auto_wrap_policy=wrapping_policy, mixed_precision=mp_policy, sharding_strategy=sharding,
                 use_orig_params=cfg.use_torch_compile, device_id=torch.cuda.current_device(), limit_all_gathers=True,
                 param_init_fn=param_init_fn)
    model.rot_emb.compute_freqs_cis(torch.device("cuda", torch.cuda.current_device()), model.config.max_expected_seq_len)
    if cfg.fsdp_activation_checkpointing:      # reference main_training_llama.py:99-102
        apply_ac(model, p=cfg.selective_checkpointing)
    compiled = False
    if cfg.use_torch_compile:
        torch._dynamo.config.accumulated_cache_size_limit = 128
        model = torch.compile(model)
        compiled = True
    optimizer = optim.AdamW(model.parameters(), lr=cfg.learning_rate, betas=(0.9, 0.95), weight_decay=0.1)
    warm = min(2000, 1000000 // 20)
    schedule = lambda x: min(1 - (1 - min(x, warm) / warm) ** 2,
                             0.1 + 0.5 * (1 - 0.1) * (1 + math.cos(min(x, 1000000) / 1000000 * math.pi)))
    scheduler = LambdaLR(optimizer, lambda x: schedule(x))

    class _NoCkpt:  # the loop insists on saving at the final step; a 7B checkpoint is not part of the metric
        def save(self, *a, **k):
            return None

    def run_train(start, stop):
        cfg.num_steps = stop
        cfg.report_interval = stop   # stock loop; the only multiple of `stop` in (start, stop] is the last step, so there
        #                              is exactly one report, at the end: loss = mean over the steps of this call
        sink = io.StringIO()
        with contextlib.redirect_stdout(sink):
            return train(cfg, model, local_rank, rank, train_loader, optimizer, scheduler, None, _NoCkpt(), start, 0)

    try:
        run_train(0, a.warmup)
    except Exception as e:
        if compiled:  # fall back to eager once (and say so)
            model = model._orig_mod
            compiled = False
            run_train(0, a.warmup)
        else:
            raise
    dist.barrier(); torch.cuda.synchronize()
    sampler = None
    if rank == 0:   # same nvidia-smi clock / throttle sampling as the other arm, during the timed region only
        try:
            root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
            if root not in sys.path:
                sys.path.insert(0, root)
            from bench import ClockSampler
            sampler = ClockSampler(local_rank)
            sampler.start()
        except Exception:
            sampler = None
    try:
        from bench import DATA_NOTE, bench_config
    except Exception:
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        sys.path.insert(0, root)
        from bench import DATA_NOTE, bench_config
    try:
        from bench import PUBLISHED_TOK_S_GPU as PUB
    except Exception:
        PUB = {"llama2_7b": 9600.0}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss = run_train(a.warmup, a.warmup + a.steps)
    e1.record()
    dist.barrier(); torch.cuda.synchronize()
    clocks = sampler.stop() if sampler is not None else None
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = ms.item() / a.steps
    value = a.batch * a.seq * world / (ms_step / 1e3)
    if rank == 0:
        print(json.dumps({
            "metric": "tokens/sec (Llama2-7B FSDP seq4k bs2)" if a.model == "llama2_7b" else f"tokens/sec ({a.model})",
            "value": round(value, 1), "unit": "tokens/s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(ms_step, 3),
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": (round(value / world / PUB[a.model], 4) if a.model in PUB else None),
            "dtype": "bf16", "data": DATA_NOTE, "impl": "reference",
            "tokens_per_sec_per_gpu": round(value / world, 1),
            "config": bench_config(a.model, a.batch * world, a.seq, f"fsdp{world}", a.ac),
            "details": {"torch_compile": compiled, "stack": "torch FSDP1 + cuBLAS + SDPA + NCCL",
                        "deps": "ibm-fms/fire absent offline -> plain-torch stand-ins in baseline/fms_shim; reference code unmodified"},
            "loss_steps": [a.warmup + 1, a.warmup + a.steps],
            "e2e": {"value": round(value, 1), "unit": "tokens/s",
                    "note": "the reference train() loop is inherently end-to-end (per-step H2D of the batch, loss.item())",
                    "h2d_bytes_per_step": a.batch * a.seq * 4 * 2, "d2h_bytes_per_step": 8},
            "gpu_launches": 0,   # none of this repo's kernels run in the reference arm (library / inductor kernels only)
            "clocks": clocks,
            "loss": float(loss) if loss is not None else None,
            "mem_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2),
        }), flush=True)
    dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    main()
