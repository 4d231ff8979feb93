#!/usr/bin/env python
"""Headline benchmark: tokens/sec for Llama2-7B FSDP, seq 4096, per-GPU batch 2, bf16, synthetic data
(BASELINE.json; the reference's `use_dummy_dataset` stream, reference dataloader_utils.py:36-57).

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus 8 --steps 10 --warmup 3
    python bench.py --impl reference ...      # the unmodified reference from baseline/_ref

Prints ONE JSON line on rank 0.  `value` = whole-job tokens/s from a device-timed region (CUDA events,
barrier + synchronize on both sides, max over ranks) of exactly K optimizer steps with device-resident
inputs; `e2e` = the same K steps driven through the public training-step API with, every step, the
host->device copy of that step's tokens/labels from pinned memory and a device->host read of the loss.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BASELINE_TOK_S_GPU = 9600.0  # BASELINE.md: Llama2-7B on 96x H100, reference README.md:16 (best published)
# best published tokens/s/GPU per model (BASELINE.md section 1, H100 column); models without a published number -> null
PUBLISHED_TOK_S_GPU = {"llama2_7b": 9600.0, "llama2_13b": 4850.0, "llama2_34b": 1830.0, "llama2_70b": 890.0}


def _args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=8)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--model", default="llama2_7b")
    p.add_argument("--seq", type=int, default=4096)
    p.add_argument("--batch", type=int, default=2)
    p.add_argument("--sharding", default="fsdp")
    p.add_argument("--hsdp_shard_size", type=int, default=0)
    p.add_argument("--collective_impl", default="auto")
    p.add_argument("--ac", default="0", help="selective activation checkpointing fraction, e.g. 0, 1/2, 1")
    p.add_argument("--precision", default="bf16", choices=["bf16", "fp8"],
                   help="fp8 = opt-in e4m3 forward GEMMs; the result is flagged non-headline")
    p.add_argument("--nlayers", type=int, default=0, help="debug only: override depth (result is flagged invalid)")
    p.add_argument("--trace", default="", help="with --profile: also export the chrome trace of the 2 profiled steps")
    p.add_argument("--profile", default="", help="write a per-kernel device-time table of 2 extra steps to this path")
    p.add_argument("--dump-outputs", default="", metavar="DIR",
                   help="after the device-timed steps, write what the last of them computed to DIR/<name>.npy")
    return p.parse_args()


DATA_NOTE = "synthetic (reference get_dummy_loader stream, random-init weights)"


def bench_config(model, global_batch, seq, parallelism, ac):
    """The SAME keys (and, for the same run, values) in both arms."""
    return {"model": model, "global_batch": global_batch, "seq_len": seq, "parallelism": parallelism,
            "selective_ac": str(ac), "data_stream": "get_dummy_loader (arange windows mod vocab, label == input)",
            "l2": "per-step working set (>=13.5 GB of weights+activations) >> 126 MB L2; no explicit flush"}


DUMP_SAMPLE = 4096   # values kept per parameter tensor by --dump-outputs


def dump_outputs(out_dir, eng, loss, grad_norm, rank):
    """Write what one training step returned and updated, as float32 ``.npy`` files: ``loss``, ``grad_norm`` and, for every
    parameter, ``param.<name>`` = the fp32 master weights after the optimizer step at DUMP_SAMPLE positions drawn from a
    fixed seed (all of a smaller tensor).  Same arguments, same inputs: two builds can be compared file by file.  The step
    is not bitwise reproducible (some kernels accumulate with atomics), so compare with a tolerance: two runs of one build
    on a B200 (1000 W) differed by 1e-4 relative in the loss and 3e-6 absolute in the weights.  Every rank takes part in
    the parameter gathers; rank 0 writes."""
    import numpy as np
    import torch

    arrays = {"loss": loss, "grad_norm": grad_norm}
    gen = torch.Generator().manual_seed(0)
    for u in eng.units:
        flat = eng.gather_unit_full(u, "master")
        for name, v in eng.named_unit_views(u, flat):
            v = v.reshape(-1)
            if v.numel() > DUMP_SAMPLE:
                v = v[torch.randint(v.numel(), (DUMP_SAMPLE,), generator=gen).sort().values.to(v.device)]
            arrays[f"param.{name}"] = v
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for name, t in arrays.items():
            np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def run_ours(a):
    import torch
    import torch.distributed as dist

    from fms_fsdp_b200.config import train_config
    from fms_fsdp_b200.models.llama import LLaMA, LLaMABlock
    from fms_fsdp_b200.parallel import ShardedAdamW, ShardedModel
    from fms_fsdp_b200.policies import apply_fsdp_checkpointing, bfSixteen
    from fms_fsdp_b200.utils.config_utils import get_model_config
    from fms_fsdp_b200.utils.train_utils import lr_schedule_fn, model_flops_per_token, peak_tflops

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == a.gpus, f"--gpus {a.gpus} but WORLD_SIZE={world}"
    torch.manual_seed(2023)
    torch.cuda.manual_seed(2023)

    from fms_fsdp_b200.ops.functional import set_gemm_precision
    set_gemm_precision(a.precision)
    mcfg = get_model_config(a.model)
    is_mamba = a.model.startswith("mamba")
    cfg = train_config()
    cfg.num_steps = 1000000
    from fms_fsdp_b200.policies.ac_handler import parse_fraction
    if is_mamba:
        # secondary (non-headline) configuration: Mamba2 hybrid of the reference's main_training_mamba.py
        from fms_fsdp_b200.models.mamba import Block, MambaConfig, MambaLMHeadModel
        mc = MambaConfig(**mcfg)
        if a.nlayers:
            mc.n_layer = a.nlayers
            mc.attn_layer_idx = [i for i in mc.attn_layer_idx if i < a.nlayers]
        cfg.seq_length, cfg.batch_size, cfg.vocab_size = a.seq, a.batch, mc.vocab_size
        with torch.device("meta"):
            model = MambaLMHeadModel(mc)
        if parse_fraction(a.ac) > 0:
            apply_fsdp_checkpointing(model, Block, a.ac)
        n_layers, width = mc.n_layer, mc.d_model
    else:
        if a.nlayers:
            mcfg.nlayers = a.nlayers
        cfg.seq_length, cfg.batch_size, cfg.vocab_size = a.seq, a.batch, mcfg.src_vocab_size
        with torch.device("meta"):
            model = LLaMA(mcfg)
        if parse_fraction(a.ac) > 0:
            apply_fsdp_checkpointing(model, LLaMABlock, a.ac)
        n_layers, width = mcfg.nlayers, mcfg.emb_dim
    eng = ShardedModel(model, sharding_strategy=a.sharding, hsdp_shard_size=a.hsdp_shard_size,
                       mixed_precision=bfSixteen, device=dev, collective_impl=a.collective_impl)
    if not is_mamba:
        model.rot_emb.compute_freqs_cis(dev, mcfg.max_expected_seq_len)
    opt = ShardedAdamW(eng, lr=cfg.learning_rate, betas=(0.9, 0.95), weight_decay=0.1)
    import copy
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lr_schedule_fn(copy.copy(cfg)))   # frozen 1M-step schedule

    from fms_fsdp_b200.ops import cuda_kernels as CK
    from fms_fsdp_b200.utils.dataloader_utils import get_dummy_loader
    from fms_fsdp_b200.utils.train_utils import train

    # BOTH arms read the reference's dummy stream through the same call: get_dummy_loader(cfg, rank, world)
    # (reference dataloader_utils.py:36-57: sample k = arange(k*S, (k+1)*S) % V, label == input, same on every rank)
    loader = get_dummy_loader(cfg, rank, world)

    def step_device(tok, lab):
        loss = eng.forward_backward(tok, lab)
        gn = eng.clip_grad_norm_(cfg.grad_clip_thresh)
        opt.step()
        sched.step()
        return loss, gn

    # device-resident copies of the batches of the warm-up and of the device-timed region (a different batch every step)
    dev_batches = []
    for _ in range(a.warmup + a.steps):
        tok, lab = next(loader)
        dev_batches.append((tok.to(dev), lab.to(dev).long()))

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    class _NoCkpt:   # train() insists on saving at the final step; a 7B checkpoint is not part of the metric
        def save(self, *args, **kw):
            return None

    def run_train(start_step, n_steps, source):
        """n_steps optimizer steps through the PUBLIC loop (train_utils.train, what main_training_llama.main calls)."""
        cfg.checkpoint_interval = 10 ** 9
        cfg.use_dummy_dataset = True
        cfg.num_steps = start_step + n_steps
        cfg.report_interval = max(1, cfg.num_steps)     # exactly one report (and its stats all-reduce), at the last step
        sink = contextlib.nullcontext() if os.environ.get("FMS_B200_BENCH_VERBOSE") \
            else contextlib.redirect_stdout(open(os.devnull, "w"))
        with sink:
            return train(cfg, eng, local_rank, rank, source, opt, sched, None, _NoCkpt(), start_step, 0)

    # warm-up: W - 1 steps on device-resident batches + 1 step through the public loop (its one-time costs -- page-locked
    # staging arena, events, tracker init -- belong to warm-up exactly like the kernels' first launches)
    for i in range(a.warmup - 1):
        loss, _ = step_device(*dev_batches[i])
    if a.warmup >= 1:
        run_train(a.warmup - 1, 1, iter([tuple(t.cpu() for t in (dev_batches[a.warmup - 1][0], dev_batches[a.warmup - 1][1].int()))]))
    sync_all()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    CK.reset_launch_count()
    CK.reset_fallback_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    e0.record()
    loss_sum = torch.zeros((), device=dev)
    for i in range(a.steps):
        loss, gn = step_device(*dev_batches[a.warmup + i])
        loss_sum += loss
    e1.record()
    sync_all()
    launches = CK.launch_count()
    fallbacks = CK.fallback_count()
    peak_alloc = torch.cuda.max_memory_allocated(dev)   # train() below resets the peak counters at its report step
    loss_timed = float(loss_sum) / a.steps      # mean loss of steps W+1 .. W+K (what the reference arm prints too)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, eng, loss, gn, rank)
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = ms.item() / a.steps

    # ---- end-to-end: K more steps through the PUBLIC training loop, fms_fsdp_b200.utils.train_utils.train()
    # (the call main_training_llama.main() makes): every step it copies that step's batch host -> device from pinned
    # staging memory and reads the step's loss back device -> host (4-byte async read-back, checked one step later).
    del dev_batches
    start_step = a.warmup + a.steps
    sync_all()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    last = run_train(start_step, a.steps, loader)
    f1.record()
    sync_all()
    ms2 = torch.tensor([f0.elapsed_time(f1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    ms_step_e2e = ms2.item() / a.steps
    clocks = sampler.stop() if rank == 0 else None

    tokens_per_step = a.batch * a.seq * world
    value = tokens_per_step / (ms_step / 1e3)
    e2e = tokens_per_step / (ms_step_e2e / 1e3)
    n_params = eng.param_count()
    flops_tok = model_flops_per_token(n_params, n_layers, width, a.seq)
    mfu = value / world * flops_tok / 1e12 / peak_tflops()
    par = {"fsdp": f"fsdp{world}", "hsdp": f"hsdp{world // eng.mesh.shard_size}x{eng.mesh.shard_size}",
           "ddp": f"ddp{world}"}.get(a.sharding, a.sharding)
    if rank == 0:
        out = {
            "metric": "tokens/sec (Llama2-7B FSDP seq4k bs2)" if a.model == "llama2_7b" else f"tokens/sec ({a.model})",
            "value": round(value, 1), "unit": "tokens/s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(ms_step, 3),
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": (round(value / world / PUBLISHED_TOK_S_GPU[a.model], 4) if a.model in PUBLISHED_TOK_S_GPU else None),
            "dtype": "bf16" if a.precision == "bf16" else "fp8-e4m3 forward GEMMs, bf16 backward", "data": DATA_NOTE,
            "impl": "ours",
            "tokens_per_sec_per_gpu": round(value / world, 1), "mfu_vs_measured_bf16_peak": round(mfu, 4),
            # mean loss over the K device-timed steps (optimizer steps W+1..W+K): directly comparable with the other arm
            "loss": round(loss_timed, 4), "loss_steps": [a.warmup + 1, a.warmup + a.steps],
            "loss_e2e": round(float(last), 4), "grad_norm": round(float(gn), 4),
            "config": bench_config(a.model, a.batch * world, a.seq, par, a.ac),
            "details": {"n_params": n_params, "collectives": eng.coll.name, "attn_impl": CK.ATTN_IMPL,
                        "gemm_impl": CK.GEMM_IMPL, "push_reduce_scatter": bool(getattr(eng, "_push_rs", False)),
                        "async_sharded_optimizer": bool(getattr(eng, "_async_sharded", False))},
            "e2e": {"value": round(e2e, 1), "unit": "tokens/s", "ms_per_step": round(ms_step_e2e, 3),
                    "api": "fms_fsdp_b200.utils.train_utils.train (the loop of main_training_llama.main)",
                    # tokens + labels, int32, copied from pinned staging memory every step; loss read back every step
                    "h2d_bytes_per_step": 2 * a.batch * a.seq * 4, "d2h_bytes_per_step": 4},
            "gpu_launches": int(launches),
            "aten_fallbacks": int(fallbacks),
            "clocks": clocks,
            # peak of torch's caching allocator, and what the DEVICE reports as in use at the end (adds the symmetric-memory
            # buffers of the peer collectives, the allocator's cache and the CUDA context)
            "mem_gb": round(max(peak_alloc, torch.cuda.max_memory_allocated(dev)) / 2**30, 2),
            "mem_device_gb": round((lambda fr_to: (fr_to[1] - fr_to[0]) / 2**30)(torch.cuda.mem_get_info(dev)), 2),
        }
        if a.nlayers:
            out["invalid"] = "debug depth override"
        if a.precision != "bf16":
            out["invalid"] = "reduced-precision run (opt-in fp8 forward GEMMs): not the headline metric"
        if fallbacks:
            out["invalid"] = f"{fallbacks} ops of the timed region ran on the ATen fallback: {dict(CK.FALLBACKS)}"
        if a.model != "llama2_7b" or a.seq != 4096 or a.batch != 2:
            out["note"] = "secondary configuration, not the BASELINE headline"
        print(json.dumps(out), flush=True)
    if a.profile:
        # per-kernel device-time table of two more steps (never part of a reported number)
        from torch.profiler import ProfilerActivity, profile
        ctx = profile(activities=[ProfilerActivity.CUDA]) if rank == 0 else contextlib.nullcontext()
        with ctx as prof:
            for i in range(2):
                tok, lab = next(loader)
                step_device(tok.to(dev), lab.to(dev).long())
            sync_all()
        if rank == 0:
            os.makedirs(os.path.dirname(a.profile) or ".", exist_ok=True)
            with open(a.profile, "w") as f:
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=60, max_name_column_width=90))
            if a.trace:
                prof.export_chrome_trace(a.trace)     # timeline for scripts/trace_gaps.py
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_reference(a):
    """Run the UNMODIFIED reference (baseline/_ref) for the same metric/config.  See baseline/README.md."""
    runner = os.path.join(ROOT, "baseline", "run_reference.py")
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "fms_fsdp")):
        if int(os.environ.get("RANK", 0)) == 0:
            print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref not installed (pip --target failed or not run)"}))
        return
    sys.argv = [runner, "--gpus", str(a.gpus), "--steps", str(a.steps), "--warmup", str(a.warmup),
                "--model", a.model, "--seq", str(a.seq), "--batch", str(a.batch), "--ac", str(a.ac)]
    import runpy
    runpy.run_path(runner, run_name="__main__")


if __name__ == "__main__":
    args = _args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
