"""Multi-GPU check (torchrun, one rank per GPU): fused NVLink collectives vs c10d/NCCL.
 1. raw kernels: p2p all-gather / pull reduce-scatter on 7B-block-sized buffers, numerics + bus bandwidth
 2. engine: same model/data trained with collective_impl=fused and =torch must agree
Rank 0 prints the results as one JSON line and, given a second argument, also writes them to that file:
    python -m torch.distributed.run --nproc-per-node N scripts/gpu_multi_check.py all [OUT.json]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

rank, world, lrank = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lrank)
dev = torch.device("cuda", lrank)
dist.init_process_group("nccl", device_id=dev)
out = {"world": world}


def timed(fn, iters=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / iters], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.item()


from fms_fsdp_b200.parallel.mesh import build_mesh
from fms_fsdp_b200.parallel.comm import TorchCollectives
from fms_fsdp_b200.parallel.fused_comm import FusedCollectives

mode = sys.argv[1] if len(sys.argv) > 1 else "all"
if mode in ("all", "raw"):
    mesh = build_mesh("fsdp")
    fc, tc = FusedCollectives(mesh, dev), TorchCollectives(mesh, dev)
    n_full = 202383360 // (world * 64) * (world * 64)  # one Llama2-7B block
    n_sh = n_full // world
    torch.manual_seed(rank)
    sh = fc.alloc_shard(n_sh, torch.bfloat16); sh.copy_(torch.randn(n_sh, device=dev))
    full_a = torch.empty(n_full, dtype=torch.bfloat16, device=dev); full_b = torch.empty_like(full_a)
    fc.begin_step(); fc.all_gather(sh, full_a); tc.all_gather(sh, full_b); torch.cuda.synchronize()
    out["allgather_equal"] = bool(torch.equal(full_a, full_b))
    ms_f = timed(lambda: fc.all_gather(sh, full_a)); ms_t = timed(lambda: tc.all_gather(sh, full_b))
    bytes_in = n_full * 2 * (world - 1) / world
    out["allgather"] = dict(fused_ms=ms_f, nccl_ms=ms_t, fused_GBs_in=bytes_in / ms_f / 1e6, nccl_GBs_in=bytes_in / ms_t / 1e6)
    g = fc.alloc_full(n_full, torch.bfloat16); g.copy_(torch.randn(n_full, device=dev) * 0.01)
    o_f = torch.zeros(n_sh, device=dev); o_t = torch.zeros(n_sh, device=dev)
    sq_f = torch.zeros((), device=dev); sq_t = torch.zeros((), device=dev)
    fc.reduce_scatter(g, o_f, 1.0 / world, sq_f); tc.reduce_scatter(g, o_t, 1.0 / world, sq_t); torch.cuda.synchronize()
    out["reduce_scatter_maxdiff"] = (o_f - o_t).abs().max().item()
    out["reduce_scatter_ref_absmax"] = o_t.abs().max().item()
    out["sumsq"] = [sq_f.item(), sq_t.item()]
    ms_f = timed(lambda: fc.reduce_scatter(g, o_f, 1.0 / world, None)); ms_t = timed(lambda: tc.reduce_scatter(g, o_t, 1.0 / world, None))
    out["reduce_scatter"] = dict(fused_ms=ms_f, nccl_ms=ms_t, fused_GBs_in=bytes_in / ms_f / 1e6, nccl_GBs_in=bytes_in / ms_t / 1e6)
    del fc, tc, full_a, full_b, g

if mode in ("all", "ag"):
    # raw fused all-gather GEMM: y = x W^T where W is gathered from the peers INSIDE the GEMM kernel
    from fms_fsdp_b200.ops import cuda_kernels as CK
    mesh = build_mesh("fsdp")
    fc = FusedCollectives(mesh, dev)
    N, Kd, Mx = 12288, 4096, 8192
    n_full = (N * Kd + 65536) // (world * 64) * (world * 64)
    n_sh = n_full // world
    torch.manual_seed(rank)
    sh = fc.alloc_shard(n_sh, torch.bfloat16); sh.copy_(torch.randn(n_sh, device=dev) * 0.02)
    full_ref = torch.empty(n_full, dtype=torch.bfloat16, device=dev)
    fc.begin_step(); fc.all_gather(sh, full_ref)
    x = torch.randn(Mx, Kd, device=dev).bfloat16()
    res = {}
    for dep in (True, False):
        full = torch.zeros(n_full, dtype=torch.bfloat16, device=dev)
        W = full[:N * Kd].view(N, Kd)
        Wref = full_ref[:N * Kd].view(N, Kd)
        req = fc.ag_request(sh, full, 0, n_full * 2, dep)
        CK.push_ag_request(req)
        if not dep:   # prefetch mode: the GEMM reads an already-complete weight, the gather fills `full`
            y = CK.gemm(x, Wref, "nt")
        else:
            y = CK.gemm(x, W, "nt")
        torch.cuda.synchronize()
        yref = CK.gemm(x, Wref, "nt")
        res["dep" if dep else "prefetch"] = dict(consumed=bool(req["consumed"]), gathered_equal=bool(torch.equal(full, full_ref)),
                                                  y_maxdiff=(y.float() - yref.float()).abs().max().item())
        def run():
            r = fc.ag_request(sh, full, 0, n_full * 2, dep); CK.push_ag_request(r); CK.gemm(x, W if dep else Wref, "nt")
        ms = timed(run)
        res["dep_ms" if dep else "prefetch_ms"] = ms
    res["plain_gemm_ms"] = timed(lambda: CK.gemm(x, Wref, "nt"))
    res["standalone_allgather_ms"] = timed(lambda: fc.all_gather(sh, full_ref))
    res["bytes_in_MB"] = n_full * 2 * (world - 1) / world / 1e6
    out["ag_gemm"] = res
    del fc

if mode in ("all", "push"):
    # fused wgrad GEMM -> reduce-scatter: the GEMM epilogue pushes every tile into the OWNER rank's staging slot over
    # NVLink (128-byte bulk stores, or 16-byte st.global as the reference), then a LOCAL slot sum == reduce-scatter.
    from fms_fsdp_b200.ops import cuda_kernels as CK
    mesh = build_mesh("fsdp")
    fc = FusedCollectives(mesh, dev)
    C = fc.C
    T, N, Kd = 8192, 4096, 11008                     # dW [N, Kd] = dy^T x  (the down projection of Llama2-7B)
    total = N * Kd // (world * 64) * (world * 64)
    n = total // world
    torch.manual_seed(100 + rank)
    dy = (torch.randn(T, N, device=dev) * 0.05).bfloat16(); x = (torch.randn(T, Kd, device=dev) * 0.05).bfloat16()
    staging = fc.shard.alloc(world * n, torch.bfloat16); staging.zero_()
    table = fc.shard.table_of(staging)               # base address of every rank's staging buffer
    slots = torch.tensor([staging.data_ptr() + s_ * n * 2 for s_ in range(world)], dtype=torch.int64, device=dev)
    mine = torch.empty(n, dtype=torch.float32, device=dev)
    ref_local = CK.gemm(dy, x, "tn").float().reshape(-1)             # this rank's full wgrad (bf16-rounded like the push)
    dist.all_reduce(ref_local)
    ref = ref_local[rank * n:(rank + 1) * n]
    res = {}
    for bulk, rotate in ((True, True), (True, False), (False, True)):
        staging.zero_()
        fc.shard.barrier(C, fc._anchor)
        def push():
            C.set_gemm_push(table, n, 0, rank, bulk, world if rotate else 1)
            C.gemm_push(dy, x)                           # layout tn, push epilogue
        push()
        fc.shard.barrier(C, fc._anchor)                  # every rank's tiles have landed in my slots
        C.reduce_scatter(slots, mine, 0, world, 0, True, 1.0, None)     # local 'world'-way sum of the slots
        torch.cuda.synchronize()
        key = ("bulk" if bulk else "direct") + ("_rot" if rotate else "")
        res[key] = dict(maxdiff=(mine - ref).abs().max().item(), absmax=ref.abs().max().item(), push_gemm_ms=timed(push))
    res["plain_gemm_ms"] = timed(lambda: CK.gemm(dy, x, "tn"))
    res["local_slot_sum_ms"] = timed(lambda: C.reduce_scatter(slots, mine, 0, world, 0, True, 1.0, None))
    res["pushed_MB_out"] = total * 2 * (world - 1) / world / 1e6
    sc = torch.tensor([float(rank + 1)], device=dev)
    fc.shard.scalar_allreduce(C, sc); torch.cuda.synchronize()
    res["scalar_allreduce"] = [sc.item(), world * (world + 1) / 2]
    out["push_wgrad"] = res
    del fc

if mode in ("all", "engine", "gn"):
    from fms_fsdp_b200.models.llama import LLaMA, LLaMAConfig
    from fms_fsdp_b200.parallel import ShardedAdamW, ShardedModel
    from fms_fsdp_b200.policies import bfSixteen

    def run(impl, strategy, shard=0, steps=4, fused_gather="1"):
        os.environ["FMS_B200_FUSED_GATHER"] = fused_gather
        torch.manual_seed(0); torch.cuda.manual_seed(0)
        cfg = LLaMAConfig(src_vocab_size=4096, emb_dim=1024, nheads=8, kvheads=4, nlayers=4, multiple_of=256, max_expected_seq_len=512)
        with torch.device("meta"):
            m = LLaMA(cfg)
        eng = ShardedModel(m, sharding_strategy=strategy, hsdp_shard_size=shard, mixed_precision=bfSixteen, device=dev, collective_impl=impl)
        opt = ShardedAdamW(eng, lr=1e-3)
        res = []
        for st in range(steps):
            g = torch.Generator().manual_seed(100 * st + rank)
            x = torch.randint(0, 4096, (2, 512), generator=g).to(dev)
            loss = eng.forward_backward(x, x)
            gn = eng.clip_grad_norm_(1.0)
            opt.step()
            res.append((loss.item(), gn.item()))
        sd = eng.full_state_dict(cpu=False)
        chk = sum(v.double().sum().item() for v in sd.values())
        return res, chk

    if mode == "engine" or True:
        # per-unit gradient comparison after ONE backward (same weights, same data)
        def grads(impl):
            torch.manual_seed(0); torch.cuda.manual_seed(0)
            cfg = LLaMAConfig(src_vocab_size=4096, emb_dim=1024, nheads=8, kvheads=4, nlayers=4, multiple_of=256, max_expected_seq_len=512)
            with torch.device("meta"):
                m = LLaMA(cfg)
            eng = ShardedModel(m, sharding_strategy="fsdp", mixed_precision=bfSixteen, device=dev, collective_impl=impl)
            g = torch.Generator().manual_seed(rank)
            x = torch.randint(0, 4096, (2, 512), generator=g).to(dev)
            eng.forward_backward(x, x)
            torch.cuda.synchronize()
            gs = {u.name: u.grad_shard.clone() for u in eng.units}
            out.setdefault("gnorm_sq_check", {})[impl] = dict(engine=eng._gnorm_sq.item(), from_shards=sum(v.double().pow(2).sum().item() for v in gs.values()),
                                                             clip=eng.clip_grad_norm_(1.0).item())
            return gs, eng
        ga, ea = grads("fused"); gb, eb = grads("torch")
        rep = {}
        for k in ga:
            d = (ga[k] - gb[k]).abs()
            rep[k] = dict(maxdiff=d.max().item(), absmax=gb[k].abs().max().item(), n_bad=int((d > 0.02 * gb[k].abs().max()).sum().item()),
                          sumsq=[ga[k].pow(2).sum().item(), gb[k].pow(2).sum().item()], first_bad=int(torch.nonzero(d > 0.02 * gb[k].abs().max())[0].item()) if (d > 0.02 * gb[k].abs().max()).any() else -1,
                          numel=ga[k].numel())
        out["unit_grad_diff"] = rep
        u = ea.root
        out["root_slots"] = [(s.name, s.offset, s.numel) for s in u.layout.slots] + [("total", u.layout.total, u.layout.shard_numel)]
        del ga, gb, ea, eb
    combos = [("fsdp", 0)] + ([("ddp", 0)] if world <= 4 else []) + ([("hsdp", world // 2)] if world >= 4 else [])
    if mode == "gn":
        combos = []
    for strat, shard in combos:
        a, ca = run("fused", strat, shard); b, cb = run("torch", strat, shard)
        out[f"engine_{strat}"] = dict(fused=a, torch=b, param_checksum=[ca, cb])
        if strat == "fsdp":
            os.environ["FMS_B200_PUSH_RS"] = "0"; os.environ["FMS_B200_ASYNC_OPT_SHARDED"] = "0"
            d_, cd = run("fused", strat, shard)
            os.environ["FMS_B200_PUSH_RS"] = "1"; os.environ["FMS_B200_ASYNC_OPT_SHARDED"] = "1"
            out["engine_fsdp_fused_pull_syncopt"] = dict(res=d_, checksum=cd)
            c, cc = run("fused", strat, shard, fused_gather="0")
            from fms_fsdp_b200.ops import cuda_kernels as CK
            out["engine_fsdp_fused_nogemmgather"] = dict(res=c, checksum=cc, ag_stats=dict(CK.AG_STATS))

if rank == 0:
    if len(sys.argv) > 2:
        with open(sys.argv[2], "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps(out))
dist.barrier(); dist.destroy_process_group()
