#!/usr/bin/env python
"""bench.py — ResNet-50 training under RayStrategy, gradient sync on libb2d (driver contract).

    python bench.py --gpus N --steps K --warmup W            # our arm (N>1: launched by torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU/gloo path
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR  # + the last step's loss / parameters / gradients

Workload (BASELINE.json configs[1]): torchvision resnet50 (random init, seed 0), synthetic
224x224 images, per-GPU batch 64, bf16 autocast, SGD momentum, DDP with
find_unused_parameters=False / gradient_as_bucket_view=True / bucket_cap_mb=25 — driven through
``RayStrategy``'s worker-side path (the same calls RayLauncher._wrapping_function makes), whose
DDP comm hook is libb2d's fused allreduce.  One "step" = forward + backward (+ per-bucket
gradient sync, overlapped) + optimizer step on every rank.  Weak scaling: per-GPU batch fixed.

Output: ONE JSON line on rank 0 (keys documented in DESIGN.md §8).
"""
import argparse
import json
import os
import socket
import statistics
import subprocess
import sys
import threading
import time
from contextlib import closing

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec, ResNet-50 RayStrategy (+ allreduce bus GB/s)"
NVLINK_NOMINAL_GBS = 900.0    # NVLink 5, per direction per GPU
EVIDENCE_TIMEOUT_S = 420     # link probe + parity + sweep + CPU baseline normally take about a minute
NVLINK_FALLBACK_GBS = 770.0   # /opt/skills/guides/B200_PROFILING.md: measured peer copy — used only if the in-run probe fails


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: 64 resnet, 16 bert, 4 gpt2)")
    ap.add_argument("--bucket-cap-mb", type=int, default=25)
    ap.add_argument("--wire", default="bf16", choices=["bf16", "fp32"],
                    help="bf16 = BASELINE.json's configuration (the strategy's own default is the reference's fp32)")
    ap.add_argument("--algo", default="auto")
    ap.add_argument("--mem", default="vmm", choices=["vmm", "ipc"])
    ap.add_argument("--max-ctas", type=int, default=None)
    ap.add_argument("--model", default="resnet50", choices=["resnet50", "resnet18", "bert-base", "gpt2-medium"])
    ap.add_argument("--strategy", default="ddp", choices=["ddp", "sharded"],
                    help="ddp = RayStrategy; sharded = RayShardedStrategy (fused reduce-scatter + Adam + all-gather)")
    ap.add_argument("--hook", default="b200", choices=["b200", "nccl_bf16", "nccl_fp32"],
                    help="b200 = libb2d; nccl_* = the reference's GPU path through the same strategy (A/B)")
    ap.add_argument("--seq", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the multi-GPU parity block (N > 1)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the short allreduce sweep vs NCCL / symm_mem (N > 1)")
    ap.add_argument("--chunk-mb", type=int, default=None, help="staged exchange: wire MiB per pipeline chunk")
    ap.add_argument("--exch-ctas", type=int, default=None)
    ap.add_argument("--no-arena-buckets", action="store_true")
    ap.add_argument("--optimizer-in-backward", action="store_true",
                    help="apply the optimizer per DDP bucket right behind its allreduce (f-2; SGD / Adam / AdamW)")
    ap.add_argument("--cpu-batch", type=int, default=8)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss, parameters and gradients of the last step as DIR/*.npy "
                         "(convolutions then use deterministic cuDNN algorithms, so that runs can be compared)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_SAMPLE = 1 << 22   # elements kept of a longer flat array: 16 MiB of float32, so at most 32 MiB in all


def dump_outputs(out_dir, torch, model, loss):
    """Write what a caller of the training step holds after the last timed step, so that two builds can be compared
    output for output: the loss (float64) and every parameter and its synchronised gradient, concatenated flat in
    ``model.parameters()`` order (float32).  A flat array longer than DUMP_SAMPLE elements is cut down to the same
    seeded sample of positions in every run; gradients are written only when every parameter has one."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    params = list(model.parameters())
    flat = {"params": torch.cat([p.detach().float().reshape(-1) for p in params])}
    if all(p.grad is not None for p in params):
        flat["grads"] = torch.cat([p.grad.detach().float().reshape(-1) for p in params])
    n = flat["params"].numel()
    idx = None
    if n > DUMP_SAMPLE:
        idx = torch.randint(0, n, (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
    for name, t in flat.items():
        if idx is not None:
            t = t[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "loss.npy"), np.array([float(loss)], dtype=np.float64))


def free_port():
    with closing(socket.socket(socket.AF_INET, socket.SOCK_STREAM)) as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (profiling recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def usable_cores():
    """Host threads this process can really run: affinity mask, capped by the cgroup CPU quota, and by
    B2D_CPU_THREADS when set (oversubscribing a quota makes the CPU arm pathologically slow)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    cap = int(os.environ.get("B2D_CPU_THREADS", "64"))   # beyond ~64 threads torch's CPU conv backward stops scaling
    return max(1, min(n, cap))


# ---- the reference arm / cpu baseline: torch DDP over gloo on the host cores ---------------------
def cpu_reference(world, batch, steps, warmup, model="resnet50", budget_s=20.0):
    """What RayStrategy(num_workers=world, use_gpu=False) executes in its workers (oracle/reference_ddp.py)."""
    from oracle import reference_ddp
    cores = usable_cores()
    cfg = {"model": model, "batch": batch, "steps": steps, "warmup": warmup, "threads_total": cores,
           "time_budget_s": budget_s, "ddp_kwargs": {"find_unused_parameters": False, "gradient_as_bucket_view": True}}
    t0 = time.time()
    res = reference_ddp.run_training(world, cfg)
    ms = 1e3 * statistics.mean(res["times"])
    return {"value": world * batch / (ms / 1e3), "unit": "images/sec", "cores": cores, "kind": "reference",
            "steps_done": len(res["times"]),
            "sample": "torch DDP/gloo fp32 (the implementation ray_lightning's use_gpu=False path dispatches to; Ray actors "
                      "replaced by torch.multiprocessing), %s, %d worker(s) x batch %d, %d threads/worker, %d warm-up + %d "
                      "timed steps, %.0f s wall" % (model, world, batch, res["threads_per_rank"], warmup, len(res["times"]), time.time() - t0),
            "ms_per_step": ms}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # --steps / --warmup are honoured; each step is a bounded sample (per-worker batch --cpu-batch) and the
    # run stops early once ~150 s of wall clock are spent, reporting the steps actually timed
    steps, warm = max(1, args.steps), max(1, min(args.warmup, 3))
    try:
        cb = cpu_reference(args.gpus, args.cpu_batch, steps, warm, args.model, budget_s=150.0)
        steps = cb["steps_done"]
    except Exception as e:  # the oracle always exists; a failure here is a bug worth seeing
        print(json.dumps({"impl": "reference", "unavailable": "cpu reference failed: %r" % (e,)}))
        return
    line = {"impl": "reference", "metric": METRIC, "value": round(cb["value"], 2), "unit": "images/sec",
            "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": round(cb["ms_per_step"], 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": "%s synthetic 224x224, RayStrategy(num_workers=%d, use_gpu=False) == torch DDP/gloo on host cores"
                                   % (args.model, args.gpus), "per_worker_batch": args.cpu_batch,
                       "global_batch": args.cpu_batch * args.gpus, "parallelism": "dp%d" % args.gpus,
                       "bounded_sample": "%d timed steps" % steps},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": round(cb["value"], 2), "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---- multi-GPU evidence that rides along with the bench line (outside every timed region) -----------------
def link_probe(comm, dist, torch, world, rank):
    """What ONE GPU pulls from ONE peer, measured here and now: cudaMemcpyAsync and a peer-read kernel with the
    library's own 16-byte access pattern, every rank pulling from its right neighbour at the same time."""
    out = {"nominal_GBps": NVLINK_NOMINAL_GBS}
    try:
        peer = (rank + 1) % world
        vals = []
        for mode in (0, 1):
            dist.barrier()
            v = comm.ctx.peer_bw(peer, 128 << 20, iters=8, mode=mode)
            t = torch.tensor([v], device="cuda")
            lo = t.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            vals.append((float(lo), float(t) / world))
        out.update({"memcpy_peer_GBps_min": round(vals[0][0], 1), "memcpy_peer_GBps_mean": round(vals[0][1], 1),
                    "peer_read_kernel_GBps_min": round(vals[1][0], 1), "peer_read_kernel_GBps_mean": round(vals[1][1], 1),
                    "how": "128 MiB x 8 from the right neighbour's arena, all ranks at once, CUDA events (b2d_peer_bw)"})
        out["peak_GBps"] = round(max(vals[0][1], vals[1][1]), 1)
        out["source"] = "measured in this run"
    except Exception as e:
        out.update({"peak_GBps": NVLINK_FALLBACK_GBS, "source": "fallback (B200_PROFILING.md peer copy); probe failed: %r" % (e,)})
    return out


def parity_block(comm, dist, torch, world, rank, dev, bucket_sizes):
    """Every algorithm the library exports, on seeded buckets of the step's own sizes + ragged ones, against the
    oracle (bit for bit for the P2P algorithms, stated tolerance for NVLS) and against NCCL on the same inputs."""
    import numpy as np
    from oracle import ddp_oracle        # the checker, never the thing measured
    sizes = sorted(set(list(bucket_sizes) + [1, 4099, (1 << 20) + 5]))
    algos = ["one_shot", "two_shot", "two_shot_tma", "staged"] + (["nvls", "nvls_fused"] if comm.nvls else [])
    scale = float(np.float32(1.0) / np.float32(world))
    failed, cases = [], 0
    key = 20000
    worst = {"fp32_vs_nccl_max_abs": 0.0, "bf16_err_vs_exact_libb2d": 0.0, "bf16_err_vs_exact_nccl": 0.0,
             "bf16_err_vs_exact_nvls": 0.0, "nvls_bf16_ulps_max": 0.0}

    def bits_equal(a, b):
        return torch.equal(a.view(torch.int32), b.view(torch.int32))

    for n in sizes:
        per_rank = [torch.randn(n, generator=torch.Generator().manual_seed(4242 + 131 * r + n % 1009)) * 2.0 ** -4 for r in range(world)]
        mine = per_rank[rank].to(dev)
        want = {"bf16": ddp_oracle.allreduce_bf16_wire(per_rank), "fp32": ddp_oracle.allreduce_fp32_wire(per_rank)}
        exact_bf = sum(ddp_oracle.wire_bf16(t, scale).double() for t in per_rank)
        # the reference's GPU path on the same inputs
        nccl_fp32 = mine / world
        dist.all_reduce(nccl_fp32)
        c = mine.to(torch.bfloat16).div_(world)
        dist.all_reduce(c)
        nccl_bf16 = c.float()
        torch.cuda.synchronize()
        worst["bf16_err_vs_exact_nccl"] = max(worst["bf16_err_vs_exact_nccl"], float((nccl_bf16.cpu().double() - exact_bf).abs().max()))
        for wire in ("bf16", "fp32"):
            for algo in algos:
                if algo == "two_shot_tma" and (wire != "bf16" or n % 8):
                    continue
                if algo == "one_shot" and n > (4 << 20):
                    continue
                cases += 1
                buf = mine.clone()
                # one arena slot per (size, wire): a change of algorithm re-fences and re-uses the region
                comm.allreduce_(buf, bucket_idx=key + 2 * sizes.index(n) + (wire == "bf16"), wire=wire, algo=algo)
                torch.cuda.synchronize()
                got = buf.cpu()
                tag = "%s/%s/n=%d" % (algo, wire, n)
                if algo.startswith("nvls"):
                    # every rank must hold the same bits; value within the stated tolerance
                    h = torch.tensor([int(got.view(torch.int32).long().sum().item()) & 0x7fffffffffff], device=dev)
                    lo, hi = h.clone(), h.clone()
                    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
                    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
                    ok = int(lo) == int(hi)
                    if wire == "fp32":
                        ok = ok and torch.allclose(got, want["fp32"], rtol=1e-5, atol=1e-8)
                    else:
                        d = (got.double() - exact_bf).abs()
                        ulp = torch.maximum(got.double().abs(), exact_bf.abs()) * 2.0 ** -7
                        ok = ok and bool((d <= ulp + 1e-30).all())
                        worst["nvls_bf16_ulps_max"] = max(worst["nvls_bf16_ulps_max"], float((d / (ulp + 1e-30)).max()))
                else:
                    ok = bits_equal(got, want[wire])
                if wire == "fp32":
                    ok = ok and torch.allclose(got, nccl_fp32.cpu(), rtol=1e-3, atol=1e-5)   # north-star tolerance vs the NCCL path
                    worst["fp32_vs_nccl_max_abs"] = max(worst["fp32_vs_nccl_max_abs"], float((got - nccl_fp32.cpu()).abs().max()))
                else:
                    e = float((got.double() - exact_bf).abs().max())
                    k = "bf16_err_vs_exact_nvls" if algo.startswith("nvls") else "bf16_err_vs_exact_libb2d"
                    worst[k] = max(worst[k], e)
                if not ok:
                    failed.append(tag)
    # one fused sharded step (reduce-scatter -> Adam -> all-gather) against the oracle's Adam on the averaged gradients
    try:
        total = 8 * 1024 * world
        shard_off = [i * 8 * 1024 for i in range(world + 1)]
        p0 = torch.randn(total, generator=torch.Generator().manual_seed(99)) * 0.05
        per_rank = [torch.randn(total, generator=torch.Generator().manual_seed(300 + r)) * 0.05 for r in range(world)]
        params = comm.arena_tensor(total)
        params.copy_(p0.to(dev))
        m, v = torch.zeros(8 * 1024, device=dev), torch.zeros(8 * 1024, device=dev)
        g = per_rank[rank].to(dev)
        torch.cuda.synchronize()
        dist.barrier()
        comm.sharded_step_(g, params, m, v, shard_off, step=1, lr=1e-2, wire="fp32", slot=7)
        torch.cuda.synchronize()
        avg = ddp_oracle.allreduce_fp32_wire(per_rank, scale)
        pn, mn, vn = p0.numpy().copy(), np.zeros(total, np.float32), np.zeros(total, np.float32)
        ddp_oracle.adam_step(pn, avg.numpy(), mn, vn, 1, 1e-2)
        cases += 1
        if not np.allclose(params.cpu().numpy(), pn, rtol=2e-5, atol=2e-6):
            failed.append("sharded_step/fp32")
    except Exception as e:
        failed.append("sharded_step raised %r" % (e,))
    flag = torch.tensor([0 if failed else 1], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    gathered = [None] * world
    dist.all_gather_object(gathered, failed[:8])
    return {"all_ok": bool(int(flag) == 1), "cases_per_rank": cases, "algos": algos, "sizes": sizes, "nvls_bound": bool(comm.nvls),
            "failed": sorted(set(x for f in gathered for x in f))[:16],
            "contract": "P2P algorithms bit-exact vs oracle.ddp_oracle (both wires); NVLS: all ranks same bits, fp32 rtol 1e-5, "
                        "bf16 within one bf16 step of the exact sum; fp32 wire vs ncclAllReduce rtol 1e-3 / atol 1e-5",
            **{k: float("%.3g" % v) for k, v in worst.items()},
            "bf16_libb2d_not_worse_than_nccl": worst["bf16_err_vs_exact_libb2d"] <= worst["bf16_err_vs_exact_nccl"] + 1e-12,
            "note": "bf16_err_vs_exact_libb2d covers the rank-ordered P2P algorithms (one rounding of an fp32 sum); the in-switch "
                    "reduction is reported separately (bf16_err_vs_exact_nvls, nvls_bf16_ulps_max)"}


def allreduce_sweep(comm, dist, torch, world, rank, sizes, iters=20, symm=True):
    """Isolated allreduce of `sizes` (bytes of bf16 wire payload) back to back on one stream: libb2d (whole fused op:
    cast + scale + exchange + write-back) next to ncclAllReduce alone, the reference's bf16 hook sequence, and
    torch.ops.symm_mem.* on a symmetric bf16 buffer.  ms = max over ranks of the per-iteration average."""
    rows = []

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        b.synchronize()
        t = torch.tensor([a.elapsed_time(b) / iters], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    sm_state = {}
    if symm:
        try:
            import torch.distributed._symmetric_memory as symm_mem
            gname = dist.group.WORLD.group_name
            try:
                symm_mem.enable_symm_mem_for_group(gname)
            except Exception:
                pass
            sm_state = {"mod": symm_mem, "group": gname}
        except Exception as e:
            sm_state = {"error": repr(e)}
    key = 30000
    for wire_bytes in sizes:
        n = wire_bytes // 2
        buf = torch.randn(n, device="cuda") * 0.01
        row = {"wire_bytes": wire_bytes, "elements": n}
        algos = ["auto", "auto_latency", "one_shot", "two_shot", "staged"] + (["nvls", "nvls_fused"] if comm.nvls else [])
        for algo in algos:
            if algo == "one_shot" and wire_bytes > (16 << 20):
                continue
            k = key + sizes.index(wire_bytes)
            try:
                comm.ctx.set_auto_profile(1 if algo == "auto_latency" else 0)
                a = "auto" if algo == "auto_latency" else algo
                row["b2d_" + algo + "_ms"] = round(timed(lambda: comm.allreduce_(buf, bucket_idx=k, wire="bf16", algo=a)), 4)
                if algo.startswith("auto"):
                    row[algo + "_algo"] = comm.ctx.plan(n, 1)[0]
            except Exception as e:
                row["b2d_" + algo + "_error"] = repr(e)[:120]
            finally:
                comm.ctx.set_auto_profile(0)

        def hook_seq():
            c = buf.to(torch.bfloat16).div_(world)
            dist.all_reduce(c)
            buf.copy_(c)
        row["nccl_bf16_hook_seq_ms"] = round(timed(hook_seq), 4)
        cb = buf.to(torch.bfloat16)
        row["nccl_bf16_allreduce_only_ms"] = round(timed(lambda: dist.all_reduce(cb)), 4)
        if "mod" in sm_state:
            try:
                t = sm_state["mod"].empty(n, dtype=torch.bfloat16, device="cuda")
                sm_state["mod"].rendezvous(t, sm_state["group"])
                t.copy_(cb)
                for name, op in (("one_shot", "one_shot_all_reduce"), ("two_shot", "two_shot_all_reduce_"), ("multimem", "multimem_all_reduce_")):
                    if name == "one_shot" and wire_bytes > (16 << 20):
                        continue
                    try:
                        f = getattr(torch.ops.symm_mem, op)
                        row["symm_mem_%s_ms" % name] = round(timed(lambda: f(t, "sum", sm_state["group"])), 4)
                    except Exception as e:
                        row["symm_mem_%s_error" % name] = repr(e)[:120]
            except Exception as e:
                row["symm_mem_error"] = repr(e)[:160]
        elif "error" in sm_state:
            row["symm_mem_error"] = sm_state["error"][:160]
        bus = 2.0 * (world - 1) / world * wire_bytes
        for k2 in [k for k in row if k.endswith("_ms")]:
            row[k2[:-3] + "_busGBps"] = round(bus / row[k2] / 1e6, 1)
        rows.append(row)
        del buf, cb
    return rows


# ---- our arm -----------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F

    from ray_lightning_b200 import RayStrategy
    from ray_lightning_b200._compat import LightningModule

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 gradient-sync path has no CPU fallback "
                         "(use --impl reference for the CPU/gloo arm)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d: launch with torchrun --nproc-per-node %d" % (args.gpus, world, args.gpus))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", str(free_port()))
    os.environ.setdefault("PL_TORCH_DISTRIBUTED_BACKEND", "nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # cuDNN's autotuner picks convolution algorithms by timing them in each run, and some of them accumulate with
    # atomics, so the same inputs give different outputs from run to run.  Outputs written for comparison come from
    # deterministic algorithms instead; at the default ResNet-50 workload they are no slower (17.36 ms/step against
    # 17.46 autotuned, one B200 at a 1000 W power limit, mean of two runs each).
    torch.backends.cudnn.benchmark = not args.dump_outputs
    torch.backends.cudnn.deterministic = bool(args.dump_outputs)

    import torchvision
    torch.manual_seed(0)
    if args.model.startswith("resnet"):
        B = args.batch or 64
        unit = "images"

        class Net(LightningModule):
            def __init__(self):
                super().__init__()
                self.net = getattr(torchvision.models, args.model)()

            def training_step(self, batch, batch_idx):
                x, y = batch
                return F.cross_entropy(self.net(x), y)

            def configure_optimizers(self):
                return torch.optim.SGD(self.parameters(), lr=0.05, momentum=0.9)

        def host_batch(g):
            return (torch.randn(B, 3, 224, 224, generator=g).contiguous(memory_format=torch.channels_last),
                    torch.randint(0, 1000, (B,), generator=g))
    else:
        import transformers
        unit = "sequences"
        if args.model == "bert-base":      # BASELINE.json configs[2]
            B, S = args.batch or 16, args.seq or 512
            cfg = transformers.BertConfig()
            make = lambda: transformers.BertForMaskedLM(cfg)
        else:                               # gpt2-medium, BASELINE.json configs[3]
            B, S = args.batch or 4, args.seq or 1024
            cfg = transformers.GPT2Config(n_embd=1024, n_layer=24, n_head=16)
            make = lambda: transformers.GPT2LMHeadModel(cfg)
        vocab = cfg.vocab_size

        class Net(LightningModule):
            def __init__(self):
                super().__init__()
                self.net = make()

            def training_step(self, batch, batch_idx):
                ids, = batch
                return self.net(input_ids=ids, labels=ids).loss

            def configure_optimizers(self):
                return (torch.optim.Adam if args.strategy == "sharded" else torch.optim.AdamW)(self.parameters(), lr=1e-4)

        def host_batch(g):
            return (torch.randint(0, vocab, (B, S), generator=g),)

    # the worker-side call sequence of RayLauncher._wrapping_function (launchers/ray_launcher.py)
    from ray_lightning_b200 import RayShardedStrategy
    kw = dict(num_workers=world, use_gpu=True, b200_wire=args.wire, b200_algo=args.algo, b200_mem=args.mem,
              b200_timing=True, b200_max_ctas=args.max_ctas, b200_exch_ctas=args.exch_ctas,
              b200_chunk_bytes=(args.chunk_mb << 20) if args.chunk_mb else None,
              b200_arena_buckets=not args.no_arena_buckets, b200_optimizer_in_backward=args.optimizer_in_backward,
              # the product sizes its arena for the model alone; the evidence blocks of this file (isolated buckets,
              # parity cases, sweep up to 64 MiB of wire) stage extra buffers
              b200_arena_extra_bytes=(1 << 30) if world > 1 else 0)
    if args.strategy == "sharded":
        strategy = RayShardedStrategy(**kw)
    else:
        kw.update(find_unused_parameters=False, gradient_as_bucket_view=True, bucket_cap_mb=args.bucket_cap_mb)
        if args.hook != "b200":
            kw["b200_enable"] = False
            if args.hook == "nccl_bf16":
                from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
                kw["ddp_comm_hook"] = default_hooks.bf16_compress_hook
        strategy = RayStrategy(**kw)
    strategy.precision = "bf16"
    strategy.set_remote(True)
    strategy.set_global_to_local([(i, 0) for i in range(world)])
    strategy.root_device = dev
    strategy._worker_setup(process_idx=rank)
    model = Net()
    if args.model.startswith("resnet"):
        model = model.to(memory_format=torch.channels_last)
    strategy.connect(model)
    strategy.model_to_device()
    strategy.configure_ddp()

    class _T:  # the two Trainer attributes setup_optimizers looks at
        pass
    strategy.setup_optimizers(_T())
    opt = strategy.optimizers[0]
    n_params = sum(p.numel() for p in model.parameters())

    g = torch.Generator().manual_seed(1000 + rank)
    host = tuple(t.pin_memory() for t in host_batch(g))
    devb = tuple(t.to(dev, non_blocking=True) for t in host)

    def step(batch, i):
        opt.zero_grad(set_to_none=True) if args.strategy == "ddp" else opt.zero_grad()
        loss = strategy.training_step(batch, i)
        strategy.backward(loss)
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n, e2e):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        last = None
        for i in range(n):
            if e2e:
                batch = tuple(t.to(dev, non_blocking=True) for t in host)
                last = float(step(batch, i))  # device->host read of the step's result, every step
            else:
                last = step(devb, i)
        b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t), last

    for i in range(args.warmup):
        step(devb, i)
    barrier()
    state = strategy.b200_state if args.strategy == "ddp" else None
    comm = state.comm if state is not None else getattr(strategy, "_comm", None)
    if comm is not None:
        comm.ctx.reset_stats()
    vis = os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")
    phys = int(vis[local]) if len(vis) > local and vis[local].isdigit() else local
    sampler = ClockSampler(phys)
    if rank == 0:
        sampler.start()
    total_ms, _ = timed(args.steps, e2e=False)
    clocks = sampler.stop() if rank == 0 else None
    torch.cuda.synchronize()
    st = comm.stats() if comm is not None else {"launches": 0, "timed_ms": 0.0, "timed_launches": 0}
    launches_timed, kernel_ms = int(st["launches"]), float(st["timed_ms"])
    timed_launches = int(st["timed_launches"])
    # the staged exchange times its NVLink kernel (the only one that can wait for a peer) on its own stream
    exch_ms, exch_timed, exch_launches = float(st.get("exch_ms", 0.0)), int(st.get("exch_timed", 0)), int(st.get("exch_launches", 0))
    last_algo = int(st.get("last_algo", 0))
    e2e_ms, last_loss = timed(args.steps, e2e=True)
    if args.dump_outputs and rank == 0:
        # right after the last timed step: the isolated runs below push random data through the same bucket slots
        dump_outputs(args.dump_outputs, torch, model, last_loss)

    # The same buckets once more, ISOLATED (no backward running, ranks aligned by a barrier): what the
    # kernel does when it is not waiting for SMs or for a slower peer.  Through the same hook entry point.
    isolated = None
    if state is not None and comm is not None and getattr(state, "seen", None):
        isolated = []
        for idx, n in sorted(state.seen.items()):
            buf = torch.randn(n, device=dev) * 0.01
            barrier()
            for _ in range(3):
                comm.allreduce_(buf, bucket_idx=idx, wire=args.wire, algo=args.algo, wait_stream=state.stream,
                                comm_stream=state.stream)
            barrier()
            it = 20
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(state.stream):
                a.record()
                for _ in range(it):
                    comm.allreduce_(buf, bucket_idx=idx, wire=args.wire, algo=args.algo, wait_stream=state.stream,
                                    comm_stream=state.stream)
                b.record()
            b.synchronize()
            t = torch.tensor([a.elapsed_time(b) / it], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            isolated.append((idx, n, float(t)))
        barrier()

    kernel_ms0, timed_launches0 = kernel_ms, timed_launches

    def emit(link, parity, sweep, with_cpu):
        """Rank 0: build and print THE json line (called once: normally after the evidence blocks, or by the
        watchdog below if those hang)."""
        kernel_ms, timed_launches = kernel_ms0, timed_launches0
        peaks, peak_src = measured_peaks()
        ms_per_step = total_ms / args.steps
        value = world * B / (ms_per_step / 1e3)
        e2e_value = world * B / (e2e_ms / args.steps / 1e3)
        wire_w = 2 if args.wire == "bf16" else 4
        per_launch_ms = kernel_ms / max(timed_launches, 1)
        buckets_per_step = launches_timed / args.steps
        if world == 1:
            # K0: 4 B read + 4 B write per gradient element, nothing else (DESIGN.md §4)
            alg_bytes_step = 8.0 * n_params
            if args.strategy == "sharded":   # stage (4 r + w w), reduce (w r), Adam p/m/v r+w + p (28), DESIGN.md §4
                alg_bytes_step = (4.0 + 2 * wire_w + 28.0) * n_params
            bound, peak, runit = "hbm", float(peaks["hbm_gbs"]), "GB/s"
            peak_note = "MEASURED_PEAKS.json hbm_gbs (%s)" % peak_src
        else:
            alg_bytes_step = 2.0 * (world - 1) / world * n_params * wire_w   # NCCL-tests bus-bandwidth convention
            if args.strategy == "sharded":   # reduce-scatter at wire width + fp32 parameter all-gather
                alg_bytes_step = (world - 1) / world * n_params * (wire_w + 4.0)
            bound, runit = "nvlink", "GB/s"
            peak = float(link["peak_GBps"]) if link else NVLINK_FALLBACK_GBS
            peak_note = "peer link probe, %s (nominal %.0f GB/s per direction)" % (link["source"] if link else "fallback", NVLINK_NOMINAL_GBS)
            if args.strategy == "sharded" and exch_timed > 0:
                # reduce-to-owner kernels (one per bucket, during backward) + the Adam-and-push kernel of the step
                kernel_ms, timed_launches = kernel_ms + exch_ms, timed_launches + exch_timed
                per_launch_ms = kernel_ms / max(timed_launches, 1)
                buckets_per_step = timed_launches / args.steps
            elif exch_timed > 0:
                # staged exchange: the dominant kernel is the exchange kernel, timed per bucket on its own stream
                kernel_ms, timed_launches = exch_ms, exch_timed
                per_launch_ms = kernel_ms / max(timed_launches, 1)
                buckets_per_step = exch_timed / args.steps
        achieved = alg_bytes_step * args.steps / (kernel_ms / 1e3) / 1e9 if kernel_ms > 0 else None
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
            if world == 1 and "k0_dram_bytes_per_element" in tj:
                traffic = tj["k0_dram_bytes_per_element"] * n_params / max(buckets_per_step, 1)
        except Exception:
            pass
        line = {
            "metric": METRIC if unit == "images" else "%s/sec, %s %s" % (unit, args.model, "RayShardedStrategy" if args.strategy == "sharded" else "RayStrategy"),
            "value": round(value, 2), "unit": unit + "/sec", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if args.wire == "bf16" else "fp32", "data": "synthetic",
            "config": {"workload": "%s synthetic %s %s(num_workers=%d, use_gpu=True) bf16-autocast, gradient sync = %s"
                                   % (args.model, "224x224" if unit == "images" else "token ids",
                                      "RayShardedStrategy" if args.strategy == "sharded" else "RayStrategy", world,
                                      ("libb2d (%s wire)" % args.wire) if args.hook == "b200" else args.hook),
                       "global_batch": B * world, "per_gpu_batch": B, "parallelism": "dp%d" % world,
                       "bucket_cap_mb": args.bucket_cap_mb, "grad_elements": n_params,
                       "l2_policy": "inputs larger than L2 (activations + 97.5 MiB of gradients per step >> 126 MB)",
                       "algo": args.algo, "algo_used": last_algo, "mem": args.mem, "nvls_bound": bool(getattr(comm, "nvls", False)),
                       "arena_buckets": bool(getattr(strategy, "b200_arena_buckets_active", False)),
                       "optimizer_in_backward": bool(args.optimizer_in_backward),
                       "strategy": args.strategy, "hook": args.hook},
            "e2e": {"value": round(e2e_value, 2), "unit": unit + "/sec", "ms_per_step": round(e2e_ms / args.steps, 3),
                    "h2d_bytes_per_step": int(sum(t.numel() * t.element_size() for t in host)) * world,
                    "d2h_bytes_per_step": 4 * world,
                    "api": "RayStrategy worker path: training_step/backward/optimizer.step with pinned-host batches, loss read back"},
            "gpu_launches": launches_timed,
            "roofline": {"bound": bound, "achieved": round(achieved, 1) if achieved else None, "peak": peak, "unit": runit,
                         "frac": round(achieved / peak, 4) if achieved else None, "traffic": traffic,
                         "kernel": ("seg_reduce_kernel (per bucket, in backward) + adam_push_kernel (step)" if args.strategy == "sharded" else
                                    "k0_cast_scale_kernel<bf16>" if world == 1 else
                                    {3: "exch_kernel<NVLS> (staged exchange, multimem.ld_reduce + multimem.st)",
                                     5: "exch_kernel<P2P> (staged exchange, peer loads + peer stores)"}.get(last_algo, "k1/k2 fused allreduce"))
                                   if args.hook == "b200" else None,
                         "algorithmic_bytes_per_step": alg_bytes_step, "launches_per_step": buckets_per_step,
                         "avg_launch_ms": round(per_launch_ms, 5), "kernel_share_of_step": round(kernel_ms / total_ms, 5),
                         "peak_source": peak_note,
                         "frac_of_nominal_900": (round(achieved / NVLINK_NOMINAL_GBS, 4) if achieved and world > 1 else None),
                         "link_level": (None if world == 1 or not achieved or last_algo != 3 else {
                             "note": "in-switch reduction: bytes that really cross one GPU's links per direction = (1 + 1/W) x N x w",
                             "GBps": round(achieved * (1.0 + 1.0 / world) / (2.0 * (world - 1) / world), 1),
                             "frac": round(achieved * (1.0 + 1.0 / world) / (2.0 * (world - 1) / world) / peak, 4)}),
                         "note": "launch durations from CUDA events on the launching stream inside the timed region (overlapped with backward); "
                                 "achieved = NCCL-tests bus bytes 2(W-1)/W x N x w per step / summed exchange-kernel time"},
            "clocks": clocks, "final_loss": last_loss if isinstance(last_loss, float) else float(last_loss),
            "allreduce_isolated": None if not isolated else {
                "note": "same bucket sizes, back to back on the comm stream with no backward running (L2-warm), max over ranks",
                "buckets": [{"index": i, "elements": n, "ms": round(ms, 5),
                             "GBps": round((8.0 * n if world == 1 else 2.0 * (world - 1) / world * n * (2 if args.wire == "bf16" else 4)) / ms / 1e6, 1)}
                            for i, n, ms in isolated],
                "GBps_total": round(sum((8.0 * n if world == 1 else 2.0 * (world - 1) / world * n * (2 if args.wire == "bf16" else 4))
                                        for _, n, _ in isolated) / sum(ms for _, _, ms in isolated) / 1e6, 1),
                "unit": "HBM GB/s (8 B/element)" if world == 1 else "NVLink bus GB/s (2(W-1)/W x wire bytes)"},
        }
        line["nvlink"] = link
        line["parity"] = parity
        line["allreduce_sweep"] = sweep
        if with_cpu and not args.no_cpu_baseline and args.model.startswith("resnet"):
            try:
                cb = cpu_reference(1, args.cpu_batch, 2, 1, args.model)
                line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
            except Exception as e:
                line["cpu_baseline"] = {"value": None, "unit": "images/sec", "cores": None, "kind": "reference",
                                        "sample": "failed: %r" % (e,)}
        print(json.dumps(line), flush=True)

    # Everything below is evidence AROUND the measurement (link probe, parity block, sweep, CPU baseline).  It contains
    # collectives; should one of them ever hang, a watchdog still prints the bench line (without that evidence) and ends
    # the process cleanly instead of leaving the driver without a number.
    def _watchdog():      # a thread: the main thread may be blocked inside a CUDA / NCCL call, where no signal handler runs
        if rank == 0:
            emit(None, {"all_ok": False, "error": "evidence blocks timed out after %d s" % EVIDENCE_TIMEOUT_S}, None, False)
        os._exit(0)

    guard = None
    if world > 1:
        guard = threading.Timer(EVIDENCE_TIMEOUT_S, _watchdog)
        guard.daemon = True
        guard.start()
    link = parity = sweep = None
    if world > 1 and comm is not None and args.hook == "b200":
        link = link_probe(comm, dist, torch, world, rank)
        if not args.no_parity:
            try:
                parity = parity_block(comm, dist, torch, world, rank, dev,
                                      sorted(state.seen.values()) if state is not None and state.seen else [])
            except Exception as e:
                parity = {"all_ok": False, "error": repr(e)[:300]}
        if not args.no_sweep:
            try:
                sweep = allreduce_sweep(comm, dist, torch, world, rank, [64 << 10, 1 << 20, 16 << 20, 64 << 20])
            except Exception as e:
                sweep = [{"error": repr(e)[:300]}]
        barrier()

    if rank == 0:
        emit(link, parity, sweep, True)
    if guard is not None:
        guard.cancel()
    barrier()
    strategy.teardown_worker()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
