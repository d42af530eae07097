#!/usr/bin/env python
"""Benchmark of the LightGlue matcher forward path on B200 (contract: see the task brief).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload at N GPUs: BASELINE.json configs[1] on every GPU -- SuperPoint-shaped synthetic pairs,
2048 keypoints, d=256, 9 layers, pruning / early exit OFF, batch = 32 pairs per step per GPU (weak
scaling: pairs are independent, each rank matches its own shard; the only collective is the final
all_gather of the match indices and scores, SURVEY.md §8e).  One "step" = one forward over one batch.

Prints ONE JSON line (rank 0).  `value` = pairs/s with inputs resident in HBM; `e2e` = pairs/s
through the public `LightGlue.forward` API with pinned HOST inputs (H2D and the D2H of the results
inside the timed region).  `roofline` = the attention kernel (dominant) against the measured bf16
peak; `cpu_baseline` = the CPU oracle (a port of the reference algorithm) on this host's cores.
`--impl reference` times that CPU implementation alone, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

N_KPTS, DESC, LAYERS, BATCH = 2048, 256, 9, 32
WORKLOAD = "superpoint_n2048_l9_prune_off_b32"
METRIC = "image pairs/sec at N=2048 kpts, 9 layers"


def algorithmic_flops_per_pair(n=N_KPTS, m=N_KPTS):
    """SURVEY.md §8d: conservative count (cross-attention similarity shared between directions)."""
    lin = 2 * 1_245_184 * (m + n)
    self_attn = 4 * 256 * (m * m + n * n)
    cross = (2 + 4) * 256 * m * n
    return 9 * (lin + self_attn + cross) + 2 * 256 * 256 * (m + n) + 2 * 256 * m * n


def attention_flops_per_launch(batch, n=N_KPTS):
    """Standard flash-attention convention, 4*Nq*Nk*dh per head: one launch covers 2*batch sequences."""
    return 4.0 * n * n * 64 * 4 * (2 * batch)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def profiled_traffic(kernel: str, batch: int, precision: str):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/traffic.json), or None
    when this run's workload is not the one that was profiled."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as f:
        d = json.load(f)
    if d.get("workload") != f"superpoint_n{N_KPTS}_l9_prune_off_b{batch}":
        return None
    return ((d.get(precision) or {}).get(kernel) or {}).get("bytes_per_launch")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
                for name, val in zip(names, f[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(res: dict, out_dir: str, cap_bytes: int = 64 << 20) -> None:
    """Write the output dict of one forward as `out_dir/<name>.npy`: floating outputs as float32, integer outputs (match
    indices, exit layers) as float64, which holds them exactly.  A per-pair list (`matches`, `scores`, `stops`) is written
    concatenated, its tensors' lengths as `<name>_lengths.npy`.  Above `cap_bytes` in all, only a fixed seeded sample of
    the pairs is written, their indices as `pairs.npy`."""
    b = res["matches0"].shape[0]

    def arrays(sel):
        out = {}
        for k, v in res.items():
            if isinstance(v, list) and len(v) == b:
                parts = [v[i] for i in sel]
                if parts and torch.is_tensor(parts[0]):
                    out[k] = torch.cat([p.cpu() for p in parts])
                    out[k + "_lengths"] = torch.tensor([len(p) for p in parts])
                else:
                    out[k] = torch.tensor(parts)
            elif torch.is_tensor(v) and v.dim() > 0 and v.shape[0] == b:
                out[k] = v[sel].cpu()
            else:
                out[k] = torch.as_tensor(v)
        return {k: t.to(torch.float32 if t.is_floating_point() else torch.float64).numpy() for k, t in out.items()}

    sel = list(range(b))
    arr = arrays(sel)
    if sum(a.nbytes for a in arr.values()) > cap_bytes:
        order = torch.randperm(b, generator=torch.Generator().manual_seed(0)).tolist()
        k = b
        while k > 1 and sum(a.nbytes for a in arr.values()) > cap_bytes:
            k = max(1, k * 3 // 4)
            sel = sorted(order[:k])
            arr = arrays(sel)
        arr["pairs"] = torch.tensor(sel, dtype=torch.float64).numpy()
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arr.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def host_cores() -> int:
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return n


class CpuReference:
    """The reference's own CPU path on pairs of the N=2048 workload.

    kind "reference": the UNMODIFIED reference file (oracle/_ref/lightglue_ref.py, copied from
    /root/reference/lightglue/lightglue.py by oracle/Makefile in the build container; it travels with the snapshot)
    -- SDPA-cpu for self-attention (lightglue.py:127-130), the shared-`sim` einsum path for cross-attention
    (216-225), fp32, pruning / early exit off (benchmark.py:117-120).  kind "port": the oracle restatement, only if
    that copy is absent."""

    def __init__(self):
        from lightglue_b200 import synth
        from oracle import ref_loader

        self.sd = synth.make_state_dict()
        self.data, _ = synth.make_pair(N_KPTS, d=DESC, b=1, seed=1000)
        self.small, _ = synth.make_pair(512, d=DESC, b=1, seed=1000)
        if ref_loader.available():
            self.kind = "reference"
            self.model = ref_loader.build_matcher(self.sd, "cpu", depth_confidence=-1, width_confidence=-1)
            self.fwd = lambda d: self.model(d)
        else:
            from oracle import lightglue_oracle as oracle

            self.kind = "port"
            self.fwd = lambda d: oracle.forward(self.sd, d)
        self.threads = self.pick_threads()

    def pick_threads(self) -> int:
        """torch's CPU path is not fastest at os.cpu_count() threads on a many-core host with a cgroup quota, and one
        N=2048 pair does not keep dozens of cores busy: time the N=512 forward of THIS model for a few (threads, pairs
        per forward) combinations and keep the best pairs/s (reported as `cores` / `pairs_per_forward`)."""
        ncpu = host_cores()
        cands = sorted({c for c in (4, 8, 16, 32, 64) if c <= ncpu} | {ncpu})
        best, best_rate, best_b = ncpu, 0.0, 1
        self.n512_ms = None
        with torch.no_grad():
            for bsz in (1, 4):
                d = self.small if bsz == 1 else {k: {kk: vv.expand(bsz, *vv.shape[1:]).contiguous() for kk, vv in v.items()}
                                               for k, v in self.small.items()}
                for c in cands:
                    if bsz > 1 and c < 16:
                        continue
                    torch.set_num_threads(c)
                    self.fwd(d)
                    t0 = time.perf_counter()
                    self.fwd(d)
                    dt = time.perf_counter() - t0
                    if bsz == 1 and (self.n512_ms is None or dt * 1e3 < self.n512_ms):
                        self.n512_ms = dt * 1e3
                    if bsz / dt > best_rate * 1.05:
                        best, best_rate, best_b = c, bsz / dt, bsz
        torch.set_num_threads(best)
        self.pairs_per_forward = best_b
        if best_b > 1:
            self.data = {k: {kk: vv.expand(best_b, *vv.shape[1:]).contiguous() for kk, vv in v.items()} for k, v in self.data.items()}
        return best

    def run(self, n_pairs: int, budget_s: float = 1e9):
        """Returns (pairs done, seconds); the output of the last forward is kept as `last`."""
        done, t0 = 0, time.perf_counter()
        with torch.no_grad():
            while done < n_pairs:
                self.last = self.fwd(self.data)
                done += self.pairs_per_forward
                if time.perf_counter() - t0 > budget_s:
                    break
        return done, time.perf_counter() - t0

    def describe(self, done, secs):
        return {"value": done / secs, "unit": "pairs/s", "cores": self.threads, "kind": self.kind,
                "host_cores": host_cores(), "n512_ms_per_pair": round(self.n512_ms, 1),
                "pairs_per_forward": self.pairs_per_forward,
                "sample": f"{done} pairs of the N=2048 workload, {self.pairs_per_forward} per forward ({secs:.1f} s), fp32, torch CPU, "
                          + ("unmodified reference lightglue.py" if self.kind == "reference" else "oracle port")}


def run_reference(args, rank: int):
    """--impl reference: the reference's own CPU implementation of the path (the unmodified reference file when
    oracle/_ref holds it, else the oracle port) on this host's cores.  One step = one forward of the calibrated number of
    N=2048 pairs (a bounded sample of the 32-pair batch); the timed steps are capped at ~100 s in total (`steps` = the steps
    actually run, `steps_requested` = K)."""
    if rank != 0:
        return
    cpu = CpuReference()
    for _ in range(min(args.warmup, 2)):
        cpu.run(1)
    t_all = time.perf_counter()
    done, secs, n_steps = 0, 0.0, 0
    for _ in range(args.steps):
        d, dt = cpu.run(1)
        done += d
        secs += dt
        n_steps += 1
        if time.perf_counter() - t_all > 100:
            break
    if args.dump_outputs:
        dump_outputs(cpu.last, args.dump_outputs)
    value = done / secs
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": n_steps, "steps_requested": args.steps, "pairs_per_step": done // max(n_steps, 1),
        "warmup": min(args.warmup, 2), "ms_per_step": 1000.0 * secs / max(n_steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": f"{cpu.pairs_per_forward} pair(s) of the N=2048 workload per step (one forward), "
                                                     "fp32, torch CPU"},
        "cpu_baseline": cpu.describe(done, secs),
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def reference_on_gpu(dev, resident, sd, batch, budget_s=60.0):
    """SURVEY 8d / BASELINE.md 4.5: the UNMODIFIED reference file on the SAME B200 -- the real bar.  benchmark.py:18-43
    protocol (warm-up, then CUDA events around each forward, mean), pruning / early exit off, at the bench batch and
    at B=1.  Variants: eager fp32 with fp16 flash SDPA (`flash=True`, lightglue.py:116-121), autocast (`mp=True`,
    480, 508-510), each SDPA backend torch offers.  `.compile()` pads to static lengths <= 1536 (439-454) and so does
    not apply to N=2048.  Returns a dict for the bench line, or {"unavailable": why}."""
    from oracle import ref_loader

    if not ref_loader.available():
        return {"unavailable": "oracle/_ref/lightglue_ref.py absent"}
    res = {"file": "oracle/_ref/lightglue_ref.py (unmodified lightglue/lightglue.py)", "protocol": "benchmark.py:18-43",
           "variants": {}}
    t_start = time.time()

    def timeit(model, data, b, warm=3, reps=10, ctx=None):
        import contextlib
        cm = ctx if ctx is not None else contextlib.nullcontext
        ts = []
        with torch.no_grad(), cm():
            for _ in range(warm):
                model(data)
            torch.cuda.synchronize(dev)
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out = model(data)
                e1.record()
                torch.cuda.synchronize(dev)
                ts.append(e0.elapsed_time(e1))
        mean = sum(ts) / len(ts)
        return {"ms_per_forward": mean, "std_ms": statistics.pstdev(ts), "pairs_per_s": b * 1000.0 / mean, "batch": b,
                "reps": reps}, out

    one = {k: {kk: vv[:1].contiguous() for kk, vv in v.items()} for k, v in resident.items()}
    variants = [("eager_flash_fp16sdpa", dict(flash=True, mp=False), None),
                ("eager_mp_autocast", dict(flash=True, mp=True), None),
                ("eager_fp32_sdpa", dict(flash=False, mp=False), None)]
    try:
        from torch.nn.attention import SDPBackend, sdpa_kernel
        for nm, be in (("flash", SDPBackend.FLASH_ATTENTION), ("efficient", SDPBackend.EFFICIENT_ATTENTION),
                       ("cudnn", SDPBackend.CUDNN_ATTENTION)):
            variants.append((f"eager_flash_sdpa_{nm}", dict(flash=True, mp=False), (lambda be=be: sdpa_kernel([be]))))
    except Exception:
        pass
    best = None
    ref_out = None
    for name, conf, ctx in variants:
        if time.time() - t_start > budget_s:
            res["variants"][name] = {"skipped": "time budget"}
            continue
        try:
            model = ref_loader.build_matcher(sd, dev, depth_confidence=-1, width_confidence=-1, **conf)
            rb, out = timeit(model, resident, batch, ctx=ctx)
            r1, _ = timeit(model, one, 1, reps=20, ctx=ctx)
            res["variants"][name] = {"batch": rb, "single": r1}
            if best is None or rb["pairs_per_s"] > best[1]:
                best = (name, rb["pairs_per_s"], r1["pairs_per_s"])
            if name == "eager_fp32_sdpa":
                ref_out = out
            del model
        except Exception as exc:  # noqa: BLE001
            res["variants"][name] = {"error": repr(exc)[:200]}
        torch.cuda.empty_cache()
    if best:
        res["best_variant"], res["pairs_per_s"], res["pairs_per_s_b1"] = best
    res["_fp32_out"] = ref_out
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="bf16x3", choices=["bf16", "bf16x3", "fp32"],
                    help="bf16x3 (default): split-bf16 tensor-core mode that reproduces the reference's match indices")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true")
    ap.add_argument("--no-other-mode", action="store_true")
    ap.add_argument("--no-extractor", action="store_true")
    ap.add_argument("--profile", action="store_true", help="2 forwards and exit (for ncu; prints nothing timed)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (rank 0's pairs; inputs are seeded)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    torch.set_grad_enabled(False)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    args.warmup = max(args.warmup, 3)

    from lightglue_b200 import LightGlue, synth
    from lightglue_b200.sharding import bind_to_gpu_numa_node

    # every rank runs next to its GPU: CPU affinity = the GPU's NUMA node, set BEFORE the pinned host buffers exist
    numa = bind_to_gpu_numa_node(local_rank)

    B = args.batch
    sd = synth.make_state_dict()
    matcher = LightGlue(features=None, depth_confidence=-1, width_confidence=-1, precision=args.precision)
    matcher.load_state_dict(sd, strict=False)
    matcher = matcher.eval().to(dev)

    # synthetic batch: B distinct seeded pairs (seeds differ per rank)
    base, _ = synth.make_pair(N_KPTS, d=DESC, b=B, seed=1000 + 16 * rank)
    host = {k: {kk: vv.contiguous().pin_memory() for kk, vv in v.items()} for k, v in base.items()}
    resident = {k: {kk: vv.to(dev) for kk, vv in v.items()} for k, v in host.items()}
    h2d_bytes = sum(vv.numel() * vv.element_size() for v in host.values() for vv in v.values())

    def step_resident():
        return matcher(resident)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    if args.profile:
        for _ in range(2):
            step_resident()
        torch.cuda.synchronize(dev)
        print(json.dumps({"profile": True, "launches_per_step": matcher.last_launch_count()}))
        return

    def run_resident(n_steps, in_flight):
        """n_steps forwards on resident inputs.  in_flight = 1: step i+1 is enqueued before step i's host-side result
        (stop, per-pair match lists) is resolved, so the GPU never waits for the host; in_flight = 0: every forward is
        resolved before the next is enqueued (the reference's calling pattern).  Either way every step's result is
        resolved before the function returns.  N > 1: the results of all steps are gathered once, after the last forward."""
        prev, last = None, None
        acc_i, acc_s = [], []
        for _ in range(n_steps):
            cur = matcher.forward_async(resident)
            if world > 1:
                # SURVEY 8e: the fixed-size results of every rank -- match indices of both images as int32 on the wire,
                # both score tensors -- are collected on the device and gathered ONCE for the run, after the last forward
                # (still inside the timed region).  A collective per step, concurrent with the next forward, cost 16 % at
                # two ranks: its channels hold SMs while they wait for the slower rank, and the persistent CTA-pair
                # kernels then run short of SMs.
                tt = cur.tensors
                acc_i.append(torch.cat([tt["matches0"], tt["matches1"]], 1).to(torch.int32))
                acc_s.append(torch.cat([tt["matching_scores0"], tt["matching_scores1"]], 1))
            if in_flight == 0:
                last = cur.result()
                continue
            if prev is not None:
                last = prev.result()
            prev = cur
        if world > 1:
            wi, ws = torch.stack(acc_i), torch.stack(acc_s)  # [steps, B, M + N]
            gi = torch.empty(world, *wi.shape, dtype=wi.dtype, device=dev)
            gs = torch.empty(world, *ws.shape, dtype=ws.dtype, device=dev)
            dist.all_gather_into_tensor(gi, wi)
            dist.all_gather_into_tensor(gs, ws)
        return prev.result() if prev is not None else last

    # warm-up: W steps in each host calling pattern (also absorbs their one-time allocations), timed to pick the
    # pattern the timed region will use; all ranks must agree, so the verdict of rank 0 is broadcast
    mode_ms = []
    for mode in (0, 1):
        run_resident(1, mode)
        torch.cuda.synchronize(dev)
        t0 = time.time()
        out = run_resident(args.warmup, mode)
        torch.cuda.synchronize(dev)
        mode_ms.append((time.time() - t0) * 1e3 / args.warmup)
    pick = torch.tensor([1 if mode_ms[1] <= mode_ms[0] else 0], device=dev)
    if world > 1:
        dist.broadcast(pick, src=0)
    in_flight = int(pick.item())
    launches_per_step = matcher.last_launch_count()

    # ---- timed region 1: inputs resident in HBM (inputs 134 MB + multi-GB workspace: larger than the 126 MB L2)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record()
    out = run_resident(args.steps, in_flight)
    e1.record()
    barrier()
    t_wall1 = time.time()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * B * args.steps / (ms / 1000.0)
    if rank == 0 and args.dump_outputs:
        dump_outputs(out, args.dump_outputs)

    # ---- timed region 2: end to end through the public API with pinned host inputs
    from lightglue_b200.pipeline import match_stream

    def run_e2e(n_steps):
        """n_steps batches from pinned host memory through the public streaming API (H2D on a copy stream one
        batch ahead, kernels, D2H of the match indices/scores into pinned host tensors)."""
        last = None
        for res in match_stream(matcher, (host for _ in range(n_steps)), dev):
            last = res
        return last

    run_e2e(4)  # warm-up: also allocates the three pinned result slots of match_stream
    barrier()
    e2s = args.steps
    e0.record()
    res = run_e2e(e2s)
    e1.record()
    barrier()
    d2h_bytes = sum(v.numel() * v.element_size() for k, v in res.items() if torch.is_tensor(v))
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * e2s / (float(t.item()) / 1000.0)

    # ---- per-kernel-class device times (separate pass: the event pairs perturb the pipeline slightly)
    roofline = None
    kernel_ms = {}
    if rank == 0:
        matcher.timing = True
        for _ in range(3):
            step_resident()
        torch.cuda.synchronize(dev)
        kt = matcher.kernel_times()
        kernel_ms = {k: {"ms_per_step": v[0] / 3.0, "launches_per_step": v[1] / 3.0} for k, v in kt.items()}
        peaks, how = measured_peaks()
        att_ms, att_n = kt["attention"]
        if att_n > 0 and args.precision != "fp32":
            ach = attention_flops_per_launch(B) / ((att_ms / att_n) / 1000.0) / 1e12
            peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
            roofline = {"kernel": "attention", "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                        "frac": ach / peak, "traffic": profiled_traffic("attention", B, args.precision),
                        "peak_source": how + ", sustained (kernel timed inside a long step)",
                        "flops_per_launch": attention_flops_per_launch(B), "avg_launch_ms": att_ms / att_n}

    # ---- assignment kernel, materialising variant (MatchAssignment.forward's declared output, lightglue.py:296):
    # the sweep that writes the [B, M+1, N+1] fp32 log-assignment matrix is HBM-bound (SURVEY.md §8d: 18.9 MB / pair)
    roofline_assign = None
    if rank == 0 and args.precision != "fp32":
        g = torch.Generator().manual_seed(3)
        xa = torch.randn(B, N_KPTS, 256, generator=g).to(dev)
        xb = torch.randn(B, N_KPTS, 256, generator=g).to(dev)
        for _ in range(2):
            matcher.log_assignment_matrix(8, xa, xb)
        matcher.timing = True
        for _ in range(3):
            matcher.log_assignment_matrix(8, xa, xb)
        torch.cuda.synchronize(dev)
        kt2 = matcher.kernel_times()
        am_ms, am_n = kt2.get("assign_matrix", (0.0, 0))
        st_ms, st_n = kt2.get("assign_stage", (0.0, 0))
        if am_n > 0 and st_n > 0:
            peaks, how = measured_peaks()
            abytes = 18.9e6 * B
            ach = abytes / ((st_ms / st_n) / 1000.0) / 1e9
            roofline_assign = {"kernel": "materialising assignment STAGE: final_proj + LSE sweep + arg-max sweep with the "
                                         "[B, M+1, N+1] fp32 matrix write + term + dustbin + tail (filter, outputs)",
                               "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                               "frac": ach / peaks["hbm_gbs"],
                               "traffic": profiled_traffic("assign_matrix", B, args.precision),
                               "algorithmic_bytes_per_launch": abytes, "avg_stage_ms": st_ms / st_n,
                               "matrix_writing_sweep_alone_ms": am_ms / am_n,
                               "matrix_writing_sweep_alone_frac": abytes / ((am_ms / am_n) / 1000.0) / 1e9 / peaks["hbm_gbs"],
                               "peak_source": how}
        del xa, xb

    # ---- the other tensor-core mode on the same resident batch, reported beside the headline (never fatal): with the
    # index-exact bf16x3 headline this is the plain-bf16 "fast" mode (operand rounding moves a few scores across
    # filter_threshold: its index differences from the headline are counted here)
    other_mode = None
    if rank == 0 and args.precision in ("bf16", "bf16x3") and not args.no_other_mode:
        oprec = "bf16" if args.precision == "bf16x3" else "bf16x3"
        try:
            m3 = LightGlue(features=None, depth_confidence=-1, width_confidence=-1, precision=oprec)
            m3.load_state_dict(sd, strict=False)
            m3 = m3.eval().to(dev)

            def run3(n):
                prev3 = None
                for _ in range(n):
                    cur3 = m3.forward_async(resident)
                    if prev3 is not None:
                        prev3.result()
                    prev3 = cur3
                return prev3.result()

            run3(3)
            torch.cuda.synchronize()
            steps3 = max(3, min(args.steps, 10))
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            o3 = run3(steps3)
            a1.record()
            torch.cuda.synchronize()
            ms3 = a0.elapsed_time(a1) / steps3
            flips = int((o3["matches0"] != out["matches0"]).sum()) + int((o3["matches1"] != out["matches1"]).sum())
            other_mode = {"precision": oprec, "value": B * 1000.0 / ms3, "unit": "pairs/s", "ms_per_step": ms3,
                          "steps": steps3, "n_gpus": 1,
                          "match_indices_differing_from_headline_mode": flips, "of_points": 2 * B * N_KPTS}
            del m3, o3
        except Exception as exc:  # noqa: BLE001
            other_mode = {"error": repr(exc)}

    # ---- next scope row (SURVEY 8f1): the SuperPoint extractor that produces the matcher's inputs, and extract + match
    # of one image pair (utils.match_pair, reference utils.py:150-165).  Random-init weights (no checkpoint offline), a
    # random 768 x 1024 image (the reference's default extraction size, resize = 1024), top-2048 keypoints.
    extractor = None
    if rank == 0 and not args.no_extractor:
        try:
            from lightglue_b200.superpoint import SuperPoint
            from lightglue_b200.utils import match_pair

            g = torch.Generator().manual_seed(11)
            im0 = torch.rand(1, 768, 1024, generator=g).to(dev)
            im1 = torch.roll(im0, shifts=(8, 16), dims=(1, 2))
            flops_img = 0.0
            hw = {0: 768 * 1024, 1: 768 * 1024, 2: 384 * 512, 3: 384 * 512, 4: 192 * 256, 5: 192 * 256}
            layers = [(64, 1, 3), (64, 64, 3), (64, 64, 3), (64, 64, 3), (128, 64, 3), (128, 128, 3), (128, 128, 3), (128, 128, 3),
                      (256, 128, 3), (65, 256, 1), (256, 128, 3), (256, 256, 1)]
            for li, (co, ci, k) in enumerate(layers):
                flops_img += 2.0 * co * ci * k * k * hw.get(li, 96 * 128)
            res = {"image": "768x1024 grayscale, synthetic", "max_num_keypoints": 2048, "algorithmic_flops_per_image": flops_img}
            peaks, how = measured_peaks()
            for prec in ("bf16x3", "fp32"):
                sp = SuperPoint(weights=None, max_num_keypoints=2048, precision=prec).eval().to(dev)
                for _ in range(2):
                    sp({"image": im0[None]})
                torch.cuda.synchronize()
                reps = 10 if prec == "bf16x3" else 3
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                for _ in range(reps):
                    sp({"image": im0[None]})
                a1.record()
                torch.cuda.synchronize()
                ms_img = a0.elapsed_time(a1) / reps
                res[prec] = {"ms_per_image": ms_img, "images_per_s": 1000.0 / ms_img,
                             "algorithmic_tflops": flops_img / (ms_img * 1e-3) / 1e12,
                             "frac_of_bf16_peak": flops_img / (ms_img * 1e-3) / 1e12 / peaks.get("bf16_tflops_sustained", 1400.0)}
                if prec == "bf16x3":
                    lg1 = LightGlue(features=None, depth_confidence=-1, width_confidence=-1, precision=args.precision)
                    lg1.load_state_dict(sd, strict=False)
                    lg1 = lg1.eval().to(dev)
                    for _ in range(2):
                        match_pair(sp, lg1, im0, im1, device=dev, resize=None)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(10):
                        f0, f1, m01 = match_pair(sp, lg1, im0, im1, device=dev, resize=None)
                    torch.cuda.synchronize()
                    ms_pair = (time.perf_counter() - t0) / 10 * 1e3
                    res["match_pair"] = {"ms_per_pair": ms_pair, "pairs_per_s": 1000.0 / ms_pair, "keypoints": int(f0["keypoints"].shape[0]),
                                         "what": "extract(image0) + extract(image1) + LightGlue forward, one pair at a time, host-synchronous "
                                                 "like the reference's utils.match_pair"}
                    del lg1
                del sp
            extractor = res
        except Exception as exc:  # noqa: BLE001
            extractor = {"error": repr(exc)[:300]}

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = CpuReference()
        cpu.run(1)
        done, dt = cpu.run(16, budget_s=12.0)
        cpu_baseline = cpu.describe(done, dt)

    # ---- the real bar (SURVEY 8d): the unmodified reference file on this same B200, same resident batch
    reference_gpu = None
    if rank == 0 and not args.no_reference_gpu:
        try:
            reference_gpu = reference_on_gpu(dev, resident, sd, B)
            ref_out = reference_gpu.pop("_fp32_out", None)
            if ref_out is not None:  # parity of the timed mode on the bench batch itself, against the reference's fp32 GPU run
                f0 = int((ref_out["matches0"] != out["matches0"]).sum()) + int((ref_out["matches1"] != out["matches1"]).sum())
                ds = float((ref_out["matching_scores0"] - out["matching_scores0"]).abs().max())
                reference_gpu["parity_of_timed_mode_vs_reference_fp32_on_this_batch"] = {
                    "match_index_flips": f0, "of_points": 2 * B * N_KPTS, "max_abs_dscore": ds}
            if reference_gpu.get("pairs_per_s"):
                reference_gpu["speedup_resident"] = value / world / reference_gpu["pairs_per_s"]
        except Exception as exc:  # noqa: BLE001
            reference_gpu = {"error": repr(exc)[:300]}

    if rank == 0:
        peaks, how = measured_peaks()
        flops = algorithmic_flops_per_pair()
        line = {
            "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"bf16": "bf16", "bf16x3": "bf16x3 (split-bf16 hi+lo operands, 3 tcgen05 MMAs per product: index-exact mode)",
                      "fp32": "f32"}[args.precision] +
                     " linears / fp16 attention operands / fp32 accumulate, softmax, LayerNorm, residual",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "pairs_per_step_per_gpu": B, "keypoints": N_KPTS, "descriptor_dim": DESC,
                       "layers": LAYERS, "precision": args.precision, "parallelism": f"pairs sharded over {world} GPU(s)", "numa_binding": numa,
                       "l2": "inputs (134 MB/step) + workspace (GBs) exceed the 126 MB L2; no explicit flush",
                       "host_pipelining": {"forwards_in_flight": in_flight, "warmup_ms_per_step_sync": mode_ms[0],
                                           "warmup_ms_per_step_one_in_flight": mode_ms[1],
                                           "note": "every step's stop / match lists are resolved inside the timed region"}},
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes},
            "gpu_launches": int(launches_per_step * args.steps),
            "clocks": clocks,
            "roofline": roofline,
            "roofline_assign": roofline_assign,
            "other_mode": other_mode,
            "extractor": extractor,
            "cpu_baseline": cpu_baseline,
            "reference_gpu": reference_gpu,
            "kernel_ms": kernel_ms,
            "whole_forward": {"algorithmic_flops_per_pair": flops,
                              "achieved_tflops": flops * value / world / 1e12,
                              "frac_of_peak": flops * value / world / 1e12 / peaks.get("bf16_tflops_sustained", 1400.0)},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
