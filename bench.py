#!/usr/bin/env python
"""bench.py — DDFA GGNN hot path: CFG graphs/sec of a full train step on B200.

Workload (default, BASELINE.json configs[2] / SURVEY.md §8 "C1"): synthetic Big-Vul-shaped batches of 1024 CFGs
per GPU x 150 nodes / 300 edges (incl. self loops), 4 x Embedding(1002,32) -> 128-d, T=8 propagation steps,
attention readout, 2-layer MLP head, BCE loss, backward, gradient all-reduce (N>1), Adam (coupled L2).
`--graphs 256` is C0 (configs[0]/[1]); the default N=1 run reports C0 as a second workload
(`secondary_workloads`).  Per-GPU batch is fixed as N grows (weak scaling; the batch shards by graphs, no
data-path collective).

  python bench.py --gpus 1 --steps K --warmup W            # our arm (CUDA, libddfa_b200.so)
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # ... and the last timed step's loss + parameters as .npy
  python bench.py --impl reference --steps K --warmup W    # reference arm: the reference path's CPU
                                                           # restatement (oracle/) on the host cores
One JSON line on stdout (rank 0).  See DESIGN.md §6 for every field.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FEAT = "_ABS_DATAFLOW_api_all_limitall_1000_limitsubkeys_1000"
CFG = dict(graphs=1024, nodes=150, edges_per_node=2.0, input_dim=1002, hidden_dim=32, n_steps=8, layers=2)
METRIC = "CFG graphs/sec (train step)"
UNIT = "graphs/s"
NUM_BATCHES = 8  # distinct resident batches rotated through the timed region


def workload_tag(graphs):
    return {1024: "C1", 256: "C0"}.get(graphs, f"B{graphs}")


def workload_config(graphs, world):
    """Identical in both arms (the driver compares the dicts)."""
    return {
        "workload": f"{workload_tag(graphs)}: {graphs} CFGs/GPU x {CFG['nodes']} nodes / {int(CFG['nodes'] * CFG['edges_per_node'])} edges, "
                    f"4xEmb(1002,32)->128-d, T={CFG['n_steps']}, attention readout, {CFG['layers']}-layer MLP, "
                    "BCE, backward, Adam (coupled L2)",
        "global_batch": graphs * world,
        "per_gpu_batch": graphs,
        "n_steps": CFG["n_steps"], "hidden": 128, "mlp_layers": CFG["layers"],
        "parallelism": f"dp{world}",
    }


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.thread = [], None, None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.rows.append((time.time(), line.strip()))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], None, set(), []
        for ts, line in self.rows:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                clk, mxc = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            mx = mxc
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk)
                try:
                    power.append(float(parts[3]))
                except ValueError:
                    pass
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # timed region shorter than the sampling period: fall back to all samples
            for ts, line in self.rows:
                parts = [p.strip() for p in line.split(",")]
                try:
                    sm.append(float(parts[1]))
                except (ValueError, IndexError):
                    pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ------------------------------------------------------------------------------------------------
# CUDA-event span profiler for selected C-ABI calls (engine.profile_hook)
# ------------------------------------------------------------------------------------------------
class SpanProfiler:
    def __init__(self, names):
        self.names = set(names)
        self.spans = {n: [] for n in names}
        self._open = {}
        self.enabled = True

    def wants(self, name):
        return self.enabled and name in self.names

    def begin(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self._open[name] = e

    def end(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.spans[name].append((self._open.pop(name), e))

    def mean_ms(self, name):
        xs = [a.elapsed_time(b) for a, b in self.spans[name]]
        return (sum(xs) / len(xs), len(xs)) if xs else (None, 0)

    def total_ms(self, name):
        return sum(a.elapsed_time(b) for a, b in self.spans[name])


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            d = json.load(f)
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                "bf16_tflops_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def ncu_traffic(kernel, n_nodes, mode):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed table of `ncu --set full`
    captures (profiles/ncu_traffic.json, written by scripts/ncu_lines.py from the .ncu-rep of the named capture), keyed by kernel,
    node count and mode.  None when no capture of that shape is committed — never a guess."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            table = json.load(f)
        e = table[kernel][f"N={n_nodes},{mode}"]
        return {"bytes": int(e["dram_read"]) + int(e["dram_write"]), "source": e.get("source")}
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference path's restatement (oracle/) on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_train_steps(graphs, steps, warmup, budget_s=None):
    """Times full train steps (fwd + BCE + bwd + Adam) of the oracle on the CPU. Returns (graphs/s, s/step, steps, threads)."""
    from deepdfa_b200 import synth
    from oracle import ggnn_oracle as O
    ncpu = os.cpu_count() or 1
    torch.manual_seed(0)
    model = O.OracleFlowGNNGGNN(FEAT, CFG["input_dim"], CFG["hidden_dim"], CFG["n_steps"], CFG["layers"], concat_all_absdf=True)
    opt = O.make_optimizer(model)
    batches = [synth.make_batch(graphs, CFG["nodes"], CFG["edges_per_node"], CFG["input_dim"], seed=i) for i in range(2)]
    probe = [synth.make_batch(min(graphs, 256), CFG["nodes"], CFG["edges_per_node"], CFG["input_dim"], seed=10 + i) for i in range(2)]

    def one(b):
        opt.zero_grad()
        loss, _ = model.training_loss(b)
        loss.backward()
        opt.step()
        return float(loss.detach())
    # The arm may use every host thread, but torch's intra-op pool oversubscribes on many-core hosts for these
    # small ops (128 threads measured 20x slower than 8): probe a few pool sizes on a 256-graph batch, keep the fastest.
    best_t, best_dt = 1, float("inf")
    for cand in sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu}):
        torch.set_num_threads(cand)
        one(probe[0])
        t0 = time.perf_counter()
        one(probe[1])
        dt = time.perf_counter() - t0
        if dt < best_dt:
            best_t, best_dt = cand, dt
        if dt > 3.0 * best_dt:
            break
    torch.set_num_threads(best_t)
    for i in range(warmup):
        one(batches[i % 2])
    t0 = time.perf_counter()
    done = 0
    for i in range(steps):
        one(batches[i % 2])
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s and done >= 2:
            break
    dt = time.perf_counter() - t0
    return graphs * done / dt, dt / done, done, torch.get_num_threads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    if args.dump_outputs:
        raise SystemExit("bench.py: --dump-outputs writes the CUDA arm's outputs; it has no --impl reference form")
    val, s_per_step, done, threads = cpu_train_steps(args.graphs, args.steps, max(min(args.warmup, 2), 1))
    out = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": done, "warmup": args.warmup,
        "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args.graphs, args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{done} full train steps of one {args.graphs}-graph {workload_tag(args.graphs)} batch (reference cannot run: dgl/"
                                   "pytorch_lightning absent; pure-PyTorch restatement oracle/ggnn_oracle.py, torch CPU, host threads as probed)"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": f"world_size={world}: rank 0 alone runs the CPU arm, one {args.graphs}-graph batch per step whatever N is",
    }
    print(json.dumps(out), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def batch_bytes(g):
    src, dst = g.edges()
    keys = [f"_ABS_DATAFLOW_{k}" for k in ("api", "datatype", "literal", "operator")] + ["_VULN"]
    n = src.numel() * src.element_size() + dst.numel() * dst.element_size() + g.batch_num_nodes().numel() * 8
    for k in keys:
        n += g.ndata[k].numel() * g.ndata[k].element_size()
    return n


class Ctx:
    """Process-wide state of our arm (device, ranks, library handle)."""
    pass


def timed_steps(ctx, fn_step, steps):
    """Milliseconds of EXACTLY `steps` calls of fn_step (barrier + synchronize on both sides, CUDA events, max over ranks)."""
    import torch.distributed as dist
    ctx.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn_step(i)
    e1.record()
    ctx.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=ctx.dev)
    if ctx.world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def dump_outputs(trainer, out_dir):
    """Writes what the caller of the timed step holds after the last timed step — the loss it returned and the module's updated
    parameters — as float32 <out_dir>/<name>.npy (1.2 MB at the default sizes), so two builds can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": trainer.loss_slot}
    arrays.update({f"param.{k}": p for k, p in trainer.module.named_parameters()})
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def roofline_lines(prof, ms_region, N, Eg, engine, peaks, mode_tag):
    """Per-kernel roofline entries from the CUDA-event spans of the instrumented (eager) region.
    P = one [N,128] fp32 plane = one activation image (hi+lo bf16).  Design bytes per launch (DESIGN.md §3):
      forward GRU step (train), packed state (round 2, the default): read s image, h image (2P); write h' image and the
        packed gate words, 8 B per element (3P)                                                                   = 5P
        (round-1 form, DDFA_PACKED_STATE=0: read s image, h image, h; write h', h' image, 4 gate planes         = 9P)
      backward GRU step (tcgen05: gate_bwd with the transposed gather folded in + dgrad3): gate_bwd reads dh, packed gates,
        h image (4P; round-1 form 6P) + E gathered ds rows, writes q x4 + dh'z (5P); dgrad reads q x4 + dh'z (5P),
        writes ds, dh (2P)                                                                     = 16P (18P) + E rows
      weight gradient, ONE launch per backward pass over all T steps: per step q x4 + s image + h image          = 6P x T
      edge gather: SURVEY.md §8(d) — E rows gathered + N rows written (+ the CSR arrays)
    and next to them SURVEY.md §8(d)'s own definitions: the GRU step's algorithmic bytes are 3P (read a/s, h; write h') and
    its FLOPs 229 376 per node-step (reference formulation, 7 D^2 MAC), against the bf16 tensor peak."""
    Dh, T = 128, CFG["n_steps"]
    P = N * Dh * 4
    share = {k: prof.total_ms(k) / ms_region for k in prof.spans}
    gather_bytes = Eg * Dh * 4 + N * Dh * 4 + Eg * 4 + (N + 1) * 4
    gf_ms, _ = prof.mean_ms("gather_fwd")
    gb_ms, _ = prof.mean_ms("gather_bwd")
    g_all = [a.elapsed_time(b) for a, b in prof.spans["gather_fwd"] + prof.spans["gather_bwd"]]
    g_ms = sum(g_all) / len(g_all)
    gru_f_ms, gru_f_n = prof.mean_ms("ddfa_gru_step_fwd")
    gru_b_ms, gru_b_n = prof.mean_ms("ddfa_gru_step_bwd")
    flops_fold = 2.0 * N * (6 * Dh * Dh)       # folded GRU GEMMs per propagation step (what the kernel multiplies, per bf16 pass)
    flops_8d = N * 229376.0                    # SURVEY.md §8(d): reference formulation per node-step

    def hbm_line(kernel, nbytes, t_ms, launches, sh, **extra):
        ach = nbytes / (t_ms * 1e-3) / 1e9
        return dict({"kernel": kernel, "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": ach / peaks["hbm_gbs"], "peak_source": peaks["source"], "bytes_per_launch": int(nbytes),
                     "avg_launch_us": t_ms * 1e3, "launches_timed": launches, "share_of_step": sh}, **extra)

    tc = engine == "tcgen05"
    from deepdfa_b200 import engine as _E
    packed = tc and bool(_E.OPTIONS.get("packed_state"))
    fwd_P, bwd_P = (5, 16) if packed else (9, 18)
    tr = ncu_traffic("gru_fwd3_kernel", N, "train") if tc else None
    fwd_line = hbm_line("gru_fwd3_kernel (GRU step forward, tcgen05: weights in TMEM, bf16x3)" if tc else "GRU step forward (simt engine)",
                        fwd_P * P, gru_f_ms, gru_f_n, share["ddfa_gru_step_fwd"], design_bytes=f"{fwd_P}P (P = N x 128 x 4 B)",
                        traffic=tr["bytes"] if tr else None, traffic_source=tr["source"] if tr else None,
                        algorithmic_bytes_8d=int(3 * P), frac_8d=3 * P / (gru_f_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                        flops_8d=flops_8d, tensor_frac_8d=flops_8d / (gru_f_ms * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"],
                        tensor_tflops_issued=3 * flops_fold / (gru_f_ms * 1e-3) / 1e12 if tc else None,
                        tensor_frac_issued=(3 * flops_fold / (gru_f_ms * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"]) if tc else None)
    wg_spans = prof.spans["wgrad_batched"]
    batched = tc and len(wg_spans) > 0
    bwd_line = hbm_line("GRU step backward: gate_bwd_tma_kernel / gate_bwd_image_kernel (+ folded transposed gather) + dgrad3_kernel" if tc
                        else "GRU step backward (simt engine)",
                        (bwd_P * P + Eg * Dh * 4) if batched else 24 * P, gru_b_ms, gru_b_n, share["ddfa_gru_step_bwd"], traffic=None,
                        tensor_tflops_issued=(3 if batched else 6) * flops_fold / (gru_b_ms * 1e-3) / 1e12 if tc else None)
    gtr = ncu_traffic("gather_sum_image_kernel", N, "train") if tc else None
    gather_line = hbm_line("gather_sum_kernel / gather_sum_image_kernel (CSR edge gather, fwd over CSR + bwd over transposed CSR)",
                           gather_bytes, g_ms, len(g_all), share["gather_fwd"] + share["gather_bwd"],
                           traffic=gtr["bytes"] if gtr else None, traffic_source=gtr["source"] if gtr else None,
                           fwd_us=gf_ms * 1e3, bwd_us=(gb_ms * 1e3 if gb_ms else None), storage_dtype="f32",
                           algorithmic_bytes_8d=int(gather_bytes))
    lines = [fwd_line, bwd_line, gather_line]
    if batched:
        wg_ms, wg_n = prof.mean_ms("wgrad_batched")
        lines.insert(2, hbm_line(f"wgrad_kernel + wgrad_reduce_kernel (weight gradients of all {T} steps in one launch)",
                                 6 * P * T, wg_ms, wg_n, share["wgrad_batched"], traffic=None,
                                 tensor_tflops_issued=3 * flops_fold * T / (wg_ms * 1e-3) / 1e12))
    roofline = dict(fwd_line, note="the forward GRU step kernel: ~24 % of the step and the hot kernel furthest below its roofline (the gate-backward + dgrad pair is the larger share, ~42 %, at ~0.95 of peak: roofline_kernels); frac = design bytes (bytes_per_launch; 5P with the packed saved state) "
                                   "over the launch time vs the measured HBM peak, frac_8d / tensor_frac_8d = SURVEY.md §8(d)'s algorithmic bytes / FLOPs")
    return roofline, lines


def measure_workload(ctx, args, graphs, full):
    """One workload (graphs per GPU) end to end.  full=False: headline value + e2e only (secondary workloads)."""
    import torch.distributed as dist
    import deepdfa_b200 as D
    from deepdfa_b200 import engine as E, synth
    from deepdfa_b200.batched_graph import BatchedCFG
    L, dev, rank, world = ctx.L, ctx.dev, ctx.rank, ctx.world
    trainer, steps = ctx.trainer, args.steps
    global_batch = graphs * world
    res = {}
    # distinct batches per rank and per slot (weak scaling: every rank has its own `graphs` graphs)
    host_batches = [synth.make_batch(graphs, CFG["nodes"], CFG["edges_per_node"], CFG["input_dim"], seed=1000 * rank + i).pin_memory()
                    for i in range(NUM_BATCHES)]
    dev_batches = [b.to(dev) for b in host_batches]
    N, Eg = dev_batches[0].num_nodes(), dev_batches[0].num_edges()
    min_warm = int(os.environ.get("DDFA_BENCH_MIN_WARMUP", "3"))   # 1 only for profiler runs (never a bench value)
    warm = max(args.warmup, min_warm)

    def step_dev(i):
        trainer.step(dev_batches[i % NUM_BATCHES], global_batch)

    trainer.use_cuda_graph = False
    for i in range(warm):            # also builds + caches the device CSR of every resident batch
        step_dev(i)
    torch.cuda.synchronize()
    l0 = L.call("ddfa_launch_count")
    step_dev(0)
    torch.cuda.synchronize()
    launches_per_step = L.call("ddfa_launch_count") - l0

    if full and not args.quick:
        # ---- instrumented region (eager launches): CUDA-event pairs around every gather / GRU-step call -> roofline -----
        prof = SpanProfiler(["gather_fwd", "gather_bwd", "ddfa_gru_step_fwd", "ddfa_gru_step_bwd", "wgrad_batched"])
        E.profile_hook = prof
        ctx.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            step_dev(i)
        ev1.record()
        ctx.barrier()
        E.profile_hook = None
        ms_instr = ev0.elapsed_time(ev1)                      # denominator of the kernel shares
        res["ms_per_step_eager_instrumented"] = ms_instr / steps
        if rank == 0:
            res["roofline"], res["roofline_kernels"] = roofline_lines(prof, ms_instr, N, Eg, args.engine, measured_peaks(), "train")

    # ---- capture one CUDA graph per resident batch (launch-bound inner loop: ~70 kernels per step) ------------------
    graph_note = "off (--no-graphs)"
    if args.cuda_graphs:
        try:
            trainer.use_cuda_graph = True
            for i in range(2 * NUM_BATCHES):        # first visit: capture, second visit: replay
                step_dev(i)
            torch.cuda.synchronize()
            graph_note = f"on (one graph per resident batch, {NUM_BATCHES} batches)"
        except Exception as exc:                    # an execution-mode downgrade, not a compute fallback: same kernels, eager launches
            trainer.use_cuda_graph = False
            trainer._graphs.clear()
            torch.cuda.synchronize()
            graph_note = f"off (capture failed: {type(exc).__name__}: {str(exc)[:120]})"
    res["cuda_graph"] = graph_note

    # ---- timed region (headline): K resident-input train steps -------------------------------------------------------------
    sampler = ClockSampler(ctx.local_rank)
    if rank == 0 and full:
        sampler.start()
        time.sleep(0.25)
    for i in range(warm):
        step_dev(i)
    t_wall0 = time.time()
    ms_total = timed_steps(ctx, step_dev, steps)
    t_wall1 = time.time()
    if rank == 0 and full:
        res["clocks"] = sampler.stop(t_wall0, t_wall1)
        if args.dump_outputs:
            dump_outputs(trainer, args.dump_outputs)
    res["final_loss"] = float(trainer.loss_slot.item())
    res["value"] = global_batch * steps / (ms_total * 1e-3)
    res["ms_per_step"] = ms_total / steps
    res["timed_ms"] = round(ms_total, 3)
    res["gpu_launches_per_step"] = int(launches_per_step)
    res["nodes"], res["edges"] = N, Eg

    # ---- e2e: host (pinned) buffers -> H2D -> device CSR build -> train step -> loss D2H, every step ----
    def fresh(b):  # a new graph object: no cached device CSR, so the whole input path is inside the timed region
        return BatchedCFG(*b.edges(), b.batch_num_nodes(), dict(b.ndata))
    for i in range(3):
        float(trainer.step(fresh(host_batches[i % NUM_BATCHES]), global_batch).item())
    state = {"nxt": fresh(host_batches[0]), "loss": None}
    trainer.prefetch(state["nxt"], global_batch)

    def step_e2e(i):
        cur = state["nxt"]
        loss_t = trainer.step(cur, global_batch)
        state["nxt"] = fresh(host_batches[(i + 1) % NUM_BATCHES])
        trainer.prefetch(state["nxt"], global_batch)          # the next step's H2D copies run on a side stream during this step
        state["loss"] = float(loss_t.item())
    ms_e2e = timed_steps(ctx, step_e2e, steps)
    res["e2e"] = {"value": global_batch * steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": batch_bytes(host_batches[0]),
                  "d2h_bytes_per_step": 4, "steps": steps,
                  "path": "FusedTrainer.step(host batch): pinned host COO + node indices -> H2D -> ddfa_build_csr -> fused train step -> loss .item()"
                          + (" (one CUDA graph per batch shape, two static input-buffer sets, next batch prefetched on a copy stream)"
                             if trainer.use_cuda_graph else " (eager launches)")}
    res["e2e_last_loss"] = state["loss"]
    if not full or args.quick:
        return res

    # ---- batch producer (SURVEY.md §8 f1): the same step fed from a device-resident graph arena by graph-id lists.  Reported
    # next to e2e, not instead of it: here only the id list crosses PCIe each step (the graphs were uploaded once).
    arena = D.GraphArena.from_graphs(host_batches, dev)
    rng = __import__("numpy").random.default_rng(rank)
    id_lists = [rng.integers(0, arena.num_graphs, graphs) for _ in range(NUM_BATCHES)]
    for i in range(3):
        float(trainer.step_ids(arena, id_lists[i % NUM_BATCHES], global_batch).item())

    def step_arena(i):
        state["loss"] = float(trainer.step_ids(arena, id_lists[i % NUM_BATCHES], global_batch).item())
    ms_arena = timed_steps(ctx, step_arena, steps)
    res["e2e_arena"] = {"value": global_batch * steps / (ms_arena * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 4 * graphs,
                        "d2h_bytes_per_step": 4, "steps": steps,
                        "path": f"graph-id list (pinned) -> H2D -> ddfa_arena_batch over a resident arena of {arena.num_graphs} graphs -> "
                                "fused train step -> loss .item()", "last_loss": state["loss"]}

    # ---- the reference user's own call sequence (INTEGRATION.md §2a): module.training_step + loss.backward() + torch.optim.Adam,
    # host batches, eager launches through autograd, loss .item() every step.  N = 1 only (under DDP the reference has no counterpart).
    if world == 1:
        torch.manual_seed(0)
        m2 = D.FlowGNNGGNNModule(FEAT, CFG["input_dim"], CFG["hidden_dim"], CFG["n_steps"], CFG["layers"], concat_all_absdf=True,
                                 engine=args.engine).to(dev)
        opt = m2.configure_optimizers()

        def step_api(i):
            b = fresh(host_batches[i % NUM_BATCHES])
            opt.zero_grad(set_to_none=True)
            loss = m2.training_step((b, {}), i)
            loss.backward()
            opt.step()
            state["loss"] = float(loss.item())
        for i in range(3):
            step_api(i)
        ms_api = timed_steps(ctx, step_api, steps)
        res["e2e_module_api"] = {"value": global_batch * steps / (ms_api * 1e-3), "unit": UNIT,
                                 "h2d_bytes_per_step": batch_bytes(host_batches[0]), "d2h_bytes_per_step": 4, "steps": steps,
                                 "path": "FlowGNNGGNNModule.training_step((host batch, {})) -> loss.backward() -> torch.optim.Adam.step() -> "
                                         "loss.item()  (autograd Function around the same kernels, eager launches, per-step allocation)",
                                 "last_loss": state["loss"]}
        del m2, opt
    return res


def measure_variable_stream(ctx, args, graphs):
    """Shuffled-epoch shape (datamodule.py:123-129): every batch has its own (N, E) — lognormal graph sizes, SURVEY.md §8(d) generator.
    The trainer pads each batch to a bucket shape so the per-shape CUDA graphs are reused (FusedTrainer, bucket_nodes / bucket_edges)."""
    from deepdfa_b200 import synth
    from deepdfa_b200.batched_graph import BatchedCFG
    trainer = ctx.trainer
    trainer.bucket_nodes, trainer.bucket_edges, trainer.max_graph_shapes = 4096, 8192, 64
    world, rank = ctx.world, ctx.rank
    global_batch = graphs * world
    n_batches = 24
    host = [synth.make_batch(graphs, CFG["nodes"], CFG["edges_per_node"], CFG["input_dim"], seed=5000 + 1000 * rank + i, variable=True).pin_memory()
            for i in range(n_batches)]
    nodes = sum(b.num_nodes() for b in host) / n_batches

    def fresh(b):
        return BatchedCFG(*b.edges(), b.batch_num_nodes(), dict(b.ndata))
    trainer.use_cuda_graph = bool(args.cuda_graphs)
    state = {"loss": None}
    for i in range(2 * n_batches):            # first visits of a bucket shape run eagerly, then capture
        float(trainer.step(fresh(host[i % n_batches]), global_batch).item())

    state["nxt"] = fresh(host[0])
    trainer.prefetch(state["nxt"], global_batch)

    def step_var(i):      # as in `e2e`: the next batch is staged (host padding + H2D on the copy stream) while this step runs
        cur = state["nxt"]
        loss_t = trainer.step(cur, global_batch)
        state["nxt"] = fresh(host[(i + 1) % n_batches])
        trainer.prefetch(state["nxt"], global_batch)
        state["loss"] = float(loss_t.item())
    ms = timed_steps(ctx, step_var, args.steps)
    shapes = sorted({(b.num_nodes(), b.num_edges()) for b in host})
    return {"value": global_batch * args.steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / args.steps, "steps": args.steps,
            "distinct_batch_shapes": len(shapes), "mean_nodes_per_batch": nodes, "bucket_shapes_captured": trainer.num_bucket_shapes(),
            "path": "FusedTrainer.step(host batch), variable=True lognormal graph sizes (mean 150 nodes), every batch a new (N, E); padded to bucket "
                    "shapes (one dummy graph of isolated nodes, zero loss weight), one CUDA graph per bucket shape, next batch prefetched; loss .item() every step",
            "last_loss": state["loss"]}


def run_ours(args):
    import torch.distributed as dist
    import deepdfa_b200 as D
    from deepdfa_b200 import _lib

    ctx = Ctx()
    ctx.rank = rank = int(os.environ.get("RANK", "0"))
    ctx.world = world = int(os.environ.get("WORLD_SIZE", "1"))
    ctx.local_rank = local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    ctx.dev = dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    ctx.L = L = _lib.lib()
    if L.call("ddfa_device_supported") != 1:
        raise SystemExit("bench.py: device is not compute capability 10.x")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    ctx.barrier = barrier

    torch.manual_seed(0)
    model = D.FlowGNNGGNNModule(FEAT, CFG["input_dim"], CFG["hidden_dim"], CFG["n_steps"], CFG["layers"], concat_all_absdf=True,
                                engine=args.engine).to(dev)
    # DDFA_AR_OVERLAP=0: one all-reduce of the whole flat buffer after the backward pass (A/B of the split exchange)
    # DDFA_EXCHANGE=p2p | nccl | auto (default; = the FusedTrainer default): p2p is the fused reduce-scatter + Adam + all-gather kernel
    # over NVLink peer memory, nccl the all-reduce + ddfa_adam_flat; auto takes p2p when the symmetric-memory set-up succeeds on all ranks
    exchange = os.environ.get("DDFA_EXCHANGE", "auto")
    ctx.trainer = trainer = D.FusedTrainer(model, overlap_allreduce=os.environ.get("DDFA_AR_OVERLAP", "1") != "0", exchange=exchange)

    # ---- data-parallel self-check (SURVEY.md §8(e) "Determinism"): k steps sharded over the N ranks vs the same k steps of the
    # unsharded global batch on one rank, same seeds — the loss curves must agree (fp32 summation order is the only difference).
    dp_parity = None
    if world > 1 and hasattr(D.FusedTrainer, "dp_self_check"):
        dp_parity = D.FusedTrainer.dp_self_check(args.engine, dev, rank, world, exchange=trainer.exchange)

    primary = measure_workload(ctx, args, args.graphs, full=True)
    secondary = []
    if args.secondary and args.graphs == 1024:
        s = measure_workload(ctx, args, 256, full=False)
        secondary.append({"config": workload_config(256, world), "value": s["value"], "unit": UNIT, "ms_per_step": s["ms_per_step"],
                          "e2e": s["e2e"], "cuda_graph": s["cuda_graph"], "timed_ms": s["timed_ms"]})
    variable = measure_variable_stream(ctx, args, args.graphs) if args.variable else None

    def leave():
        # Captured CUDA graphs hold NCCL kernels; tearing the communicator down under them can block (seen at N = 2:
        # the JSON line was out, the process never exited).  Drop the graphs, drain the device and leave without the
        # collective teardown — nothing else runs in this process.
        trainer._graphs.clear()
        trainer._stream_slots.clear()
        torch.cuda.synchronize()
        if world > 1:
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)
        return 0

    if rank != 0:
        return leave()

    # ---- cpu baseline on this box's host cores (bounded sample) ----------------------------------------
    if os.environ.get("DDFA_BENCH_SKIP_CPU") == "1" or args.quick:     # profiler / scaling A/B runs only
        cpu_val, cpu_s, cpu_done, cpu_threads = None, None, 0, 0
    else:
        cpu_val, cpu_s, cpu_done, cpu_threads = cpu_train_steps(args.graphs, 8, 1, budget_s=20.0)

    N = primary["nodes"]
    out = {
        "metric": METRIC, "value": primary["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": primary["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if args.engine == "simt" else "f32 (GRU GEMMs: bf16x3 split operands, f32 accumulate)",
        "data": "synthetic", "config": workload_config(args.graphs, world),
        "engine": args.engine,
        "l2": f"per-step working set ~{N * 128 * 4 * 49 / 1e9:.2f} GB of saved activations > 126 MB L2; {NUM_BATCHES} distinct resident batches rotated",
        "timed_ms": primary["timed_ms"],
        "clocks": primary.get("clocks"),
        "e2e": primary["e2e"], "e2e_arena": primary.get("e2e_arena"), "e2e_module_api": primary.get("e2e_module_api"),
        "e2e_variable": variable,
        "gpu_launches": int(primary["gpu_launches_per_step"] * args.steps), "gpu_launches_per_step": primary["gpu_launches_per_step"],
        "cuda_graph": primary["cuda_graph"], "ms_per_step_eager_instrumented": primary.get("ms_per_step_eager_instrumented"),
        "roofline": primary.get("roofline"), "roofline_kernels": primary.get("roofline_kernels"),
        "secondary_workloads": secondary,
        "dp_parity": dp_parity,
        "allreduce": None if world == 1 else ("fused peer-memory kernel: reduce-scatter + Adam + all-gather over NVLink (ddfa_allreduce_adam_p2p), no NCCL in the step"
                                              if trainer.exchange == "p2p" else "split: small gradients on a side stream during the weight-gradient launch, GGNN weight "
                                              "gradients after it" if trainer.overlap_allreduce else "single call after the backward pass"),
        "exchange": None if world == 1 else {"requested": exchange, "used": trainer.exchange, "note": trainer.exchange_note},
        "cpu_baseline": {"value": cpu_val, "unit": UNIT, "cores": cpu_threads, "kind": "port",
                         "sample": f"{cpu_done} full train steps of one {args.graphs}-graph {workload_tag(args.graphs)} batch, oracle/ggnn_oracle.py (torch CPU)"},
        "final_loss": primary["final_loss"], "e2e_last_loss": primary["e2e_last_loss"],
    }
    print(json.dumps(out), flush=True)
    return leave()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--graphs", type=int, default=CFG["graphs"], help="graphs per GPU per step (1024 = C1, 256 = C0)")
    ap.add_argument("--engine", choices=["simt", "tcgen05"], default=os.environ.get("DDFA_B200_ENGINE", "tcgen05"))
    ap.add_argument("--no-graphs", dest="cuda_graphs", action="store_false", help="launch every kernel eagerly in the timed region")
    ap.add_argument("--no-secondary", dest="secondary", action="store_false", help="skip the C0 second workload of the default run")
    ap.add_argument("--no-variable", dest="variable", action="store_false", help="skip the variable-shape stream line")
    ap.add_argument("--quick", action="store_true", help="headline value + e2e only (no per-kernel spans, arena / module-API lines, CPU baseline): scaling A/Bs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the loss and the updated parameters of the last one "
                                                          "to DIR/<name>.npy (same arguments, same inputs)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
