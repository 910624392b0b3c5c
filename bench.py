#!/usr/bin/env python
"""bench.py - multi-crop images/sec of the EsViT self-distillation training step (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU)
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores (oracle port)

A "step" is one full training step over one synthetic batch: teacher fwd on 2 global crops, student fwd/bwd on
2 global + 8 local crops, DDINOLoss (view + region), packed center all-reduce, per-tensor clip, AdamW, teacher EMA.
`value` = images/s with the crops already resident in HBM; `e2e` = the same step fed from pinned HOST buffers
(H2D of all crops + D2H of the loss inside the timed region).  One JSON line on stdout (rank 0).
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "multi-crop images/sec, Swin-T W7 pretrain step (2 global 224^2 + 8 local 96^2 crops, DDINOLoss V+R, K=65536)"
WORKLOAD = "swin_tiny_w7 2+8 crops DDINOLoss out_dim=65536 (BASELINE.json configs[1])"


def attention_core_tflops(timed, n_eager):
    """SURVEY.md 8(d) metric 2: algorithmic FLOPs of the attention core (QK^T + PV over the ws*ws slots of every window
    the reference computes, padded ones included; head_dim 32) / measured kernel time, forward and backward separately
    (backward = the standard 2.5x: recompute S, dP, dQ, dK, dV).  The QKV / proj GEMMs are separate kernels here."""
    out = {}
    for key, name, mult in (("fwd", "esvit_window_attn_fwd", 1.0), ("bwd", "esvit_window_attn_bwd", 2.5)):
        sel = [t for t in timed if t["name"] == name and "windows" in t]
        if not sel:
            continue
        flops = sum(mult * t["windows"] * t["nH"] * 2 * 2 * (t["ws"] ** 2) ** 2 * 32 for t in sel)
        ms = sum(t["ms"] for t in sel)
        out[key] = {"tflops": flops / (ms / 1e3) / 1e12, "gflop_per_step": flops / n_eager / 1e9, "ms_per_step": ms / n_eager}
    return out


def describe(args):
    """metric / workload strings; the defaults are BASELINE.json configs[1], other --arch values are parity-test configs."""
    if args.arch == "swin_tiny_w7" and args.local_crops == 8 and args.out_dim == 65536:
        return METRIC, WORKLOAD
    return (f"multi-crop images/sec, {args.arch} pretrain step (2 global 224^2 + {args.local_crops} local 96^2 crops, "
            f"DDINOLoss V+R, K={args.out_dim})",
            f"{args.arch} 2+{args.local_crops} crops DDINOLoss out_dim={args.out_dim} (not the headline config)")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="esvit_b200", choices=["esvit_b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="images per GPU per step")
    ap.add_argument("--arch", default="swin_tiny_w7")
    ap.add_argument("--out-dim", type=int, default=65536)
    ap.add_argument("--local-crops", type=int, default=8)
    ap.add_argument("--device", default=None, help="reference arm only: cpu (default) or cuda (eager oracle)")
    ap.add_argument("--ref-batch", type=int, default=2, help="reference arm: images per bounded-sample step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--profile", default=None, help="write a torch.profiler kernel table of 1 step to this path")
    ap.add_argument("--min-warmup", type=int, default=3, help="floor on warm-up steps (profiling runs lower it)")
    ap.add_argument("--no-graph", action="store_true", help="run the step eagerly instead of as a replayed CUDA graph")
    ap.add_argument("--optimizer", default="fused", choices=["fused", "torch"])
    ap.add_argument("--no-gpu-reference", action="store_true",
                    help="skip the `gpu_reference` entry (the unmodified reference modules timed on the same GPUs)")
    ap.add_argument("--gpu-ref-steps", type=int, default=10)
    ap.add_argument("--gpu-ref-precisions", default="bf16,fp16")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step computed (loss, loss centers, a seeded sample of the student "
                         "and teacher parameters) as DIR/<name>.npy in float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def load_ncu_traffic() -> dict:
    """{kernel key: {"dram_bytes", "algorithmic_bytes", "ncu_launch", "commit"}} from profiles/ncu_traffic.json."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        return {}


def cuda_parity_loss(arch: str, out_dim: int, n_local: int, batch: int, dev) -> float:
    """first-step DDINO loss of the CUDA path on the cpu_baseline's inputs: same seed-0 random-init weights, same
    seeded crops, DropPath 0, centers 0 (what oracle/step.py computes in its first step)."""
    from esvit_b200 import engine
    step, student, teacher, loss_mod = engine.make_step(arch=arch, out_dim=out_dim, ncrops=2 + n_local, dense=True,
                                                        device=dev, drop_path=0.0, seed=0)
    crops = [c.to(dev) for c in synthetic_crops(batch, n_local, 0)]
    with torch.no_grad():
        t = teacher(crops[:2])
        s = student(crops)
        l = float(loss_mod(s, t, 0, None))
    del step, student, teacher, loss_mod
    return l


def synthetic_crops(batch: int, n_local: int, rank: int):
    """BASELINE.md §2.3: per-rank generator 1234+r, N(0,1) fp32 crops."""
    g = torch.Generator().manual_seed(1234 + rank)
    crops = [torch.randn(batch, 3, 224, 224, generator=g) for _ in range(2)]
    crops += [torch.randn(batch, 3, 96, 96, generator=g) for _ in range(n_local)]
    return crops


def dump_outputs(out_dir: str, loss, student, teacher, loss_mod, per_param: int = 4096) -> None:
    """What a caller of the step holds after it: the loss, the updated loss centers and the updated student / teacher
    parameters, one float32 .npy each.  The parameters hold ~10^8 values, so each contributes a fixed seeded sample of
    at most `per_param` elements (all of a smaller one), concatenated in named_parameters() order; two builds run with
    the same arguments sample the same elements."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().reshape(1), "center": loss_mod.center, "center_grid": loss_mod.center_grid}
    for name, net in (("student_params", student), ("teacher_params", teacher)):
        g = torch.Generator().manual_seed(0)
        parts = []
        for p in net.parameters():
            flat = p.detach().reshape(-1)
            if flat.numel() > per_param:
                flat = flat[torch.randint(flat.numel(), (per_param,), generator=g).to(flat.device)]
            parts.append(flat.float())
        arrays[name] = torch.cat(parts)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def max_over_ranks(ms: float, device) -> float:
    if dist.is_initialized():
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return ms


def barrier_sync():
    if dist.is_initialized():
        dist.barrier()
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------
def pick_cpu_threads(sd, spec, crops) -> int:
    """All the host threads the reference path can USE: eager fp32 torch on many small ops collapses when
    oversubscribed (128 threads measured 150x slower than 8-16 on the pool's hosts), so the thread count is
    calibrated on one teacher forward among {8,16,32,64} capped by the cores this process may run on."""
    from oracle import swin as S
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    try:  # cgroup v2 CPU quota
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            avail = max(1, min(avail, int(int(q) / int(p))))
    except Exception:
        pass
    best, best_t = 1, float("inf")
    for n in (8, 16, 32, 64):
        if n > avail and n != 8:
            break
        n = min(n, avail)
        torch.set_num_threads(n)
        with torch.no_grad():
            S.multicrop_forward([c[:1] for c in crops[:2]], sd, spec)  # warm
            t0 = time.perf_counter()
            S.multicrop_forward([c[:1] for c in crops[:2]], sd, spec)
            dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    return best


def cpu_reference_steps(arch: str, out_dim: int, n_local: int, batch: int, steps: int, warmup: int, device: str = "cpu"):
    """The oracle port of the reference step (oracle/step.py) timed on the host cores (all threads)."""
    from esvit_b200.engine import SWIN_SPECS
    from oracle import step as ST
    from oracle import swin as S
    spec_d = SWIN_SPECS[arch]
    spec = S.SwinSpec(img_size=224, embed_dim=spec_d["embed_dim"], depths=tuple(spec_d["depths"]),
                      num_heads=tuple(spec_d["num_heads"]), window_size=spec_d["window_size"], use_dense_prediction=True)
    # random-init weights of the architecture, through the product's module constructors (same init law as the reference)
    from esvit_b200.engine import build_network
    torch.manual_seed(0)
    net = build_network(dict(spec_d), out_dim, True)
    sd = {k: v.detach() for k, v in net.state_dict().items()}
    del net
    crops = [c.to(device) for c in synthetic_crops(batch, n_local, 0)]
    cores = pick_cpu_threads(sd, spec, crops) if device == "cpu" else 1
    torch.set_num_threads(cores)
    orc = ST.OracleStep(sd, spec, 2 + n_local, out_dim, device=device)
    losses = []
    if device != "cpu":
        def run(n):
            for _ in range(n):
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    losses.append(orc.step(crops))
            torch.cuda.synchronize()
    else:
        def run(n):
            for _ in range(n):
                losses.append(orc.step(crops))
    run(warmup)
    t0 = time.perf_counter()
    run(steps)
    dt = (time.perf_counter() - t0) / steps
    return dt, cores, losses


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    device = args.device or "cpu"
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    if device == "cpu":
        steps, warmup = min(steps, 3), min(warmup, 1)  # bounded sample: ~1-8 s per B=2 step depending on the host
        batch = args.ref_batch
    else:
        batch = args.batch
    kind = "port"
    if device != "cpu":
        from baseline import reference_gpu as RG
        if RG.available():  # the UNMODIFIED reference modules (baseline/_ref) through train_one_epoch's sequence
            from esvit_b200.engine import SWIN_SPECS
            torch.cuda.set_device(0)
            dev = torch.device("cuda", 0)
            crops = [c.to(dev) for c in synthetic_crops(batch, args.local_crops, 0)]
            prec = args.gpu_ref_precisions.split(",")[0]
            r = RG.time_reference(dict(SWIN_SPECS[args.arch]), args.out_dim, 2 + args.local_crops, crops, dev, prec, steps,
                                  warmup, SWIN_SPECS[args.arch]["drop_path_rate"])
            dt, cores, kind = r["ms_per_step"] / 1e3, 0, "reference"
        else:
            dt, cores, _ = cpu_reference_steps(args.arch, args.out_dim, args.local_crops, batch, steps, warmup, device)
    else:
        dt, cores, _ = cpu_reference_steps(args.arch, args.out_dim, args.local_crops, batch, steps, warmup, device)
    val = batch / dt
    sample = f"{steps} steps of batch {batch} ({WORKLOAD}), fp32, oracle port (oracle/step.py), {cores} threads" \
        if device == "cpu" else (f"{steps} steps of batch {batch}, " + ("unmodified reference modules (baseline/_ref) on cuda"
                                 if kind == "reference" else "oracle port eager on cuda with bf16 autocast"))
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus,
           "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32" if device == "cpu" else "bf16", "data": "synthetic",
           "config": {"workload": WORKLOAD, "batch_per_step": batch, "device": device},
           "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": kind, "sample": sample},
           "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


# ---------------------------------------------------------------------------------------------------------
def main():
    global METRIC, WORKLOAD
    args = parse()
    METRIC, WORKLOAD = describe(args)
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs CUDA (there is no CPU fallback of the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"

    from esvit_b200 import _lib, engine
    B, n_local = args.batch, args.local_crops
    ncrops = 2 + n_local
    base_lr = 5e-4 * (B * world) / 256.0
    use_graph = (not args.no_graph) and args.optimizer == "fused"
    step, student, teacher, loss_mod = engine.make_step(
        arch=args.arch, out_dim=args.out_dim, ncrops=ncrops, dense=True, device=dev, lr=base_lr, ddp=world > 1,
        optimizer=args.optimizer, cuda_graph=use_graph)
    student.train()
    teacher.train()
    host = [c.pin_memory() for c in synthetic_crops(B, n_local, rank)]
    crops = [c.to(dev) for c in host]
    wd, mom, epoch = 0.04, 0.996, 1  # epoch >= freeze_last_layer so the last layer trains (steady-state work)

    def one_step(imgs):
        return step(imgs, epoch, base_lr, wd, mom)

    # ---- roofline of the dominant kernel: CUDA events around each launch, in EAGER steps (events cannot be
    # recorded inside a replayed graph); these steps double as the warm-up the graph capture needs -------------
    l = one_step(crops)  # first step untimed: lazy module loading / attribute calls must not pollute the per-kernel timings
    torch.cuda.synchronize()
    _lib.reset_counters()
    _lib.time_entry_point(["esvit_dino_ce_bwd", "esvit_dino_ce_fwd", "esvit_dino_ce_q_bwd", "esvit_dino_ce_q_fwd", "esvit_row_softmax_q", "esvit_window_attn_bwd", "esvit_window_attn_fwd",
                            "esvit_gemm_bias_act", "esvit_gemm_mul_colsum", "esvit_gemm_bf16", "esvit_gemm_mul_colsum2",
                            "esvit_gemm_wgrad", "esvit_add_ln_fwd", "esvit_add_ln_bwd", "esvit_patch_embed_fwd",
                            "esvit_patch_embed_bwd"])
    n_eager = 2 if args.min_warmup >= 3 else 1
    for _ in range(n_eager):
        l = one_step(crops)
    torch.cuda.synchronize()
    timed = _lib.timed_results()
    launches_per_step = _lib.launch_count() // n_eager
    _lib.time_entry_point(None)
    for _ in range(max(args.warmup, args.min_warmup)):  # graph mode: the first of these captures, the rest replay
        l = one_step(crops)
    torch.cuda.synchronize()
    assert torch.isfinite(l).item(), "non-finite loss in warm-up"

    # ---- timed region: K steps, device-resident inputs ---------------------------------------------------
    K = args.steps
    sampler = ClockSampler(local_rank)
    barrier_sync()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        l = one_step(crops)
        float(l)  # the loss is read back every step, as train_one_epoch does (main_esvit.py:546, :596): ranks stay in step
    e1.record()
    barrier_sync()
    clocks = sampler.stop() if rank == 0 else None
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, l, student, teacher, loss_mod)
    launches = launches_per_step * K  # esvit_b200 kernels per step (counted in the eager steps) x K
    ms_per_step = ms / K
    value = world * B / (ms_per_step / 1e3)

    # ---- end to end: pinned host crops -> H2D every step, loss read back every step ----------------------
    e2e = None
    if not args.no_e2e:
        # Every step's crops start in PINNED HOST memory and are copied to the device inside the timed region; the copy
        # of batch i+1 runs on a side stream while step i computes (what a prefetching DataLoader with
        # pin_memory + non_blocking .cuda() gives main_esvit.py:513), and every step's loss is read back (4 B, D2H +
        # host sync, like metric_logger.update(loss=loss.item()) at :596).
        h2d = sum(c.numel() * c.element_size() for c in host)
        copy_stream = torch.cuda.Stream()
        bufs = [[torch.empty_like(c) for c in crops] for _ in range(2)]
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]

        def prefetch(slot):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[slot])
                for dbuf, hbuf in zip(bufs[slot], host):
                    dbuf.copy_(hbuf, non_blocking=True)
                ready[slot].record(copy_stream)

        def run_e2e(nsteps):
            for slot in (0, 1):
                consumed[slot].record()
            prefetch(0)
            lv = 0.0
            for i in range(nsteps):
                cur = i & 1
                prefetch(cur ^ 1)                                   # batch i+1: H2D overlaps step i
                torch.cuda.current_stream().wait_event(ready[cur])
                out = one_step(bufs[cur])
                consumed[cur].record()
                lv = float(out)                                      # D2H of the loss + host sync, every step
            return lv

        run_e2e(2)
        barrier_sync()
        e0.record()
        lv = run_e2e(K)
        e1.record()
        barrier_sync()
        ms_e = max_over_ranks(e0.elapsed_time(e1), dev) / K
        e2e = {"value": world * B / (ms_e / 1e3), "unit": "images/s", "ms_per_step": ms_e,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "last_loss": lv,
               "h2d": "pinned host -> device on a side stream, overlapped with the previous step"}

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")
    roofline, roofline_others = None, []
    if timed:
        def agg(name, bytes_fn, label, extra=None):
            sel = [t for t in timed if t["name"] == name and (extra is None or extra(t))]
            if not sel:
                return None
            ms = sum(t["ms"] for t in sel)
            alg = sum(bytes_fn(t) for t in sel)
            ach = alg / (ms / 1e3) / 1e9
            return {"kernel": label, "timed_in": f"{n_eager} eager step(s) before the graph-replayed region (CUDA events per launch)",
                    "bound": "hbm", "achieved": ach, "peak": hbm_peak, "peak_source": peak_src, "unit": "GB/s",
                    "frac": ach / hbm_peak, "traffic": None, "launch_ms": ms / len(sel),
                    "algorithmic_bytes": alg / len(sel), "launches_timed": len(sel), "ms_per_step": ms / n_eager}
        Tg, Tl = 49, 9
        rows_s = B * (2 * Tg + n_local * Tl)
        rows_t = B * 2 * Tg
        # the CE kernels run on stored teacher probabilities (esvit_dino_ce_q_*) unless ESVIT_CE_Q=0
        used_q = any(t["name"] == "esvit_dino_ce_q_fwd" for t in timed)
        ce_q = "_q" if used_q else ""
        ce_fwd_name, ce_bwd_name = "esvit_dino_ce%s_fwd" % ce_q, "esvit_dino_ce%s_bwd" % ce_q
        # attention backward (the largest of this repo's kernels by time): reads qkv (6C) + dO (2C) + O (2C), writes dqkv
        # (6C) bytes per token -> 16*C per token (DESIGN.md section 4); forward: 8*C per token
        wtag = "7_kernel" if "w14" not in args.arch else "14_kernel + 7_kernel (stage 3)"
        r_bwd = agg("esvit_window_attn_bwd", lambda t: 16 * t["tokens"] * t["C"], f"window_attn_bwd{wtag} (all launches of a step)")
        r_fwd = agg("esvit_window_attn_fwd", lambda t: 8 * t["tokens"] * t["C"], f"window_attn_fwd{wtag} (all launches of a step)")
        # region-row CE backward: read student rows + each paired teacher row once + write bf16 grads:
        # (170 + 98 + 170) rows x K x 2 B per image (SURVEY.md 8d)
        r_ce = agg(ce_bwd_name, lambda t: (2 * rows_s + rows_t) * t["K"] * 2, "dino_ce%s_bwd_kernel (region rows)" % ce_q,
                   extra=lambda t: t["rows"] == rows_s)
        # tcgen05 fc1 GEMM + bias + GELU: reads A (M*K) and W, writes out and gelu' (2*M*N) in bf16
        r_gemm = agg("esvit_gemm_bias_act", lambda t: 2 * (t["M"] * t["K"] + t["N"] * t["K"] + 2 * t["M"] * t["N"]),
                     "tg::gemm_bias_act_kernel tcgen05 fc1+bias+GELU (all launches of a step)")
        # same kernel, third epilogue (fc2 dgrad * gelu' + column sums): reads dy (M*K), W2^T, gelu' (M*N), writes d(pre) (M*N)
        r_gemm2 = agg("esvit_gemm_mul_colsum", lambda t: 2 * (t["M"] * t["K"] + t["N"] * t["K"] + 2 * t["M"] * t["N"]),
                      "tg::gemm_bias_act_kernel tcgen05 fc2-dgrad*gelu'+colsum (all launches of a step)")
        # dram__bytes_read.sum + dram__bytes_write.sum per launch from `ncu --set full` captures: read from the JSON that
        # scripts/ncu_summarize.py wrote from the capture (with the commit it was taken at), never pasted in here
        traffic = load_ncu_traffic()
        for r, key in ((r_bwd, "window_attn_bwd"), (r_fwd, "window_attn_fwd"), (r_ce, "dino_ce_bwd"),
                       (r_gemm, "gemm_bias_act"), (r_gemm2, "gemm_mul_colsum")):
            if r and key in traffic:
                r["traffic"] = traffic[key]
        # second-generation GEMM family (every Linear): bytes = operands read + result written; flops = 2 M N K
        def gemm_bytes(t):
            out_b = 2 * t["M"] * t["N"] * (2 if t.get("pre") else 1)
            return 2 * (t["M"] * t["K"] + t["N"] * t["K"]) + out_b
        bf_peak = peaks.get("bf16_tflops_sustained", 1400.0)

        def with_flops(r, name, flops_fn, extra=None):
            if r:
                sel = [t for t in timed if t["name"] == name and (extra is None or extra(t))]
                fl = sum(flops_fn(t) for t in sel)
                ms_ = sum(t["ms"] for t in sel)
                r["tflops"] = fl / (ms_ / 1e3) / 1e12
                r["tensor_frac_of_sustained_bf16"] = r["tflops"] / bf_peak
            return r
        g_fwd = with_flops(agg("esvit_gemm_bf16", gemm_bytes, "tg2::gemm_kernel forward Linear (+bias / +GELU) (all launches of a step)",
                               extra=lambda t: not t["b_mn"]),
                           "esvit_gemm_bf16", lambda t: 2.0 * t["M"] * t["N"] * t["K"], lambda t: not t["b_mn"])
        g_dgr = with_flops(agg("esvit_gemm_bf16", gemm_bytes, "tg2::gemm_kernel input gradient (MN-major B) (all launches of a step)",
                               extra=lambda t: t["b_mn"]),
                           "esvit_gemm_bf16", lambda t: 2.0 * t["M"] * t["N"] * t["K"], lambda t: t["b_mn"])
        g_mul = with_flops(agg("esvit_gemm_mul_colsum2", lambda t: 2 * (t["M"] * t["K"] + t["N"] * t["K"] + 2 * t["M"] * t["N"]),
                               "tg2::gemm_kernel fc2-dgrad * gelu' + colsum (all launches of a step)"),
                           "esvit_gemm_mul_colsum2", lambda t: 2.0 * t["M"] * t["N"] * t["K"])
        g_wgr = with_flops(agg("esvit_gemm_wgrad", lambda t: 2 * t["T"] * (t["N"] + t["K"]) + 4 * t["N"] * t["K"],
                               "tg2::gemm_kernel weight gradient (MN-major A and B, split-K) + fold (all launches of a step)"),
                           "esvit_gemm_wgrad", lambda t: 2.0 * t["T"] * t["N"] * t["K"])
        r_lnf = agg("esvit_add_ln_fwd", lambda t: t["T"] * t["C"] * ((4 if t["has_x"] else 0) + (2 if t["has_delta"] else 0) + 4 + 2),
                    "add_ln_fwd_kernel (all launches of a step)")
        r_lnb = agg("esvit_add_ln_bwd", lambda t: 16 * t["T"] * t["C"], "add_ln_bwd_kernel (all launches of a step)")
        r_cef = agg(ce_fwd_name, lambda t: (rows_s + rows_t) * t["K"] * 2, "dino_ce%s_fwd_kernel (region rows)" % ce_q,
                    extra=lambda t: t["rows"] == rows_s)
        r_pef = agg("esvit_patch_embed_fwd", lambda t: t["B"] * (3 * t["H"] * t["W"] * 4 + (t["H"] // 4) * (t["W"] // 4) * t["E"] * 4),
                    "patch_embed_fwd2_kernel (all launches of a step)")
        r_peb = agg("esvit_patch_embed_bwd", lambda t: t["B"] * (3 * t["H"] * t["W"] * 4 + (t["H"] // 4) * (t["W"] // 4) * t["E"] * 4),
                    "patch_embed_bwd2_kernel (all launches of a step)")
        # teacher rows once: read bf16 logits, write fp16 probabilities (all launches: cls + region rows)
        r_rsq = agg("esvit_row_softmax_q", lambda t: t["rows"] * t["K"] * 4, "row_softmax_q_kernel (all teacher rows of a step)")
        for r, key in ((g_fwd, "gemm_bf16"), (g_mul, "gemm_mul_colsum"), (g_wgr, "gemm_wgrad"), (r_lnf, "add_ln_fwd"), (r_lnb, "add_ln_bwd")):
            if r and key in traffic:
                r["traffic"] = traffic[key]
        cands = [r for r in (r_bwd, r_fwd, r_ce, r_gemm, r_gemm2, g_fwd, g_dgr, g_mul, g_wgr, r_lnf, r_lnb, r_cef, r_pef, r_peb, r_rsq) if r]
        if cands:
            cands.sort(key=lambda r: -r["ms_per_step"])
            roofline, roofline_others = cands[0], cands[1:]

    # whole step against the dense bf16 tensor roofline: algorithmic FLOPs per image-step of SURVEY.md 8(a)
    GFLOP_PER_IMAGE = {("swin_tiny_w7", 8): 154.4, ("swin_small_w14", 10): 429.3, ("swin_base_w14", 10): 715.5}
    step_roofline = None
    gf = GFLOP_PER_IMAGE.get((args.arch, n_local)) if args.out_dim == 65536 else None
    if gf:
        pk = peaks.get("bf16_tflops_sustained", 1400.0)
        ach = gf * value / 1e3 / world  # TFLOP/s per GPU
        step_roofline = {"bound": "tensor", "achieved": ach, "peak": pk, "unit": "TFLOP/s", "frac": ach / pk,
                         "peak_source": "measured sustained bf16 (MEASURED_PEAKS.json)" if "bf16_tflops_sustained" in peaks else "fallback",
                         "gflop_per_image_step": gf}

    if args.profile and rank == 0:
        step.use_cuda_graph = False
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            one_step(crops)
            torch.cuda.synchronize()
        with open(args.profile, "w") as f:
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=60, max_name_column_width=90))
        if os.environ.get("ESVIT_PROFILE_STACKS"):  # who launches the small ATen copy / add / fill kernels
            with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU], with_stack=True, record_shapes=True) as prof2:
                one_step(crops)
                torch.cuda.synchronize()
            rows = [e for e in prof2.key_averages(group_by_input_shape=True, group_by_stack_n=8)
                    if e.key in ("aten::copy_", "aten::add_", "aten::add", "aten::fill_", "aten::zero_", "aten::cat",
                                 "aten::clone", "aten::contiguous", "aten::sum", "aten::mul", "aten::mul_", "aten::div",
                                 "aten::_to_copy", "aten::index", "aten::where", "aten::stack")]
            rows.sort(key=lambda e: -e.count)
            with open(args.profile + ".stacks.txt", "w") as f:
                for e in rows[:90]:
                    f.write(f"{e.key} x{e.count} cuda_total={e.device_time_total:.0f}us shapes={e.input_shapes}\n")
                    for fr in e.stack[:8]:
                        f.write(f"      {fr}\n")

    from esvit_b200.engine import SWIN_SPECS
    drop_path = SWIN_SPECS[args.arch]["drop_path_rate"]
    parity_cuda = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        parity_cuda = cuda_parity_loss(args.arch, args.out_dim, n_local, args.ref_batch, dev)

    # free the product path (graphs first: they hold the captured NCCL work) before the reference arms run
    own_mem_gib = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    last_loss = float(l)
    del l
    step._graphs.clear()
    del step, student, teacher, loss_mod
    import gc
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

    # ---- the reference's own PyTorch modules on the same GPU(s), same workload, same batch ------------------
    gpu_reference = None
    if not args.no_gpu_reference:
        try:
            from baseline import reference_gpu as RG
            if not RG.available():
                gpu_reference = {"unavailable": "baseline/_ref missing (run __graft_entry__.build() where /root/reference exists)"}
            else:
                runs = []
                for prec in [x for x in args.gpu_ref_precisions.split(",") if x]:
                    torch.cuda.reset_peak_memory_stats(dev)
                    r = RG.time_reference(dict(SWIN_SPECS[args.arch]), args.out_dim, ncrops, crops, dev, prec,
                                          args.gpu_ref_steps, 3, drop_path)
                    r["value"] = world * B / (r["ms_per_step"] / 1e3)
                    runs.append(r)
                best = max(runs, key=lambda r: r["value"])
                gpu_reference = {
                    "what": "UNMODIFIED reference modules (models/swin_transformer.py, models/vision_transformer.py DINOHead, "
                            "main_esvit.py DDINOLoss; baseline/_ref) driven through train_one_epoch's sequence "
                            "(main_esvit.py:507-598): autocast, DDP at N>1, per-parameter clip, torch AdamW, EMA loop",
                    "same_config": True, "batch_per_gpu": B, "n_gpus": world, "unit": "images/s",
                    "value": best["value"], "ms_per_step": best["ms_per_step"], "precision": best["precision"], "runs": runs,
                    "speedup_value": value / best["value"],
                    "speedup_e2e": (e2e["value"] / best["value"]) if e2e else None}
        except Exception as ex:  # noqa: BLE001 - the reference arm must never take the product line down
            gpu_reference = {"error": repr(ex)[:400]}

    cpu_baseline, parity_check = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        dt, cores, ol = cpu_reference_steps(args.arch, args.out_dim, n_local, args.ref_batch, 3, 1)
        cpu_baseline = {"value": args.ref_batch / dt, "unit": "images/s", "cores": cores, "kind": "port",
                        "sample": f"3 steps (+1 warm-up) of batch {args.ref_batch} of the same workload, fp32, "
                                  f"oracle/step.py on {cores} host threads, {dt:.2f} s/step"}
        tol = 5e-3
        err = abs(parity_cuda - ol[0]) / abs(ol[0])
        parity_check = {"what": f"first-step DDINO loss, batch {args.ref_batch}, seed-0 weights, DropPath 0: CUDA path vs CPU oracle",
                        "cuda_loss": parity_cuda, "oracle_loss": ol[0], "rel_err": err, "tol": tol, "ok": bool(err < tol)}

    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": K,
               "warmup": max(args.warmup, args.min_warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
               "config": {"workload": WORKLOAD, "arch": args.arch, "batch_per_gpu": B, "global_batch": B * world,
                          "crops": f"2x224^2 + {n_local}x96^2", "out_dim": args.out_dim, "parallelism": f"dp{world}",
                          "drop_path": drop_path,
                          "optimizer": "esvit fused clip+AdamW+EMA" if args.optimizer == "fused" else "torch AdamW fused",
                          "cuda_graph": use_graph,
                          "timed_loop": "loss.item() every step (main_esvit.py:546,596)",
                          "l2": "per-step working set (>10 GB of activations/logits) >> 126 MB L2; no explicit flush"},
               "gpu_launches": launches, "clocks": clocks, "e2e": e2e, "roofline": roofline, "roofline_others": roofline_others,
               "cpu_baseline": cpu_baseline, "parity_check": parity_check, "gpu_reference": gpu_reference,
               "step_roofline": step_roofline, "peak_mem_gib": own_mem_gib, "loss": last_loss}
        try:  # SURVEY.md 8(d) second metric; never allowed to break the contract line
            out["window_attention_core"] = attention_core_tflops(timed, n_eager) if timed else None
        except Exception as ex:  # noqa: BLE001
            out["window_attention_core"] = {"error": repr(ex)}
        print(json.dumps(out), flush=True)
    sys.stdout.flush()
    sys.stderr.flush()
    if dist.is_initialized():
        # orderly teardown: every CUDA graph that captured NCCL work was destroyed above (step._graphs.clear()) and the
        # device is idle, so the communicator can be torn down.  A watchdog hard-exits only if NCCL still fails to return.
        def _watchdog():
            time.sleep(60)
            os._exit(0)
        threading.Thread(target=_watchdog, daemon=True).start()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
