#!/usr/bin/env python
"""bench.py -- training-step throughput of the rasterizer hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input: activations -> preprocess ->
(all-to-all) -> tile binning + sort -> alpha blend -> fused L1+SSIM -> backward of all of it
(/root/reference/train_internal.py:139-196 minus optimizer / densification, SURVEY.md 8d).
Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement" for the definition of every key.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "grendel-gs_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = "train-step Gaussians/s (preprocess+forward+loss+backward)"
UNIT = "Gaussians/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", help="c2 = 2M Gaussians @1920x1080 (BASELINE.json configs[1])")
    ap.add_argument("--n", type=int, default=0, help="override Gaussian count")
    ap.add_argument("--views", type=int, default=0, help="cameras per step (bsz); default = --gpus (one view per GPU, weak "
                    "scaling); fewer views than GPUs shards every render into tile-row strips over several GPUs")
    ap.add_argument("--no-extra", action="store_true", help="skip the untimed extras at N > 1 (strong-scaling leg, parity)")
    ap.add_argument("--cpu-sample", type=int, default=250_000, help="Gaussians in the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--time-optimizer", action="store_true",
                    help="also time the fused Adam step (gs_adam_step) on the rank's parameters, reported separately under "
                         "'optimizer' (the headline metric excludes the optimizer, SURVEY.md 8d)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy: the loss, the "
                         "gradients of the six parameters, the screen-space gradient and the radii of a fixed, seeded "
                         "sample of Gaussians (compare two builds output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def workload(args):
    from gs_b200 import synthetic as syn
    cfg = dict(syn.CONFIGS[args.workload])
    if args.n:
        cfg["n"] = args.n
    return cfg


# ---------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks DURING the timed region")
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.nvml, self.samples, self._stop = None, [], False

    def _nvml_loop(self):
        n = self.nvml
        h = n.nvmlDeviceGetHandleByIndex(self.gpu)
        smax = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        while not self._stop:
            try:
                try:
                    reasons = n.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    reasons = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM), smax, reasons))
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        # In-process NVML polling: spawning nvidia-smi inside the timed region stalls the driver for ~100 ms on an
        # 8-GPU box (measured: 18.0 vs 5.6 ms/step), which would be charged to the step.
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            threading.Thread(target=self._nvml_loop, daemon=True).start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self._stop = True
            time.sleep(0.03)
            bits = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
            reasons = sorted({name for _, _, r in self.samples for b, name in bits.items() if r & b})
            sm = [s[0] for s in self.samples]
            return {"sm_mhz": float(np.median(sm)) if sm else None,
                    "sm_max_mhz": float(self.samples[0][1]) if self.samples else None, "reasons": reasons,
                    "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); smax.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        med = float(np.median(sm)) if sm else None
        return {"sm_mhz": med, "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the oracle (kind "port": the reference has no CPU path and its CUDA source is absent)
# ---------------------------------------------------------------------------------------------------
def cpu_arm(cfg, sample_n, steps, warmup):
    from gs_b200 import synthetic as syn
    from oracle.oracle import Oracle
    cores = os.cpu_count() or 1
    o = Oracle(np.float32, threads=cores)
    W, H = cfg["width"], cfg["height"]
    n = min(sample_n, cfg["n"])
    cam = syn.make_camera(W, H)
    sc = syn.make_scene(n, W, H, seed=0)
    gt = syn.make_gt_image(W, H)
    for _ in range(warmup):
        out = o.train_step(sc, cam, gt)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        o.train_step(sc, cam, gt)
        ts.append(time.perf_counter() - t0)
    dt = float(np.median(ts))
    V, R = int((out["pre"]["radii"] > 0).sum()), int(out["fwd"]["R"])
    return dict(value=n / dt, unit=UNIT, cores=cores, kind="port", ms_per_step=dt * 1e3, steps=steps, warmup=warmup,
                ms_min=min(ts) * 1e3, ms_max=max(ts) * 1e3, visible=V, instances_R=R,
                sample=f"{n} of {cfg['n']} Gaussians (seed 0, same distribution; realised V = {V}, R = {R}) on the full "
                       f"{W}x{H} view, forward+loss+backward, oracle/gs_oracle.c with OpenMP on {cores} threads, "
                       f"median of {steps} steps after {warmup} warm-ups")


def run_reference(args):
    """--impl reference: the CPU implementation of the path timed on the host cores.  The reference ships no
    CPU path and its CUDA rasterizer source is an absent submodule (SURVEY.md F1/F3), so this arm is the
    oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = workload(args)
    steps, warmup = args.steps, 2
    r = cpu_arm(cfg, args.cpu_sample, steps, warmup)
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {cfg['n']} Gaussians @ {cfg['width']}x{cfg['height']}, bounded CPU sample"},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "ms_min", "ms_max", "visible",
                                               "instances_R")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def alg_bytes(N, V, Vp, R, P, T):
    """Algorithmic (compulsory) bytes per stage, SURVEY.md section 8(d)."""
    return {"10 preprocess": 16 * N + 292 * V, "binning": 44 * Vp + 44 * R + 8 * T, "70 render": 40 * R + 20 * P,
            "loss": 27 * P, "b10 render": 76 * R + 20 * P, "b20 preprocess": 304 * V + 236 * N}


def build_trainer(args, cfg, B, dev, rank, world, **kw):
    """Trainer over B cameras of the workload.  Scenes that fit comfortably on the host (c1, c2) are generated whole on
    every rank and sliced (the round-1 scene, bit for bit); larger ones (c3, c4) shard-wise, each rank only its own
    Gaussians (synthetic.make_scene_shard)."""
    import torch
    from gs_b200 import pipeline, synthetic as syn
    W, H, N = cfg["width"], cfg["height"], cfg["n"]
    cams = syn.make_batch_cameras(W, H, B)
    gts = [torch.from_numpy(syn.make_gt_image(W, H, seed=1 + k)).pin_memory() for k in range(B)]
    if N <= 4_000_000:
        scene = syn.make_scene(N, W, H, seed=0)
        return pipeline.Trainer(scene, cams, gts, dev, rank, world, **kw)
    lo, hi = N * rank // world, N * (rank + 1) // world
    scene = syn.make_scene_shard(N, lo, hi, W, H, seed=0)
    return pipeline.Trainer(scene, cams, gts, dev, rank, world, shard=(lo, hi, N), **kw)


def timed_steps(trainer, steps, resident, barrier_sync):
    """EXACTLY `steps` steps between a barrier + synchronise on both sides; one CUDA event per step boundary.
    -> (total ms on this rank, per-step ms list, last return value of step())."""
    import torch
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    barrier_sync()
    evs[0].record()
    out = None
    for i in range(steps):
        out = trainer.step(resident=resident)
        evs[i + 1].record()
    barrier_sync()
    per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
    return evs[0].elapsed_time(evs[steps]), per, out


def dump_outputs(trainer, loss, out_dir, n_total, rank, world, dev):
    """Writes what the last step of `trainer` computed, as a caller of Trainer.step receives it, to out_dir/<name>.npy:
    the loss, the gradients of the six raw parameters, and per view the screen-space gradient (means2D.grad, which
    densification reads) and the radii, all of one fixed, seeded sample of the Gaussians.  Each rank contributes the
    sampled rows of its contiguous shard and rank 0 writes them in order, so the files have the same rows and layout for
    any number of GPUs.  The sample keeps the files under 64 MB."""
    import torch
    import torch.distributed as dist
    p = trainer.params
    B = len(trainer.dcams)
    rows = min(n_total, 1 << 16, (60 << 20) // (4 * (59 + 3 * B)))   # 59 parameter floats per Gaussian, 3 per view
    sample = np.sort(np.random.default_rng(0).choice(n_total, size=rows, replace=False))
    lo = n_total * rank // world
    local = torch.from_numpy(sample[(sample >= lo) & (sample < lo + trainer.n_local)] - lo).to(dev)
    m2 = trainer.means2D
    m2_grad = torch.stack([t.grad for t in m2]) if isinstance(m2, list) else m2.grad
    part = {f"grad{name}": getattr(p, name).grad[local] for name in
            ("_xyz", "_features_dc", "_features_rest", "_scaling", "_rotation", "_opacity")}
    part["grad_means2D"] = m2_grad[:, local]
    part["radii"] = trainer._radii_local[:, local].float()
    part = {k: v.float().cpu().numpy() for k, v in part.items()}
    total = torch.tensor([loss], dtype=torch.float64, device=dev)
    parts = [part]
    if world > 1:
        dist.all_reduce(total)                     # every rank's loss covers its own strips
        parts = [None] * world
        dist.all_gather_object(parts, part)
    if rank != 0:
        return
    out = {k: np.concatenate([q[k] for q in parts], axis=1 if k in ("grad_means2D", "radii") else 0) for k in part}
    out["loss"] = np.array(float(total.item()), np.float64)
    out["sample_rows"] = sample.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from gs_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the hot path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    # A/B of kernel variants (include/grendel_gs_b200.h, gs_debug_set): GS_B200_DEBUG_FLAGS=2 python bench.py;
    # a run with flags set is labelled in config.debug_flags and is NOT the shipped configuration
    debug_flags = int(os.environ.get("GS_B200_DEBUG_FLAGS", "0"))
    if debug_flags:
        _lib.debug_set(debug_flags)

    cfg = workload(args)
    W, H, N = cfg["width"], cfg["height"], cfg["n"]
    # default: one view per GPU per step -- weak scaling in views, Gaussians sharded (README.md:344 "4 GPU bsz 4");
    # --views B < GPUs shards every render into tile-row strips over several GPUs (the strong-scaling direction)
    B = args.views or world
    P_pix, T = W * H, ((W + 15) // 16) * ((H + 15) // 16)
    steps, warmup = args.steps, max(3, args.warmup)
    trainer = build_trainer(args, cfg, B, dev, rank, world)

    def barrier_sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- leg 1: inputs resident in HBM --------------------------------------------------------
    for _ in range(warmup):
        trainer.step(resident=True)
    barrier_sync()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    _lib.profile_enable(True)
    ms, per_step, _ = timed_steps(trainer, steps, True, barrier_sync)
    stages = _lib.profile_read()
    _lib.profile_enable(False)
    clocks = sampler.stop() if rank == 0 else None
    ms_step = max_over_ranks(ms) / steps
    info = trainer.last_info()  # realised V, V', R on this rank
    tot = torch.tensor([info["V"], info["Vp"], info["R"], info["P_local"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot)   # the step of ALL ranks: sums over the job
    job = dict(V=int(tot[0]), Vp=int(tot[1]), R=int(tot[2]), P=int(tot[3]))

    # ---- leg 2: end to end through the public operator with HOST buffers ------------------------
    for _ in range(2):
        trainer.step(resident=False)
    ms2, per_step_e2e, loss_host = timed_steps(trainer, steps, False, barrier_sync)
    ms_e2e = max_over_ranks(ms2) / steps
    h2d, d2h = trainer.io_bytes_per_step()
    if args.dump_outputs:   # before anything below runs another step or moves the parameters
        dump_outputs(trainer, loss_host, args.dump_outputs, N, rank, world, dev)

    # ---- optional: the fused Adam step on this rank's six parameter tensors, after both timed regions ------------
    optimizer = None
    if args.time_optimizer:
        from gs_b200.optim import FusedAdam
        p = trainer.params
        lrs = {"_xyz": 0.00016, "_features_dc": 0.0025, "_features_rest": 0.0025 / 20, "_opacity": 0.05, "_scaling": 0.005,
               "_rotation": 0.001}            # arguments/__init__.py:110-119
        opt = FusedAdam([{"params": [getattr(p, k)], "lr": v, "name": k} for k, v in lrs.items()], lr=0.0, eps=1e-15)
        trainer.step(resident=True)           # leaves gradients in place
        for _ in range(3):
            opt.step(grad_scale=1.0 / B)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a0.record()
        n_opt = 20
        for _ in range(n_opt):
            opt.step(grad_scale=1.0 / B)
        a1.record()
        torch.cuda.synchronize()
        adam_ms = a0.elapsed_time(a1) / n_opt
        elems = sum(t.numel() for t in p.raw_parameters())
        optimizer = {"kernel": "k_adam (gs_adam_step)", "ms_per_step": adam_ms, "elements": elems,
                     "alg_bytes": 28 * elems, "achieved_gbs": 28 * elems / (adam_ms * 1e-3) / 1e9,
                     "note": "one launch for the six parameter tensors incl. the 1/bsz gradient scaling; not part of value/e2e"}

    # ---- diagnostics, OUTSIDE both timed regions: wall clock per phase with a device synchronise after each phase
    # (serialises host and device, so the phases add up to more than ms_per_step; max over ranks) ----------------
    phase_ms = None
    if world > 1:
        os.environ["GS_B200_TRACE"] = "1"
        trainer.trace = {}
        n_tr = 5
        for _ in range(n_tr):
            trainer.step(resident=True)
        del os.environ["GS_B200_TRACE"]
        keys = sorted(trainer.trace)
        tt = torch.tensor([trainer.trace[k] / n_tr for k in keys], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        phase_ms = {k: round(float(v), 4) for k, v in zip(keys, tt.tolist())}
    exchange_kind = None
    if world > 1:
        from gs_b200 import exchange as _ex
        if trainer._peer is None:
            exchange_kind = "NCCL all_to_all_single"
        elif _ex.MODE == "direct":
            exchange_kind = ("direct placement over NVLink peer memory: k_xr_pack stores every field into its final row of the "
                             "destination's SoA receive region, the backward pulls gradient rows (gs_xr_*)")
        else:
            exchange_kind = "NVLink peer-memory stores fused into the row pack kernels (gs_xchg_pack_p2p)"
    balance_log = list(trainer.balance_log)

    # ---- extras at N > 1, OUTSIDE the timed regions: (a) the strong-scaling direction the headline does not exercise
    # (ONE view cut into N strips; N/2 views over N GPUs), (b) multi-GPU parity on a small scene against the CPU oracle
    extra, parity = None, None
    if world > 1 and not args.no_extra:
        extra = {}
        del trainer
        torch.cuda.empty_cache()
        for name, nb in (("strong_1view", 1), (f"views_{world // 2}", world // 2)):
            if nb < 1 or nb == B or (nb > 1 and name == "strong_1view"):
                continue
            try:   # diagnostics must not cost the headline its line
                tr2 = build_trainer(args, cfg, nb, dev, rank, world)
                for _ in range(warmup + 5):   # moving strips: a few more steps until the allocator has seen every size
                    tr2.step(resident=True)
                m2, _, _ = timed_steps(tr2, max(5, steps // 2), True, barrier_sync)
                ms2v = max_over_ranks(m2) / max(5, steps // 2)
                i2 = tr2.last_info()
                t2 = torch.tensor([i2["R"], i2["Vp"]], dtype=torch.float64, device=dev)
                dist.all_reduce(t2)
                extra[name] = {"views_per_step": nb, "ms_per_step": ms2v, "gaussians_per_s": N * nb / (ms2v * 1e-3),
                               "instances_R_job": int(t2[0]), "splats_rendered_job": int(t2[1]),
                               "strips_per_view": [len(st.gpu_ids) for st in tr2._strategies],
                               "division_rows_view0": list(tr2._strategies[0].division_pos),
                               "division_moves": len(tr2.balance_log) - 1, "feedback_lag": tr2.feedback_lag}
                del tr2
            except Exception as e:   # noqa: BLE001
                extra[name] = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()
        try:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import mgpu_parity
            parity = mgpu_parity.check(dev, rank, world, verbose=False)
        except Exception as e:   # noqa: BLE001 -- a parity failure must show up in the line, not kill the numbers
            parity = {"ok": False, "error": repr(e)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ----------------------------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    # algorithmic bytes of the step of ALL ranks (every rank preprocesses its shard for all B views, renders the splats it
    # received, scores its strips) and of rank 0 alone (its kernels are the ones timed by the stage timers below)
    ab_job = alg_bytes(N * B, job["V"], job["Vp"], job["R"], job["P"], T * B)
    ab = alg_bytes(trainer_n_local(N, rank, world) * B, info["V"], info["Vp"], info["R"], info["P_local"], T * B)
    per_stage = {k: v[0] / v[1] for k, v in stages.items()}
    launches = {k: v[1] for k, v in stages.items()}
    key_of = {"10 preprocess": "10 preprocess", "70 render": "70 render", "b10 render": "b10 render",
              "b20 preprocess": "b20 preprocess"}
    dom = max(per_stage, key=per_stage.get)
    units = max(1, launches[dom] // steps)  # launches of that stage per step
    if dom in key_of:
        dom_bytes = ab[key_of[dom]] / units
    elif dom.startswith("loss"):
        dom_bytes = ab["loss"] / units / 2
    else:
        dom_bytes = ab["binning"] / units
    achieved = dom_bytes / (per_stage[dom] * 1e-3) / 1e9
    # DRAM bytes per launch and issue-slot utilisation of that kernel from the committed ncu --set full capture
    # (profiles/traffic.json; only valid for the workload it was captured on: c2 at N=1)
    traffic, secondary = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if dom in tj["stages"] and args.workload == "c2" and world == 1 and not args.n and not debug_flags:
            traffic = tj["stages"][dom]["dram_bytes_per_launch"]
            secondary = {"bound": "instruction issue", "issue_slots_busy_pct": tj["stages"][dom]["issue_active_pct"],
                         "note": "blend kernels do 256 (pixel,splat) evaluations per 40-76 B instance: issue-bound, "
                                 "HBM idle by construction (SURVEY.md 8d)", "source": tj.get("source", "profiles/")}
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "secondary_bound": secondary, "peak_source": peak_src,
                "alg_bytes_per_launch": dom_bytes, "avg_launch_ms": per_stage[dom],
                "stage_ms_per_launch": {k: round(v, 4) for k, v in per_stage.items()},
                "scope": "kernel figures: rank 0's launches; step figures: the whole job (all ranks, all views)",
                "step_alg_bytes": float(sum(ab_job.values())),
                "step_frac_of_hbm_roofline": float(sum(ab_job.values())) / (ms_step * 1e-3) / 1e9 / (peak * world)}

    value = N * B / (ms_step * 1e-3)
    spread = lambda v: {"min": round(min(v), 4), "median": round(float(np.median(v)), 4), "max": round(max(v), 4)}
    scaling = "weak" if B == world or world == 1 else "strong"
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": f"{args.workload}: {N} Gaussians (sh_degree 3) @ {W}x{H}, {B} view(s)/step, "
                                   f"Gaussians sharded {world} way(s), pixels sharded by tile rows",
                       "views_per_step": B, "views_per_s": B / (ms_step * 1e-3), "visible": job["V"],
                       "instances_R": job["R"], "splats_rendered": job["Vp"], "counts_scope": "summed over all ranks and views",
                       "l2_policy": f"inputs ({236 * N // world // 1_000_000} MB parameters per rank + binning state) exceed the 126 MB L2",
                       "loss_check": loss_host,
                       "ms_per_step_rank0": {"resident": spread(per_step), "e2e": spread(per_step_e2e),
                                             "note": "per-step CUDA-event times on rank 0 inside the timed regions"}},
            "e2e": {"value": N * B / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "gpu_launches": int(sum(v for k, v in launches.items() if k not in ("30 InclusiveSum", "50 SortPairs"))),
            "library_calls": {"cub::DeviceScan": int(launches.get("30 InclusiveSum", 0)),
                              "cub::DeviceRadixSort": int(launches.get("50 SortPairs", 0))},
            "roofline": roofline, "clocks": clocks}
    if debug_flags:
        line["config"]["debug_flags"] = debug_flags
    if optimizer is not None:
        optimizer["frac_of_hbm_peak"] = optimizer["achieved_gbs"] / peak
        line["optimizer"] = optimizer
    if phase_ms is not None:  # multi-GPU only; measured outside the timed regions (see above)
        line["phase_ms_serialised"] = phase_ms
        line["config"]["exchange"] = exchange_kind
    if len(balance_log) > 1:
        line["config"]["load_balance"] = {"division_moves": len(balance_log) - 1, "first": balance_log[0][1][0],
                                          "last": balance_log[-1][1][0], "note": "tile-row boundaries of view 0 before / after "
                                          "the timing feedback (finish_strategy_final)"}
    if extra:
        line["extra"] = extra
    if parity is not None:
        line["config"]["parity"] = parity
    if not args.no_cpu_baseline:
        r = cpu_arm(cfg, args.cpu_sample, 3, 2)
        line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "ms_min", "ms_max", "visible",
                                                  "instances_R")}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def trainer_n_local(N, rank, world):
    return N * (rank + 1) // world - N * rank // world


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
