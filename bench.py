#!/usr/bin/env python
"""bench.py -- images/sec of the k-diffusion sampling hot path on B200.

One "step" = one complete sampler call over one batch of synthetic latents per GPU on the image_transformer_v2 denoiser.
`--config` selects the BASELINE.json workload (default cfg2 = configs[1], the one the headline metric is quoted on):

    cfg2  sample_heun 50 steps (99 evaluations), 256x256 shifted-window model, batch 32 per GPU
    cfg3  sample_dpmpp_2m 25 steps, 256x256 neighbourhood-attention model, batch 64 per GPU
    cfg4  sample_euler_ancestral 50 steps + BrownianTreeNoiseSampler, 256x256 neighbourhood model, batch 32 per GPU (256 over 8)
    cfg5  sample_heun 50 steps, 512x512 hourglass depths [2,2,4] widths [256,512,1024], batch 16 per GPU (128 over 8)

    python bench.py [--config cfgN] [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # N>1: launched by torch.distributed.run
    python bench.py --impl reference ...                                  # the reference algorithm's CPU port (oracle/)

Weak scaling: every rank samples its own batch.  Prints ONE JSON line on rank 0 (contract: task statement / DESIGN.md section 6).
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for p in (str(ROOT), str(ROOT / "k-diffusion_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch

UNIT = "images/s"
SIGMA_MIN, SIGMA_MAX = 1e-2, 160.0
DUMP_LIMIT_BYTES = 64 * 10**6
_NA_RAW = {"model": {"type": "image_transformer_v2", "input_channels": 3, "input_size": [256, 256], "patch_size": [4, 4],
                     "depths": [2, 2, 4], "widths": [128, 256, 512], "loss_config": "karras", "loss_weighting": "soft-min-snr",
                     "dropout_rate": [0.0, 0.0, 0.1], "augment_prob": 0.0, "sigma_data": 0.5, "sigma_min": 1e-2, "sigma_max": 160,
                     "sigma_sample_density": {"type": "cosine-interpolated"}}}      # reference configs/config_oxford_flowers.json
CONFIGS = {
    "cfg2": dict(fixture="cfg2_sw256_shapes.json", sampler="heun", steps=50, res=256, batch=32,
                 metric="images/sec (256x256, Heun 50-step)",
                 what="image_transformer_v2 256x256 (oxford_flowers shifted-window config)"),
    "cfg3": dict(raw=_NA_RAW, sampler="dpmpp_2m", steps=25, res=256, batch=64,
                 metric="images/sec (256x256, DPM++(2M) 25-step, neighborhood attention)",
                 what="image_transformer_v2 256x256 (oxford_flowers config: 7x7 neighborhood attention x2 levels + global)"),
    "cfg4": dict(raw=_NA_RAW, sampler="euler_ancestral", steps=50, res=256, batch=32,
                 metric="images/sec (256x256, Euler-ancestral 50-step + BrownianTree, neighborhood attention)",
                 what="image_transformer_v2 256x256 (oxford_flowers config, neighborhood attention), BrownianTreeNoiseSampler with one seed per image"),
    "cfg5": dict(raw={"model": dict(_NA_RAW["model"], input_size=[512, 512], widths=[256, 512, 1024], depths=[2, 2, 4],
                                    dropout_rate=[0.0, 0.0, 0.0])},
                 sampler="heun", steps=50, res=512, batch=16, metric="images/sec (512x512, Heun 50-step, widths 256/512/1024)",
                 what="image_transformer_v2 512x512 hourglass depths [2,2,4] widths [256,512,1024] (neighborhood x2 + global, S=1024)"),
}
SAMPLER_NAME = {"heun": "sample_heun", "dpmpp_2m": "sample_dpmpp_2m", "euler_ancestral": "sample_euler_ancestral"}


def nfe_of(sampler, steps):
    return 2 * steps - 1 if sampler == "heun" else steps


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed sampler calls (default 5; 3 for cfg5)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default: the BASELINE config's)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-extras", action="store_true", help="skip the roofline, parity and cpu_baseline legs")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--parity-seconds", type=float, default=25.0, help="CPU budget of the parity leg (oracle run of one image)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the images the last timed step sampled (all ranks, float32) to DIR/samples.npy; beyond "
                         f"{DUMP_LIMIT_BYTES // 10**6} MB a seeded subset of whole images, their indices in DIR/samples_index.npy")
    args = ap.parse_args()
    args.wl = CONFIGS[args.config]
    if args.batch is None:
        args.batch = args.wl["batch"]
    if args.steps is None:
        args.steps = 3 if args.config == "cfg5" else 5
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours (the reference leg times shortened schedules on other inputs)")
    return args


def dump_outputs(directory, samples):
    """samples [N, C, H, W] on the host -> DIR/samples.npy (float32).  The inputs are seeded, so two builds run with the same
    arguments can be compared file for file; above DUMP_LIMIT_BYTES a fixed seeded subset of whole images is kept."""
    import numpy as np
    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    samples = samples.float()
    per_image = samples[0].numel() * samples.element_size()
    if samples.shape[0] * per_image > DUMP_LIMIT_BYTES:
        keep = max(1, DUMP_LIMIT_BYTES // per_image - 1)          # leaves room for the index file
        idx = torch.randperm(samples.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        samples = samples[idx]
        np.save(out / "samples_index.npy", idx.double().numpy())
    np.save(out / "samples.npy", samples.contiguous().numpy())


def raw_model_config(wl):
    if "fixture" in wl:
        return json.loads((ROOT / "tests" / "golden" / wl["fixture"]).read_text())["config"]
    return json.loads(json.dumps(wl["raw"]))


def workload_config(args, n_gpus):
    wl, batch = args.wl, args.batch
    nfe = nfe_of(wl["sampler"], wl["steps"])
    return {"workload": f"{args.config}: {SAMPLER_NAME[wl['sampler']]} {wl['steps']} steps ({nfe} model evaluations), {wl['what']}, synthetic seeded "
                        f"weights, Karras schedule rho=7 sigma [{SIGMA_MIN}, {SIGMA_MAX}], batch {batch} per GPU",
            "baseline_config": args.config, "sampler": wl["sampler"], "sampler_steps": wl["steps"], "nfe_per_image": nfe, "resolution": wl["res"],
            "per_gpu_batch": batch, "global_batch": batch * n_gpus, "parallelism": f"dp{n_gpus} (batch shards, no per-step collective)",
            "l2": "256 MiB buffer rewritten between timed steps; per-step activation working set also exceeds the 126 MB L2"}


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)          # the poller must not outlive a bench that fails before stop()
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "nvidia-smi unavailable"}
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for ts, line in self.lines:
            if not (t0 <= ts <= t1 + 0.3):
                continue
            f = [v.strip() for v in line.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(self.NAMES, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU legs (the ONLY place bench.py touches oracle/)
# ------------------------------------------------------------------------------------------------
def oracle_model(wl, inner=None):
    """(oracle module, oracle denoiser) with the synthetic weights of seed 1 (the recipe depends on key/shape/seed only)."""
    import k_diffusion as K
    from oracle import kdiff_oracle as O
    from oracle.fixtures import synth_sd
    cfg = K.config.load_config(raw_model_config(wl))
    if inner is None:
        inner = K.config.make_model(cfg)
    sd = synth_sd({k: list(v.shape) for k, v in inner.state_dict().items()}, 1)
    return O, O.make_denoiser(sd, cfg["model"])


def oracle_sample(O, model, wl, x, sigmas, seeds=None):
    if wl["sampler"] == "heun":
        return O.sample_heun(model, x, sigmas)
    if wl["sampler"] == "dpmpp_2m":
        return O.sample_dpmpp_2m(model, x, sigmas)
    g = torch.Generator().manual_seed(7)          # timing only: any unit-normal stream costs the same
    return O.sample_euler_ancestral(model, x, sigmas, noise_sampler=lambda a, b: torch.randn(x.shape, generator=g))


def cpu_port_setup(wl):
    O, model = oracle_model(wl)
    # pick the torch thread count that is actually fastest on this host (all-cores oversubscribes cgroup-limited boxes)
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    x = torch.randn(1, 3, wl["res"], wl["res"])
    best, cores = None, 1
    for n in sorted({c for c in (8, 16, 32, 64, avail) if c <= avail}):
        torch.set_num_threads(n)
        model(x, torch.ones(1))
        t0 = time.perf_counter()
        model(x, torch.ones(1))
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, cores = dt, n
    torch.set_num_threads(cores)
    return O, model, cores, best


def cpu_port_time(O, model, wl, batch, budget_s, t_fwd):
    """Time the oracle's sampler on `batch` images with as many Karras steps as fit the budget; scale to the full NFE."""
    res, full_nfe = wl["res"], nfe_of(wl["sampler"], wl["steps"])
    g = torch.Generator().manual_seed(123)
    x = torch.randn(batch, 3, res, res, generator=g) * SIGMA_MAX
    per_step = 2 if wl["sampler"] == "heun" else 1
    steps = max(2, min(wl["steps"], int((budget_s / max(t_fwd * batch, 1e-3) + (1 if per_step == 2 else 0)) // per_step)))
    sigmas = O.get_sigmas_karras(steps, SIGMA_MIN, SIGMA_MAX)
    t0 = time.perf_counter()
    oracle_sample(O, model, wl, x, sigmas)
    dt = time.perf_counter() - t0
    nfe = nfe_of(wl["sampler"], steps)
    ips = batch / (dt * full_nfe / nfe)
    how = "the full schedule, nothing extrapolated" if nfe == full_nfe else "images/s EXTRAPOLATED by the NFE ratio"
    return ips, (f"{batch} image(s) x {nfe} of {full_nfe} model evaluations ({SAMPLER_NAME[wl['sampler']]} {steps} of {wl['steps']} Karras steps) "
                 f"in {dt:.1f} s, {how}")


def cpu_sample_batch(wl, budget_s, t_fwd):
    """Images in the cpu_baseline sample: as many full schedules as fit the budget (1..8), so a fast host still does ~10 s of work."""
    return max(1, min(8, int(budget_s / max(t_fwd * nfe_of(wl["sampler"], wl["steps"]), 1e-3))))


def run_reference(args, rank, world):
    if rank != 0:
        return
    wl = args.wl
    O, model, cores, t_fwd = cpu_port_setup(wl)
    total_budget = 170.0
    per = total_budget / max(1, args.steps + args.warmup)
    vals, sample = [], ""
    for i in range(args.warmup + args.steps):
        ips, sample = cpu_port_time(O, model, wl, cpu_sample_batch(wl, per, t_fwd), per, t_fwd)
        if i >= args.warmup:
            vals.append(ips)
    v = len(vals) / sum(1.0 / a for a in vals)
    line = {"metric": wl["metric"], "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * args.batch / v, "ms_per_step_note": "EXTRAPOLATED: each timed step is a bounded sample of the workload (cpu_baseline.sample: "
            "as many images with the full schedule as fit the step's time budget, else one image with a shortened schedule scaled by the NFE ratio); "
            "ms_per_step = batch / images/s -- the full batch was not run on the CPU",
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp32", "data": "synthetic", "impl": "reference", "config": workload_config(args, args.gpus),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "per step: " + sample + "; CPU torch fp32 port of the reference algorithm (oracle/kdiff_oracle.py); "
                                       "the reference itself is Python and /root/reference does not travel to the GPU box"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# per-kernel device times of the graph-replayed step (CUPTI activity records through torch.profiler)
# ------------------------------------------------------------------------------------------------
def kernel_family(name):
    """Kernel name (as CUPTI reports it) -> the family names of kdb_launch_breakdown."""
    name = name.replace("(int)", "").replace(" ", "")
    if "gemm_tc_kernel<64,5>" in name:
        return "patch_out"
    for key, fam in (("ffn_fused", "gemm_tc"), ("gemm_tc", "gemm_tc"), ("gemm_simt", "gemm_simt"), ("attn_", "attn_tc"), ("patch_in", "patch_in"), ("patch_out", "patch_out"),
                     ("fold_norm", "fused_norm"), ("ew_kernel", "solver"), ("precond", "precond"), ("noise_", "noise"),
                     ("conditioning", "cond"), ("rmsnorm", "rmsnorm"), ("qknorm", "qknorm_rope"), ("geglu_kernel", "geglu")):
        if key in name:
            return fam
    return "other (torch copies)"


def graph_kernel_times(fn):
    """[(family, kernel name, start_us, duration_ms)] of every kernel `fn()` executes, in start order, from CUPTI activity records.
    Unlike CUDA events between eager launches this times the kernels INSIDE the replayed CUDA graph: no event, no host launch gap,
    programmatic-launch overlap as in the timed step.  Returns None when the profiler is unavailable."""
    try:
        from torch.autograd import DeviceType
        from torch.profiler import ProfilerActivity, profile
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        out = []
        for e in prof.events():
            if e.device_type != DeviceType.CUDA:
                continue
            name = e.name
            if name.startswith("Memcpy") or name.startswith("Memset") or name.startswith("cudaGraph"):
                continue
            out.append((kernel_family(name), name, float(e.time_range.start), float(e.time_range.elapsed_us()) / 1000.0))
        out.sort(key=lambda r: r[2])
        # Under programmatic dependent launch a kernel is resident (prologue, then parked in griddepcontrol.wait) while its
        # predecessor still runs, and CUPTI's duration includes that wait: the raw durations of one evaluation summed to 2.11 ms
        # against a 1.69 ms span (profiles/r2_bench_cfg2_first.json).  Attribute to each kernel only the time after the previous
        # kernel ENDED (one stream, in-order completion): the exclusive durations sum to the span exactly.
        excl, prev_end = [], None
        for fam, name, start, dur in out:
            end = start + dur * 1000.0
            lo = start if prev_end is None else max(start, min(prev_end, end))
            excl.append((fam, name, start, (end - lo) / 1000.0))
            prev_end = end if prev_end is None else max(prev_end, end)
        return excl or None
    except Exception as exc:          # measurement aid only
        print(f"bench: torch.profiler unavailable ({exc!r}); falling back to CUDA events between eager launches", file=sys.stderr)
        return None


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank, local, world = int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            sys.exit(f"--gpus {args.gpus} needs `python -m torch.distributed.run --nproc-per-node {args.gpus} bench.py ...`")
        args.gpus = world
    import torch.distributed as dist

    import k_diffusion as K
    from k_diffusion import _native
    S = K.sampling
    wl = args.wl
    RES, NFE = wl["res"], nfe_of(wl["sampler"], wl["steps"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg = K.config.load_config(raw_model_config(wl))
    inner = K.config.make_model(cfg)
    if rank == 0:
        K.synth.synth_init_(inner, seed=1)
    inner = inner.to(dev).eval().set_precision(args.precision)
    bcast_bytes = K.parallel.broadcast_weights(inner, src=0)          # the single collective: weights at init
    model = K.config.make_denoiser_wrapper(cfg)(inner)
    B = args.batch
    lo, hi = K.parallel.shard_range(B * world, rank, world)
    seeds = K.parallel.sample_seeds(123, lo, hi)
    x = K.parallel.init_noise(seeds, (3, RES, RES), SIGMA_MAX, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run_sampler(xin, steps=None, x_seeds=seeds):
        sig = S.get_sigmas_karras(wl["steps"] if steps is None else steps, SIGMA_MIN, SIGMA_MAX, device=dev)
        if wl["sampler"] == "heun":
            return S.sample_heun(model, xin, sig, disable=True)
        if wl["sampler"] == "dpmpp_2m":
            return S.sample_dpmpp_2m(model, xin, sig, disable=True)
        ns = S.BrownianTreeNoiseSampler(xin, SIGMA_MIN, SIGMA_MAX, seed=list(x_seeds))      # cfg4: one Brownian path per image
        return S.sample_euler_ancestral(model, xin, sig, disable=True, noise_sampler=ns)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step_device(_):
        flush.zero_()
        return run_sampler(x)

    x_host = x.cpu().pin_memory()
    out_host = torch.empty_like(x_host).pin_memory()

    def step_e2e(_):
        flush.zero_()
        xd = x_host.to(dev, non_blocking=True)                        # H2D of this step's inputs (pinned)
        out = run_sampler(xd)                                         # public API call
        out_host.copy_(out, non_blocking=True)                        # D2H of this step's result
        return out

    def timed(fn, k, w):
        for i in range(w):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = S.total_kernel_launches()
        t0 = time.time()
        e0.record()
        for i in range(k):
            last = fn(i)
        e1.record()
        barrier()
        t1 = time.time()
        return max_over_ranks(e0.elapsed_time(e1)), S.total_kernel_launches() - n0, t0, t1, last

    clocks = ClockSampler(local) if rank == 0 else None
    time.sleep(0.3)
    ms, launches, t0, t1, last = timed(step_device, args.steps, args.warmup)
    clk = clocks.stop(t0, t1) if clocks else None
    dumped = K.parallel.gather_samples(last).cpu() if args.dump_outputs else None
    del last
    ms_e2e, _, _, _, _ = timed(step_e2e, args.steps, 1)
    out = step_device(0)
    finite = bool(torch.isfinite(out).all())
    value = world * B * args.steps / (ms / 1000.0)
    e2e = world * B * args.steps / (ms_e2e / 1000.0)

    roofline = cpu_baseline = breakdown = parity = None
    if rank == 0 and not args.no_extras:
        # --- per-kernel device times.  Preferred: CUPTI activity records of ONE replay of the very graph that was timed (no events,
        # no host gaps, programmatic-launch overlap included).  Fallback: CUDA events after every eager launch of a shorter schedule
        # behind a gate kernel (kdb_profile_gate), which adds ~8 us of event / serialisation overhead per launch.
        class _P:
            pass
        prof = _P()
        recs = graph_kernel_times(lambda: run_sampler(x))
        if recs is not None:
            prof.launches = [(fam, ms_) for fam, _, _, ms_ in recs]
            prof_evals, prof_how = NFE, ("CUPTI activity records (torch.profiler) of one replay of the timed CUDA graph, no events between kernels, "
                                         "no host launch gaps; each kernel is charged the time from the END of its predecessor to its own end "
                                         "(programmatic launch makes kernels resident early, so raw durations overlap and over-count)")
            span_ms = (recs[-1][2] + recs[-1][3] * 1000.0 - recs[0][2]) / 1000.0
        else:
            prof_steps = 5 if wl["sampler"] == "heun" else 9
            os.environ["KDB200_CUDA_GRAPH"] = "0"
            run_sampler(x, prof_steps)
            torch.cuda.synchronize()
            with _native.profile(gate_ms=40.0 if RES <= 256 else 120.0) as prof:
                run_sampler(x, prof_steps)
            os.environ["KDB200_CUDA_GRAPH"] = "1"
            prof_evals = nfe_of(wl["sampler"], prof_steps)
            prof_how = (f"CUDA events after every launch of one eager {SAMPLER_NAME[wl['sampler']]} with {prof_steps} Karras steps behind a gate kernel "
                        "(each interval carries ~8 us of event / serialisation overhead)")
            span_ms = None
        prof.by_family = {}
        for f_, t_ in prof.launches:
            c_, tot_ = prof.by_family.get(f_, (0, 0.0))
            prof.by_family[f_] = (c_ + 1, tot_ + t_)
        total = sum(t for _, t in prof.by_family.values())
        breakdown = {f: {"launches": c, "ms": round(t, 3), "share": round(t / total, 4)} for f, (c, t) in
                     sorted(prof.by_family.items(), key=lambda kv: -kv[1][1])}
        # dominant kernel = the tcgen05 GEMM behind every nn.Linear on the token stream (94 % of the model's MACs).
        # Launches are matched to shapes by execution order (k_diffusion.models.flops.linear_layers).
        gemm_fams = [f for f in prof.by_family if f.startswith("gemm")]
        g_times = [t for f, t in prof.launches if f.startswith("gemm")]
        fused_ffn = os.environ.get("KDB200_NO_FFN_FUSE", "0") != "1"
        seq = K.models.flops.launch_layers(cfg["model"], B, fused_ffn)
        per_shape, per_level = {}, {}
        for idx, t in enumerate(g_times):
            label, M_, N_, K_, macs_ = seq[idx % len(seq)]
            key = (label.split(" ", 1)[-1] if " " in label else label.rstrip("0123456789"), M_, N_, K_, macs_)
            c, tot = per_shape.get(key, (0, 0.0))
            per_shape[key] = (c + 1, tot + t)
            lvl = label[:2] if label.startswith("L") else ("mid" if label.startswith("mid") else "merge/split")
            fl, tt = per_level.get(lvl, (0.0, 0.0))
            per_level[lvl] = (fl + 2.0 * macs_, tt + t)
        g_launch, g_ms = len(g_times), sum(g_times)
        flops = 2.0 * K.models.flops.linear_macs(cfg["model"], B) * (len(g_times) / len(seq))
        peaks_file = ROOT / "MEASURED_PEAKS.json"
        if peaks_file.exists():
            peak, which = json.loads(peaks_file.read_text())["bf16_tflops_sustained"], "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        else:
            peak, which = 1400.0, "fallback (B200_PROFILING.md sustained 1.4 PFLOP/s)"
        ach = flops / (g_ms / 1000.0) / 1e12
        shapes = []
        for (kind, M_, N_, K_, macs_), (c, tot) in sorted(per_shape.items(), key=lambda kv: -kv[1][1])[:8]:
            tf = 2.0 * macs_ * c / (tot / 1000.0) / 1e12
            shapes.append({"op": kind, "M": M_, "N": N_, "K": K_, "launches": c, "avg_launch_us": round(1000.0 * tot / c, 2),
                           "achieved": round(tf, 1), "frac": round(tf / peak, 4), "share_of_step": round(tot / total, 4)})
        by_level = {lvl: {"achieved": round(fl / (tt / 1000.0) / 1e12, 1), "frac": round(fl / (tt / 1000.0) / 1e12 / peak, 4),
                          "gemm_ms_per_eval": round(tt / prof_evals, 4)} for lvl, (fl, tt) in sorted(per_level.items())}
        # attention kernels: algorithmic flops (q k^T and p v) per launch family
        a_times = [t for f, t in prof.launches if f.startswith("attn")]
        attn = None
        if a_times:
            a_fl = 2.0 * K.models.flops.attention_macs(cfg["model"], B) * prof_evals
            attn = {"launches": len(a_times), "ms_per_eval": round(sum(a_times) / prof_evals, 4),
                    "achieved_tflops": round(a_fl / (sum(a_times) / 1000.0) / 1e12, 1), "share_of_step": round(sum(a_times) / total, 4)}
        ncu_file = ROOT / "profiles" / "r2_ncu_full_summary.json"
        traffic, traffic_note = None, "no ncu capture committed for this build"
        if ncu_file.exists():
            try:
                first = json.loads(ncu_file.read_text())["roofline_kernel"]
                unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
                traffic = 0.0
                for key, val in first.items():          # ncu picks the unit per value: "dram__bytes_read.sum [Mbyte]", "... [Kbyte]"
                    if key.startswith("dram__bytes_read.sum [") or key.startswith("dram__bytes_write.sum ["):
                        traffic += float(val) * unit[key[key.index("[") + 1:-1]]
                traffic_note = ("dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the heaviest shape (" + first["launch"] +
                                "), from the committed ncu --set full capture profiles/r2_ncu_full_summary.json")
            except (KeyError, ValueError, StopIteration):
                pass
        roofline = {"bound": "tensor", "kernel": "gemm_tc_persist / gemm_tc_kernel (tcgen05 GEMM, all token-stream Linear layers: " +
                                                 "+".join(sorted(gemm_fams)) + ")",
                    "achieved": round(ach, 2), "peak": peak, "unit": "TFLOP/s", "frac": round(ach / peak, 4), "peak_source": which,
                    "avg_launch_us": round(1000.0 * g_ms / max(g_launch, 1), 2), "launches": g_launch,
                    "share_of_step": round(g_ms / total, 4), "traffic": traffic, "traffic_note": traffic_note, "by_shape": shapes,
                    "by_level": by_level, "attention": attn,
                    "profile_ms_per_eval": round(total / prof_evals, 4), "timed_ms_per_eval": round(ms / args.steps / NFE, 4),
                    "graph_span_ms_per_eval": None if span_ms is None else round(span_ms / prof_evals, 4),
                    "how": prof_how + "; achieved = 2 x Linear MACs of the GEMM launches (reference flops.py accounting) / their summed device time; "
                           "profile_ms_per_eval = sum of the (exclusive) kernel times per model evaluation = graph span minus idle gaps, "
                           "timed_ms_per_eval = the timed bench step / NFE"}
        # --- parity of the benchmarked path (same model object, precision, batch, graph runner) against the fp32 CPU oracle, image 0
        try:
            O, o_model = oracle_model(wl, inner)
            xs = x[:1].cpu()
            t0c = time.perf_counter()
            o_model(xs, torch.ones(1))
            t_f = time.perf_counter() - t0c
            per_step = 2 if wl["sampler"] == "heun" else 1
            p_steps = max(2, min(wl["steps"], int(args.parity_seconds / max(t_f, 1e-3) // per_step)))
            if wl["sampler"] != "euler_ancestral":
                sig_p = O.get_sigmas_karras(p_steps, SIGMA_MIN, SIGMA_MAX)
                want = oracle_sample(O, o_model, wl, xs, sig_p)
                got = run_sampler(x, p_steps)[:1].cpu()
            else:      # stochastic: feed the oracle the very noise our Brownian tree produces for image 0
                ns = S.BrownianTreeNoiseSampler(x[:1], SIGMA_MIN, SIGMA_MAX, seed=[seeds[0]])
                sig_p = O.get_sigmas_karras(p_steps, SIGMA_MIN, SIGMA_MAX)
                want = O.sample_euler_ancestral(o_model, xs, sig_p, noise_sampler=lambda a, b: ns(float(a), float(b)).cpu())
                got = run_sampler(x, p_steps)[:1].cpu()
            d = (got.double() - want.double())
            budget = None
            bfile = ROOT / "tests" / "golden" / "bf16_budget.json"
            if bfile.exists() and args.precision == "bf16":
                budget_key = "cfg5shape_sw_heun2" if args.config == "cfg5" else "cfg2_heun10"
                budget = json.loads(bfile.read_text()).get(budget_key, {}).get("rel_l2")
            parity = {"rel_l2": float(d.norm() / want.double().norm()), "max_abs": float(d.abs().max()), "ref_rms": float(want.double().pow(2).mean().sqrt()),
                      "image": 0, "sampler_steps": p_steps, "of_steps": wl["steps"], "vs": "oracle/kdiff_oracle.py fp32 on the CPU, same weights / latent / schedule",
                      "path": f"{args.precision} token stream, fused RMSNorm, CUDA-graph replay, batch {B} (image 0 compared)",
                      "reference_own_bf16_rel_l2": budget,
                      "note": "reference_own_bf16_rel_l2 = distance of the reference under torch.autocast(bf16) from its own fp32 output "
                              "(tests/golden/bf16_budget.json: cfg2 model, Heun 10 steps; for cfg5 the 512x512 / 256-512-1024 shifted-window "
                              "variant, Heun 2 steps) -- the scale of a legitimate bf16 deviation"}
        except Exception as exc:           # the parity leg must never cost the bench line
            parity = {"error": repr(exc)}
        if world == 1:
            O, cpu_model, cores, t_fwd = cpu_port_setup(wl)
            v, sample = cpu_port_time(O, cpu_model, wl, cpu_sample_batch(wl, args.cpu_seconds, t_fwd), args.cpu_seconds, t_fwd)
            cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}

    if rank == 0:
        line = {"metric": wl["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": args.precision, "data": "synthetic", "config": workload_config(args, world),
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": out_host.numel() * 4,
                        "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": launches, "clocks": clk, "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity,
                "parity_rel_l2": None if not parity else parity.get("rel_l2"),
                "kernel_breakdown": breakdown, "weights_broadcast_bytes": bcast_bytes, "output_finite": finite,
                "native_library": str(_native.LIB_PATH.relative_to(ROOT))}
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
