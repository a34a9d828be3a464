#!/usr/bin/env python3
"""Benchmark of the NR-NeRF render hot path on B200 (driver contract: see the task statement).

    python bench.py --gpus N --steps K --warmup W                  # this framework, BASELINE configs[1] per GPU
    python bench.py --impl reference --gpus N --steps K ...        # the reference's own CPU path on the host cores
    python bench.py --workload cfg4|render|sweep ...               # the other BASELINE configs (see below)
    python bench.py --steps K --warmup W --dump-outputs DIR        # + the last timed step's outputs as DIR/<name>.npy

Default workload (BASELINE.json configs[1]): one training step of configs/example_sequence.txt -- N_rand = 1024 rays per
GPU, 64 coarse + 128 fine network evaluations per ray, 8x256 MLP, ray bending on, perturb = 1, raw_noise_std = 1,
offsets / rigidity / divergence regularisers on, backward, Adam -- on synthetic rays shaped like the example sequence
(there is no dataset on the box).  Metric: rays/sec (whole job, all ranks).  Weak scaling: the per-GPU batch is fixed.
  --workload cfg4    BASELINE configs[3]: the same step at 8192 rays per rank (N_rand = 65536 over 8 GPUs)
  --workload render  BASELINE configs[2]: full-frame test-time forward 504 x 378, fixed pose, one latent per frame
  --workload sweep   BASELINE configs[4]: 1k-1M rays x {64,128,256} samples single pass, forward and forward+backward

N > 1 (one process per GPU, torchrun): rays are sharded by rows; the gradients live in ONE flat arena per rank that is summed
in place by one NCCL all-reduce per step (forward + backward replayed as a CUDA graph, collectives and Adam launched around
it).  `--reducer peer` keeps the arena in a CUDA-IPC window instead and lets the optimizer launch sum the ranks' arenas over
NVLink while applying Adam (nonrigid_nerf_b200/csrc/peer.cu): the whole iteration -- forward, backward, reduce + Adam, loss
gather -- is then ONE CUDA graph per rank.
"""
import argparse
import faulthandler
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
faulthandler.enable()      # a crash inside native code leaves a Python traceback on stderr

METRIC = "rays/sec (64c+128f samples, 8x256 MLP), example_sequence training step"
N_RAND = 1024
N_SAMPLES, N_IMPORTANCE = 64, 64
FLOP_PER_POINT = 1_016_320          # SURVEY.md 8(d): forward, per point evaluation (NeRF 984,576 + bender 31,744)
POINTS_PER_RAY = N_SAMPLES + (N_SAMPLES + N_IMPORTANCE)
ALG_BYTES_PER_RAY = 32 + 128 + 12 + 44 + 4    # SURVEY.md 8(d): rays + latent + target in, maps + loss out


def make_args():
    a = types.SimpleNamespace()
    a.chunk, a.N_samples, a.N_importance, a.N_iters = 32768, N_SAMPLES, N_IMPORTANCE, 200000
    a.offsets_loss_weight, a.divergence_loss_weight, a.rigidity_loss_weight = 60.0, 3.0, 0.0005
    a.ray_bending_latent_size = 32
    return a


def synth_batch(rs, n, n_images=86):
    """Rays like get_rays_np on the 384x512 example frames + uniform targets + (image, y, x) indices."""
    H, W, focal = 384, 512, 256.61
    img = rs.randint(0, n_images, size=n)
    y, x = rs.randint(0, H, size=n), rs.randint(0, W, size=n)
    dirs = np.stack([(x - W * 0.5) / focal, -(y - H * 0.5) / focal, -np.ones(n)], -1).astype(np.float32)
    ang = (img.astype(np.float32) / n_images - 0.5) * 0.6
    c, s = np.cos(ang), np.sin(ang)
    rays_d = np.stack([c * dirs[:, 0] + s * dirs[:, 2], dirs[:, 1], -s * dirs[:, 0] + c * dirs[:, 2]], -1).astype(np.float32)
    rays_o = np.stack([0.3 * s, np.zeros(n), 0.4 + 0.0 * s], -1).astype(np.float32)
    target = rs.uniform(0, 1, size=(n, 3)).astype(np.float32)
    idx = np.stack([img, y, x], -1).astype(np.int64)
    return rays_o, rays_d, target, idx


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"tf_burst": float(d.get("bf16_tflops", 1590.0)), "tf_sustained": float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1400.0))),
                "hbm_gbs": float(d.get("hbm_gbs", 6500.0)), "source": "measured (MEASURED_PEAKS.json: cuBLAS bf16 burst / sustained, copy bandwidth)"}
    return {"tf_burst": 1590.0, "tf_sustained": 1400.0, "hbm_gbs": 6500.0, "source": "fallback (B200_PROFILING.md figures)"}


class ClockSampler:
    def __init__(self, dev_index):
        self.path = f"/tmp/nrn_clocks_{os.getpid()}.csv"
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.f = open(self.path, "w")
            self.p = subprocess.Popen(["nvidia-smi", f"--id={dev_index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.remove(self.path)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def workload_text(n_rand):
    return (f"example_sequence training step: N_rand={n_rand}/GPU, 64c+128f, 8x256 MLP, ray bending on, perturb=1, "
            "raw_noise_std=1, offsets+rigidity+divergence regularisers, backward, Adam")


# ---------------------------------------------------------------------------------------------
# CPU arm: the reference's own code (oracle/_ref, copied by oracle/make_ref.py) or, if absent, the oracle port --
# the only place bench.py executes anything under oracle/
# ---------------------------------------------------------------------------------------------
def cpu_baseline(n_rays, steps, warmup):
    """The reference's training step on the host cores, at the thread count that serves it best: PyTorch's CPU kernels stop
    scaling on these shapes long before a 128-thread box is full (and collapse when oversubscribed), so a short calibration
    on a 256-ray slice picks among {all cores, 64, 32, 16}; the timed run is the full n_rays-ray step at that count."""
    from oracle import reference_arm as RA
    host = os.cpu_count() or 1
    cands = sorted({c for c in (host, 64, 32, 16, 8) if c <= host}, reverse=True)
    calib = {}
    for c in cands:
        calib[c] = RA.training_rate(synth_batch, 256, 1, 1, c, make_args())[0]
    threads = max(calib, key=calib.get)
    rate, sec, kind = RA.training_rate(synth_batch, n_rays, steps, warmup, threads, make_args())
    return {"value": rate, "unit": "rays/s", "cores": threads, "kind": kind, "seconds_per_step": sec, "host_cores": host,
            "calibration_rays_per_s_by_threads": {str(k): v for k, v in calib.items()},
            "sample": f"the full {n_rays}-ray training step (forward, three regularisers, backward, torch.optim.Adam), {warmup} warm-up + "
                      f"median of {steps} steps, torch.set_num_threads({threads}) = the fastest of {cands} on a 256-ray calibration step"}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    steps = max(1, min(args.steps, 8))      # ~1.5 s per 1024-ray step on the box's cores: bounded to a few minutes
    cb = cpu_baseline(args.n_rand, steps, min(args.warmup, 2))
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "rays/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": min(args.warmup, 2), "ms_per_step": cb["seconds_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text(args.n_rand),
                       "note": "the reference's training_wrapper_class.forward + backward + torch.optim.Adam on the host CPU cores "
                               "(unmodified sources from oracle/_ref when present, else the oracle port); the CPU arm does not shard: "
                               "one N_rand-ray step regardless of --gpus"},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "host_cores", "calibration_rays_per_s_by_threads") if k in cb},
            "e2e": {"value": cb["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
def build_models(dev, H):
    """Models exactly as create_nerf builds them (train.py:556-721), default inits, bender output layers re-drawn."""
    torch.manual_seed(0)
    embed_fn, input_ch = H.get_embedder(10, 0)
    bender = H.ray_bending(input_ch, 32, "simple_neural", embed_fn).to(dev)
    with torch.no_grad():
        bender.network[-1].weight.normal_(0, 0.01)
        bender.rigidity_network[-1].weight.normal_(0, 0.1)
    kw = dict(D=8, W=256, input_ch=input_ch, output_ch=5, skips=[4], input_ch_views=0, use_viewdirs=False, ray_bender=bender,
              ray_bending_latent_size=32)
    coarse = H.NeRF(num_ray_samples=N_SAMPLES, **kw).to(dev)
    fine = H.NeRF(num_ray_samples=N_SAMPLES + N_IMPORTANCE, **kw).to(dev)
    return coarse, fine, bender


def roofline_block(per_step, n_rand, peaks, traffic):
    """SURVEY.md 8(d): the fused passes are dense contractions -> tensor-core roofline on algorithmic FLOPs
    (1,016,320 per point evaluation, forward; DGRAD and WGRAD each the same).  Peak = sustained cuBLAS bf16 (the kernels are
    timed inside a long step); the burst fraction and the HBM view are given next to it."""
    flops = n_rand * POINTS_PER_RAY * FLOP_PER_POINT
    kinds = {}
    for k in ("field_fwd", "field_dgrad", "wgrad"):
        ms = per_step.get(k, 0.0)
        if ms > 0:
            tf = flops / (ms * 1e-3) / 1e12
            kinds[k] = {"ms_per_step": ms, "tflops": tf, "frac_sustained": tf / peaks["tf_sustained"], "frac_burst": tf / peaks["tf_burst"]}
    dom = max(kinds, key=lambda k: kinds[k]["ms_per_step"]) if kinds else None
    roof = {"bound": "tensor", "kernel": dom, "unit": "TFLOP/s", "peak": peaks["tf_sustained"], "peak_burst": peaks["tf_burst"],
            "peak_source": peaks["source"], "per_kernel": kinds,
            "note": "algorithmic FLOPs per step of one kernel kind (coarse + fine launch) = N_rand x 192 x 1,016,320"}
    if dom:
        roof["achieved"], roof["frac"] = kinds[dom]["tflops"], kinds[dom]["frac_sustained"]
        roof["frac_burst"] = kinds[dom]["frac_burst"]
        tb = (traffic or {}).get(dom)
        roof["traffic"] = tb
        alg_bytes = n_rand * ALG_BYTES_PER_RAY + 13.0e6     # rays in / maps out + one pass over weights and gradients
        roof["hbm_view"] = {"peak_gbs": peaks["hbm_gbs"], "algorithmic_bytes_per_step": alg_bytes,
                            "dram_bytes_per_step": tb, "traffic_over_algorithmic": (tb / alg_bytes) if tb else None,
                            "dram_gbs": (tb / (kinds[dom]["ms_per_step"] * 1e-3) / 1e9) if tb else None,
                            "note": "the activation / gradient stash between forward, DGRAD and WGRAD is design traffic, not algorithmic"}
    return roof


def read_traffic():
    for name in ("r02_traffic.json", "r01_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            with open(p) as f:
                d = json.load(f)
            d["_source"] = "profiles/" + name
            return d
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="train", choices=["train", "cfg4", "render", "sweep"])
    ap.add_argument("--n-rand", type=int, default=None, help="rays per GPU per step (train: 1024, cfg4: 8192)")
    ap.add_argument("--reducer", default="nccl", choices=["peer", "nccl"],
                    help="multi-GPU gradient reduction: nccl = in-place all-reduce over the gradient arena (default: the path exercised at every "
                         "N); peer = sum over NVLink peer memory fused into the Adam launch, whole step in one CUDA graph (verified at N = 2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="run the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-breakdown", action="store_true", help="skip the instrumented per-kernel pass")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (mean and per-ray loss, updated parameters, their gradients) "
                         "as DIR/<name>.npy, to compare two builds on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload in ("render", "sweep")):
        ap.error("--dump-outputs applies to this implementation's training step (--workload train or cfg4)")
    args.warmup = max(args.warmup, 3)
    if args.n_rand is None:
        args.n_rand = 8192 if args.workload == "cfg4" else N_RAND
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.workload in ("render", "sweep"):
        from scripts import bench_workloads
        bench_workloads.run(args, rank, local_rank, world)
        return

    import torch.distributed as dist
    from nonrigid_nerf_b200 import _lib, optim, parallel, run_nerf_helpers as H

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    coarse, fine, bender = build_models(dev, H)
    n_images = 86
    latents = [torch.zeros(32, device=dev).normal_(0, 0.1).requires_grad_(True) for _ in range(n_images)]
    grad_vars = latents + list(bender.parameters()) + list(coarse.parameters()) + list(fine.parameters())
    optimizer = optim.Adam(grad_vars, lr=5e-4, betas=(0.9, 0.999))   # train.py:656-658; flat parameters + gradient arena
    render_kwargs_train = {"network_query_fn": None, "perturb": 1.0, "N_importance": N_IMPORTANCE, "network_fine": fine,
                           "N_samples": N_SAMPLES, "network_fn": coarse, "ray_bender": bender, "use_viewdirs": False,
                           "white_bkgd": False, "raw_noise_std": 1.0, "ndc": False, "lindisp": False, "near": 0.0022, "far": 1.0024}
    targs = make_args()
    dataset_extras = {"imageid_to_timestepid": list(range(n_images))}
    train_fn = parallel.get_parallelized_training_function(coarse, latents, fine_model=fine, ray_bender=bender)
    local_module = train_fn.module      # training_wrapper_class: the per-rank step DataParallel used to wrap

    reducer_note = "single GPU"
    peer_red = None
    if world > 1:
        if args.reducer == "peer":
            try:
                from nonrigid_nerf_b200 import peer
                peer_red = peer.PeerArenaReducer(optimizer, slot_floats=max(1 << 16, args.n_rand))
                parallel.attach_optimizer(optimizer, peer_red)
                reducer_note = "peer memory: ranks' gradient arenas summed over NVLink inside the Adam launch (csrc/peer.cu)"
            except Exception as exc:  # noqa: BLE001 -- e.g. CUDA IPC not permitted in this container
                ok = torch.tensor([0.0], device=dev)
                print(f"[bench] peer-memory reducer unavailable on rank {rank} ({type(exc).__name__}: {exc})", file=sys.stderr)
                peer_red = None
                reducer_note = f"nccl all-reduce over the gradient arena (peer set-up failed: {type(exc).__name__})"
        if peer_red is None:
            parallel.attach_optimizer(optimizer)     # NCCL, in place over the arena
            if args.reducer == "nccl":
                reducer_note = "nccl all-reduce, in place over the gradient arena"

    n_global = args.n_rand * world
    lo, hi = parallel.shard_bounds(n_global, world, rank)
    rs = np.random.RandomState(1234)     # identical on every rank: every rank knows the global batch and uploads ITS row block
    pool = 8
    host = [synth_batch(rs, n_global, n_images) for _ in range(pool)]
    pinned = [[torch.from_numpy(np.ascontiguousarray(a[lo:hi])).pin_memory() for a in b] for b in host]
    h2d_bytes = int(sum(t.numel() * t.element_size() for t in pinned[0]))

    def upload(batch):
        return [t.to(dev, non_blocking=True) for t in batch]

    resident = [upload(b) for b in pinned]
    global_step = torch.full((), 1000.0, dtype=torch.float32, device=dev)   # device scalar: the graph follows the schedule
    fused_collectives = world == 1 or peer_red is not None

    def local_step(rays_o, rays_d, target, idx):
        """One iteration on this rank's rows: forward, per-ray loss, backward of the GLOBAL mean (train.py:1606-1607),
        gradient reduction + Adam, and the per-ray losses of all ranks for the caller's log line."""
        optimizer.zero_grad()                                    # one memset over the gradient arena
        losses = local_module(targs, rays_o, rays_d, 100, render_kwargs_train, target, global_step, 0, dataset_extras, idx)
        (losses.sum() / n_global).backward()
        if fused_collectives:
            optimizer.step()                                     # 1 GPU: Adam; N GPUs: peer reduce + Adam, same launch
            gathered = peer_red.gather_rows(losses) if peer_red is not None else losses.detach()
            global_step.add_(1.0)
            return gathered.mean(), gathered
        return losses.detach()

    graphed = None
    if not args.no_graph:
        try:
            from nonrigid_nerf_b200.graphs import GraphedStep
            graphed = GraphedStep(local_step, resident[0], warmup=3)
        except Exception as exc:  # noqa: BLE001 - fall back to the eager loop, and say so in the JSON line
            import traceback
            traceback.print_exc()
            print(f"[bench] CUDA graph capture failed ({type(exc).__name__}: {exc}); running eagerly", file=sys.stderr)
            graphed = None
            torch.cuda.synchronize()

    lrate, lrate_decay, iteration = 5e-4, 250, [0]

    def step(batch):
        iteration[0] += 1
        optimizer.set_lr(lrate * (0.1 ** (iteration[0] / (lrate_decay * 1000))))   # per-iteration decay of train.py:1631-1642
        out = graphed(*batch) if graphed is not None else local_step(*batch)
        if fused_collectives:
            return out
        # NCCL reducer: collectives outside the graph -- in-place arena all-reduce + Adam, then the loss all-gather
        optimizer.step()
        global_step.add_(1.0)
        gathered = torch.empty(world * (hi - lo), dtype=out.dtype, device=dev)
        dist.all_gather_into_tensor(gathered, out.contiguous())
        return gathered.mean(), gathered

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(loop_steps, e2e):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(loop_steps):
            if e2e:
                # host -> device copy of this step's inputs from pinned memory (straight into the graph's input buffers)
                out = step(pinned[i % pool] if graphed is not None else upload(pinned[i % pool]))
                out[0].item()                            # device -> host read of the step's result
            else:
                out = step(resident[i % pool])
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    for i in range(args.warmup):
        step(resident[i % pool])
    _lib.device_error_check()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_total, last = timed(args.steps, e2e=False)      # headline: the plain step (no instrumentation inside the graph)
    # copied to the host at once: the graph's output buffers are overwritten by the windows that follow
    outputs = None
    if args.dump_outputs and rank == 0:
        outputs = {"loss": last[0], "ray_loss": last[1],
                   "params": torch.cat([p.detach().reshape(-1) for p in grad_vars]),
                   "grads": torch.cat([p.grad.reshape(-1) for p in grad_vars])}
        outputs = {k: v.float().cpu().numpy() for k, v in outputs.items()}
    ms_e2e, _ = timed(args.steps, e2e=True)
    clocks = sampler.stop() if sampler else None
    # per-kernel breakdown: the same K steps once more with CUDA event records around every launch of this repo's
    # kernels (external event-record nodes inside the re-captured graph; they cost a few us per step themselves)
    per_step, ms_instrumented = {}, None
    # (the instrumented re-capture is skipped with the peer reducer: its kernels spin on the other ranks' flags, and a second
    # graph with event-record nodes in between is not something this bench needs -- the per-kernel breakdown is a per-GPU
    # quantity, reported by the N = 1 and NCCL runs)
    if not args.no_breakdown and peer_red is None:
        _lib.timing_enable(True)
        if graphed is not None:
            graphed = GraphedStep(local_step, resident[0], warmup=1)
            for i in range(3):
                step(resident[i % pool])
        ms_instrumented, _ = timed(args.steps, e2e=False)
        kinds = _lib.timing_read()
        _lib.timing_enable(False)
        # launches per step: forward / DGRAD / composite / composite backward 2 (coarse + fine), divergence 2 (fwd + bwd),
        # WGRAD 3 (fine, coarse, divergence; each followed by its split reduction, timed with it)
        launches = {"wgrad": 3}
        per_step = {k: (kinds[k][0] / (kinds[k][1] / float(launches.get(k, 2))) if kinds[k][1] else 0.0) for k in kinds}
    _lib.device_error_check()

    final_loss = float(step(resident[0])[0].item())
    if peer_red is not None:
        peer_red.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if outputs is not None:
        # float32; about 9 MB in all (1.07 M parameters and as many gradients, one loss per ray of the global batch)
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    value = n_global * args.steps / (ms_total * 1e-3)
    e2e_value = n_global * args.steps / (ms_e2e * 1e-3)
    peaks = read_peaks()
    traffic = read_traffic() if args.n_rand == N_RAND else None
    roof = roofline_block(per_step, args.n_rand, peaks, traffic)
    if traffic:
        roof["traffic_source"] = traffic.get("_source")
    step_tf = 3 * args.n_rand * POINTS_PER_RAY * FLOP_PER_POINT / (ms_total / args.steps * 1e-3) / 1e12
    line = {
        "metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 (tensor-core operands; f32 accumulate)", "data": "synthetic",
        "config": {"workload": workload_text(args.n_rand),
                   "parallelism": f"ray-sharded x{world}; gradient reduction: {reducer_note}",
                   "inputs": "every rank draws the global batch from the shared seed and uploads its own row block from pinned memory",
                   "l2": "per-step working set (activation + gradient stash, ~1.9 GB at 1024 rays) exceeds the 126 MB L2; 8 rotating input batches"},
        "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
        "gpu_launches": (32 if world == 1 else 36) * args.steps,
        # this repo's kernels per step, counted in profiles/r02_launches_step.csv (32 of the step's 63 launches, 94 % of its GPU
        # time): 3 weight packs, 1 coarse sampler, 2 field forwards, 2 composites, 1 ray loss + 4 scalings, 3 divergence, 2
        # composite backwards, 4 absmax, 2 field DGRADs, 3 WGRADs + 3 reductions, 2 optimizer (N GPUs: 3 peer reduce + Adam and
        # 3 loss-gather launches instead of the 2 optimizer launches)
        "kernel_ms_per_step": per_step, "ms_per_step_instrumented": (ms_instrumented / args.steps) if ms_instrumented else None,
        "cuda_graph": graphed is not None, "whole_step_in_graph": graphed is not None and fused_collectives,
        "step_tflops_algorithmic": step_tf, "step_frac_of_sustained_peak": step_tf / peaks["tf_sustained"],
        "final_loss": final_loss,
        "roofline": roof,
        "clocks": clocks,
    }
    if not args.no_cpu_baseline and world == 1:      # the CPU arm is timed next to the N = 1 run only
        cb = cpu_baseline(N_RAND, 5, 1)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "host_cores", "calibration_rays_per_s_by_threads") if k in cb}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
