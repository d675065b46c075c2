#!/usr/bin/env python
"""bench.py — depth maps/sec @ KITTI 352x1216, Swin-L, 20 DDIM steps (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W          our arm (one rank per GPU under torchrun for N > 1)
  python bench.py --impl reference ...                   the reference's CPU path (oracle port), rank 0 only

A "step" is one forward of the per-GPU batch (BASELINE config 3: 4 images, 352x1216, Swin-L, T=20) through the
plugin (`Diffusion_DCbase_Model.forward`): Swin-L backbone + HAHI neck + FPN + T-step DDIM loop + decoder, all
inside the CUDA engine (no torch compute op is left on the path); for N > 1 the batch shards by rank (weak scaling: 4
images/GPU = BASELINE config 4 at N = 8).  The path has no exchange step: by default every rank keeps (e2e: copies to
its own host buffer) the depth maps of its shard and there is NO data-path collective; `--gather step` adds an
all-gather of the depth maps per step on a side stream (`shard.DepthGatherer`; what nn.DataParallel's gather does in
the reference, src/main.py:434), `--gather blocking` waits for it on the compute stream (the round-1 behaviour).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRICS = {  # BASELINE.json's metric is quoted on C3; the other workloads are labelled as what they are
    "C3": "depth maps/sec @ KITTI 352x1216, Swin-L, 20 DDIM steps",
    "C2": "depth maps/sec @ NYUv2 228x304, ResNet-50, 20 DDIM steps",
    "C5": "depth maps/sec @ NYUv2 480x640, Swin-L, 50 DDIM steps",
    "C1": "depth maps/sec @ NYUv2 228x304, ResNet-18, 5 DDIM steps",
}
GOLDEN_OF = {"C3": "g_swinl_c3", "C2": "g_res50_c2", "C5": "g_swinl_c5", "C1": "g_res18_c1"}
WORKLOADS = {  # name -> (family, T, per-GPU batch, H, W, GFLOP per map: BASELINE.md work table)
    "C3": ("swinl", 20, 4, 352, 1216, 7258.7),
    "C2": ("res50", 20, 8, 228, 304, 270.5),
    "C5": ("swinl", 50, 8, 480, 640, 12083.0),
    "C1": ("res18", 5, 1, 228, 304, 86.8),  # BASELINE configs[0]: the reference's own CPU-runnable case (contract tests)
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def committed_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the newest committed
    `ncu --set full` summary under profiles/ (rNN_loop_convs_ncu_full_summary.csv); None if no row matches.  It is
    evidence from that capture, not a measurement of this run — the line says which file."""
    import csv
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_loop_convs_ncu_full_summary.csv")), reverse=True):
        try:
            rows = list(csv.reader(open(path)))
        except OSError:
            continue
        hdr = rows[0]
        if "dram__bytes_read.sum" not in hdr:
            continue
        ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        unit = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}.get(rows[1][ir], 1e6)
        hits = [r for r in rows[2:] if len(r) > iw and kernel_key in r[0].replace(" ", "")]
        if hits:
            vals = [(float(r[ir]) + float(r[iw])) * unit for r in hits]
            return sum(vals) / len(vals), os.path.relpath(path, ROOT)
    return None, None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in self.rows), "samples": len(self.rows)}


DUMP_BYTES = 64 << 20  # --dump-outputs writes at most this much in all


def dump_outputs(out, directory):
    """Write every tensor of the output dict `out` as <directory>/<name>.npy (float64 stays float64, everything else
    float32).  Each array keeps at most an equal share of DUMP_BYTES: a larger one is written as the 1-D array of its
    elements at a fixed, seeded, sorted sample of its flat indices, so two builds of the project write comparable files."""
    import numpy as np
    arrays = {k: v.detach() for k, v in out.items() if torch.is_tensor(v)}
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        t = t.to("cpu", torch.float64 if t.dtype == torch.float64 else torch.float32)
        cap = DUMP_BYTES // len(arrays) // t.element_size()
        if t.numel() > cap:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            t = t.reshape(-1)[idx]
        np.save(os.path.join(directory, name + ".npy"), t.numpy())


def cpu_reference_maps_per_s(workload, steps=1, warmup=0):
    """The reference's CPU path (oracle port of its forward: same torch CPU ops, all host threads) on a bounded
    sample of the workload: ONE image of the configured size per step."""
    from oracle import configs, restate
    import dd_helpers  # noqa: F401  (tests/ helper: mirror construction under the golden seed)
    family, T, _, H, W, _ = WORKLOADS[workload]
    m = dd_helpers.build_mirror(family, T)
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    sample = restate.synthetic_sample(1, H, W, configs.SEED_INPUTS)
    noise = restate.synthetic_noise(1, H, W, configs.SEED_NOISE)
    bb = configs.FAMILIES[family]["backbone_name"]
    for _ in range(warmup):
        restate.forward(sd, sample, bb, T, noise)
    t0 = time.perf_counter()
    for _ in range(steps):
        out = restate.forward(sd, sample, bb, T, noise)
    dt = (time.perf_counter() - t0) / steps
    cpu_reference_maps_per_s.last_logits = out["logits"]  # image 0 of the workload: the full-resolution parity reference
    cpu_reference_maps_per_s.last_output = out
    return 1.0 / dt, dt, f"1 image {H}x{W}, T={T}, full forward (backbone+neck+FPN+loop+decoder), fp32, {torch.get_num_threads()} threads"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C3", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--gather", default="none", choices=["none", "step", "blocking"],
                    help="N > 1: none = no data-path collective (each rank keeps its shard's depth maps); step = all-gather "
                         "them every step on a side stream; blocking = ... and wait for it on the compute stream")
    ap.add_argument("--exact", action="store_true", help="exact 3-pass fp16 split everywhere (no fp8 correction products)")
    ap.add_argument("--cpu-threads", type=int, default=0, help="host threads for the CPU reference (0 = physical cores)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the output dict of the last timed step (rank 0's) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    family, T, B, H, W, gflop_map = WORKLOADS[args.workload]
    METRIC = METRICS[args.workload]
    cfg = {"workload": f"{args.workload}: {family} backbone, T={T} DDIM steps, {B}x{H}x{W} per GPU (synthetic)",
           "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"batch-shard x{world}" + ("" if world == 1 else {
               "none": ", no data-path collective (each rank keeps its shard's depth maps)",
               "step": ", all-gather of the depth maps every step on a side stream",
               "blocking": ", blocking all-gather of the depth maps every step"}[args.gather]),
           "l2": "per-step working set ~1.3 GB of activations streamed per conv >> 126 MB L2 (no cross-step reuse)"}

    def host_threads():
        if args.cpu_threads > 0:
            return args.cpu_threads
        # 32 threads was the fastest of {16, 32, 64, 128} for this forward on the pool's hosts (0.101 / 0.114 / 0.081 /
        # 0.020 maps/s): oneDNN's small convs stop scaling and then oversubscribe
        try:
            import psutil
            return min(psutil.cpu_count(logical=False) or os.cpu_count() or 1, 32)
        except Exception:
            return min(os.cpu_count() or 1, 32)

    if args.impl == "reference":
        if rank != 0:
            return 0
        torch.set_num_threads(host_threads())
        # bounded: one image per step
        n_timed = args.steps
        n_warm = min(args.warmup, 1)
        v, dt, what = cpu_reference_maps_per_s(args.workload, steps=n_timed, warmup=n_warm)
        if args.dump_outputs:
            dump_outputs(cpu_reference_maps_per_s.last_output, args.dump_outputs)
        what += f"; {n_timed} timed + {n_warm} warm-up executions of ONE image each (bounded sample of the {B}-image step)"
        # `steps` / `warmup` are what was EXECUTED (the request was --steps K --warmup W: see `requested`); each executed
        # step is one image, not the per-GPU batch of the config — maps/s normalises that
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": "maps/s", "n_gpus": args.gpus, "steps": n_timed,
            "warmup": n_warm, "requested": {"steps": args.steps, "warmup": args.warmup},
            "executed": {"steps": n_timed, "warmup": n_warm, "images_per_step": 1},
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": "maps/s", "cores": torch.get_num_threads(), "kind": "port", "sample": what},
            "e2e": {"value": v, "unit": "maps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    import diffusiondepth_b200 as dd
    from diffusiondepth_b200 import shard
    from oracle import configs, restate
    import dd_helpers
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (our arm) needs a B200; there is no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line: NCCL prints its "NCCL version ..." banner with printf when the communicator is
        # created (NCCL_DEBUG=VERSION on the pool's boxes), so file descriptor 1 points at stderr while that happens
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()  # eager communicator creation: the banner is out before stdout comes back
            torch.cuda.synchronize()
        finally:
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    model = dd_helpers.build_mirror(family, T).to(dev)
    model.depth_head.use_cuda_graph = not args.no_graph
    model.depth_head.check_range = False
    model.depth_head.fp8_corrections = not args.exact
    first, _ = shard.shard_range(B * world, rank, world)
    host = restate.synthetic_sample(B, H, W, configs.SEED_INPUTS, first=first)
    host["noise"] = restate.synthetic_noise(B, H, W, configs.SEED_NOISE, first=first)
    host = {k: v.pin_memory() for k, v in host.items()}
    resident = {k: v.to(dev) for k, v in host.items()}

    # N > 1: the single collective of the path (all-gather of the depth maps) runs on a side stream into rotating buffers
    # (shard.DepthGatherer), so no rank's next step queues behind a slower peer's current one
    gatherer = shard.DepthGatherer(B * world) if world > 1 and args.gather != "none" else None

    last = {}

    def step_resident():
        with torch.no_grad():
            out = model(resident)
        last["out"] = out
        pred = out["pred"]
        if gatherer is None:
            return pred
        return gatherer.result(gatherer.submit(pred)) if args.gather == "blocking" else gatherer.submit(pred)

    # end to end = the call a user of the reference makes (src/main.py:456-470): pinned host sample -> device ->
    # net(sample) -> host, every step; the initial latent is drawn on the device by the head, exactly as the reference
    # does (head :283).  Serving-style double buffering: the inputs of step i+1 are copied on a side stream while step i
    # computes, and step i's depth maps land in a pinned host buffer asynchronously and are read one step later.
    copy_stream = torch.cuda.Stream(device=dev)
    out_host = [torch.empty(B, 1, H, W, dtype=torch.float32).pin_memory() for _ in range(2)]
    pending = {"inputs": None, "done": None, "slot": 0}

    def fetch_inputs():
        with torch.cuda.stream(copy_stream):
            d = {k: v.to(dev, non_blocking=True) for k, v in host.items() if k != "noise"}
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return d, ev

    def step_e2e_serial():
        # the same call with nothing overlapped: copy in, compute, blocking copy out
        with torch.no_grad():
            out = model({k: v.to(dev, non_blocking=True) for k, v in host.items() if k != "noise"})
        if gatherer is None:
            return out["pred"].to("cpu", non_blocking=False)
        return shard.gather_depth(out["pred"], B * world)[first:first + B].to("cpu", non_blocking=False)

    def step_e2e():
        cur = torch.cuda.current_stream()
        d, ev = pending["inputs"] if pending["inputs"] is not None else fetch_inputs()
        cur.wait_event(ev)
        for t in d.values():
            t.record_stream(cur)
        pending["inputs"] = fetch_inputs()  # next step's host->device copy overlaps this step's compute
        with torch.no_grad():
            out = model(d)
        pred = gatherer.result(gatherer.submit(out["pred"]))[first:first + B] if gatherer is not None else out["pred"]
        if pending["done"] is not None:
            pending["done"].synchronize()  # the previous step's result is now readable on the host
        slot = pending["slot"]
        out_host[slot].copy_(pred, non_blocking=True)
        done = torch.cuda.Event()
        done.record(cur)
        pending["done"], pending["slot"] = done, slot ^ 1
        return out_host[slot]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    per_rank = {}

    def timed(fn, steps, tag=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if gatherer is not None:
            gatherer.drain()  # the last steps' all-gathers belong to the timed region
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            allms = [torch.zeros_like(ms) for _ in range(world)]
            dist.all_gather(allms, ms)
            v = sorted(float(t.item()) / steps for t in allms)
            if tag:
                per_rank[tag] = {"min": v[0], "median": v[len(v) // 2], "max": v[-1], "unit": "ms_per_step",
                                 "what": "each rank's own CUDA-event time over the K steps; the reported value uses the max"}
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    for _ in range(max(args.warmup, 3)):
        step_resident()
    eng = next(iter(model.depth_head._engines.values()))
    eng.poll_status()  # the split must not have overflowed on this workload
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms = timed(step_resident, args.steps, "resident")
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(last["out"], args.dump_outputs)  # before any later call can reuse the engine's output buffers
    if gatherer is not None:
        # the same steps WITHOUT the collective: each rank's own pace.  With it, every rank's clock stops when the slowest
        # peer has delivered its last shard, so `resident` shows one number for all ranks; this one shows the spread
        # (power-capped GPUs of one box differ by a few per cent) that bounds weak-scaling efficiency from outside.
        def step_local():
            with torch.no_grad():
                return model(resident)["pred"]
        timed(step_local, args.steps, "compute_only_no_gather")
    launches = eng.last_launch_count * args.steps
    value = B * world * args.steps / (ms / 1e3)
    step_e2e()
    ms_e2e = timed(step_e2e, args.steps, "e2e")
    e2e_value = B * world * args.steps / (ms_e2e / 1e3)
    ms_serial = timed(step_e2e_serial, args.steps)
    rank_means = None
    if world > 1:  # outside the timed regions: every rank really produced its shard (different images -> different means)
        with torch.no_grad():
            pm = model(resident)["pred"].clamp(max=1e3).mean().reshape(1)
        allm = [torch.zeros_like(pm) for _ in range(world)]
        dist.all_gather(allm, pm)
        rank_means = [float(t.item()) for t in allm]
    h2d = sum(v.numel() * v.element_size() for k, v in host.items() if k != "noise")
    d2h = B * H * W * 4

    # parity of THIS run (BASELINE.md: "parity gate reported with every throughput number"): image 0 of rank 0's shard
    # against the committed golden of the real reference (sub-sampled for the large cases), and further down, when the
    # CPU leg runs, against the fp32 restatement on every pixel
    parity, z0 = None, None
    if rank == 0:
        import numpy as np
        head = model.depth_head
        head.capture_logits = True
        with torch.no_grad():
            model(resident)
        z0 = head.last_logits[:1].float().cpu()
        head.capture_logits = False
        gpath = os.path.join(ROOT, "tests", "golden", GOLDEN_OF[args.workload] + ".npz")
        if os.path.exists(gpath):
            gz = np.load(gpath, allow_pickle=False)
            st = int(gz["logits_stride"])
            dz = (z0[..., ::st, ::st] - torch.from_numpy(gz["logits"])).abs().double()
            parity = {"case": GOLDEN_OF[args.workload], "against": f"real reference forward (golden, logits sub-sampled x{st})",
                      "max_dz": dz.max().item(), "rms_dz": dz.pow(2).mean().sqrt().item(), "tolerance": 1e-3,
                      "what": "|dz| on the decoder logit == relative depth error", "n": dz.numel(),
                      "mode": "exact 3-pass fp16 split" if args.exact else "fp8 correction products on convA / convB / noise_embedding.3"}

    # roofline of the dominant kernel: the 256->256 3x3 conv (convA/convB = 79 % of the loop's FLOPs)
    pk = peaks()
    roof = None
    if rank == 0:
        cin, cout = (256, 256) if family == "swinl" else (256, 64)
        iters = 20
        kms = eng.bench_conv(cin, cout, iters)
        P = B * ((H + 1) // 2) * ((W + 1) // 2)
        flops = 2.0 * P * cout * 9 * cin  # algorithmic (one fp32-grade product-sum per MAC), not the 3x issued
        ach = flops / (kms * 1e-3) / 1e12
        f8 = (cout == 256 and not args.exact)
        kname = (f"conv3x3_halo_kernel<{cin},{cout},{64 if f8 else 32},EPI_SPLIT,PAIR{',F8' if f8 else ''}>" if cout == 256
                 else f"conv3x3_swap_kernel<{cin},{cout},32,EPI_F32_STATS,HALO>")
        traffic, tsrc = committed_traffic(f"conv3x3_halo_kernel<{cin},{cout},{64 if f8 else 32},1,1,{1 if f8 else 0}>" if cout == 256
                                          else f"conv3x3_swap_kernel<{cin},{cout},32,0,1>")
        passes = 2.0 if f8 else 3.0  # pass-equivalents issued per algorithmic MAC (an e4m3 K=32 MMA = half an fp16 pass)
        roof = {"bound": "tensor", "kernel": kname, "achieved": ach, "peak": pk["tf_burst"],
                "unit": "TFLOP/s", "frac": ach / pk["tf_burst"], "issued_frac": passes * ach / pk["tf_burst"],
                "pass_equivalents": passes, "ceiling_frac": 1.0 / passes,
                "ms_per_launch": kms, "traffic": (traffic if args.workload == "C3" else None),
                "traffic_source": (f"ncu --set full dram__bytes_read+write per launch, read from the committed {tsrc} (not measured in this run)"
                                   if traffic else "no committed ncu row for this kernel"),
                "algorithmic_bytes": 4.0 * P * (cin + cout), "peak_source": pk["source"] + ", bf16 burst",
                "note": ("achieved = algorithmic FLOPs (one fp32-grade product per MAC); the operand split issues "
                         f"{passes:g} fp16-pass-equivalents of tensor work per MAC, so {1.0 / passes:.2f} of the bf16 peak is the ceiling")}
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        torch.set_num_threads(host_threads())
        v, dt, what = cpu_reference_maps_per_s(args.workload, steps=1, warmup=0)
        cpu = {"value": v, "unit": "maps/s", "cores": torch.get_num_threads(), "kind": "port", "sample": what,
               "seconds": dt}
        zr = getattr(cpu_reference_maps_per_s, "last_logits", None)
        if parity is not None and zr is not None and z0 is not None and tuple(zr.shape) == tuple(z0.shape):
            dzf = (z0 - zr.float()).abs().double()  # same image, same noise: the CPU leg's own output, every pixel
            parity["full_resolution"] = {"against": "fp32 CPU restatement of the reference (this run's cpu_baseline leg), all pixels",
                                         "max_dz": dzf.max().item(), "rms_dz": dzf.pow(2).mean().sqrt().item(), "n": dzf.numel()}
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": "maps/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": ("f32 (fp32-grade products on tcgen05: 3-pass fp16 split, fp32 accumulate in TMEM" +
                      (")" if args.exact or family != "swinl" else "; convA / convB / noise_embedding.3: fp16 hi*hi + two e4m3 correction products)")),
            "data": "synthetic",
            "config": cfg, "clocks": clocks, "gpu_launches": launches, "parity": parity,
            "per_rank_ms_per_step": per_rank or None, "per_rank_output_mean": rank_means,
            "e2e": {"value": e2e_value, "unit": "maps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps,
                    "serial": {"value": B * world * args.steps / (ms_serial / 1e3), "ms_per_step": ms_serial / args.steps,
                               "what": "same call, copies not overlapped (blocking D2H every step)"},
                    "pipeline": "double-buffered: step i+1 inputs H2D on a side stream during step i; depth maps D2H "
                                "async into pinned memory, read one step later"},
            "roofline": roof, "cpu_baseline": cpu,
            "algorithmic_tflops": value * gflop_map / 1e3, "frac_of_bf16_sustained": value * gflop_map / 1e3 / pk["tf_sustained"]}))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
