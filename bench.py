#!/usr/bin/env python
"""Benchmark of the MoGe-2 hot path (BASELINE.json metric: images/sec, ViT-L, 518 px, fp16).

  python bench.py --gpus 1 --steps K --warmup W                 engine arm (this repo, sm_100a kernels)
  torchrun ... bench.py --gpus N ...                              one rank per GPU, weak scaling (fixed images per GPU)
  python bench.py --impl reference ...                            the reference algorithm on the host cores (oracle port)
  python bench.py ... --dump-outputs DIR                          also write the last timed step's infer() outputs to DIR/*.npy

A "step" is one `MoGeModel.infer()` over one batch of synthetic 518x518 images per GPU.  Rank 0 prints ONE JSON line.
  value  : images/s with the inputs already resident in HBM (device-timed, max over ranks)
  e2e    : images/s through the public API with HOST buffers: pinned host -> H2D -> infer -> D2H of every output
  roofline      : encoder GEMM launches of the tcgen05 kernel (tensor bound), flops / CUDA-event time, live
  roofline_decoder / roofline_attention : the other two kernel classes
  cpu_baseline  : the oracle port (restated reference algorithm, fp32) timed on this box's host cores (rank 0, N=1)
"""
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

# One hardware work queue per CUDA stream (default: 8 queues shared by all streams of the process).  The gather / copy side streams
# must never share a queue with the compute stream: a stream that waits for a peer's flag would stall the kernels queued behind it.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import torch  # noqa: E402


METRIC = "images/sec ViT-L 518px fp16 (MoGe-2 infer)"      # BASELINE.json metric, same string on both arms


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="images per GPU per step")
    ap.add_argument("--size", default="vitl")
    ap.add_argument("--res", type=int, default=518)
    ap.add_argument("--tokens", type=int, default=1369, help="requested base tokens (1369 -> native 37x37 grid at 518 px)")
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-images", type=int, default=12, help="bounded CPU sample: single-image infers of the oracle port (~1.3 s each on 16 cores)")
    ap.add_argument("--dump-ops", default=None, help="write the per-launch profile (name, ms, flops, bytes) to this JSON file")
    ap.add_argument("--config", type=int, default=0, help="0: the driver's default line (BASELINE.json configs[1]/[3]); 3: mixed-aspect "
                    "~700-token ViT-L-normal bf16 batch (configs[2]); 5: ViT-B resolution / aspect sweep (configs[4])")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the same-box PyTorch-CUDA comparator (gpu_baseline)")
    ap.add_argument("--gpu-baseline-kernels", default=None, help="write the torch.profiler kernel list of one batch-1 comparator pass here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the infer() outputs of the last timed step (rank 0) to DIR/<name>.npy as float32; above 64 MB in all, "
                         "a fixed, seeded sample of pixels (see dump_outputs)")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "engine" or a.config != 0):
        ap.error("--dump-outputs applies to the engine arm of the default workload")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d["bf16_tflops_sustained"], "source": "measured (MEASURED_PEAKS.json, sustained)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled (~every 50-100 ms) while the timed region runs."""

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.th = index, [], threading.Event(), None

    def _run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.05)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag.set()
        if self.th:
            self.th.join(6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


DUMP_BYTES = 64 * 10**6


def dump_outputs(out, path, H, W):
    """Write one infer() result to `path`/<name>.npy as float32 (mask as 0 / 1).  Pixels outside the mask, which infer() fills
    with inf in points / depth and with 0 in normal, are written as 0: every file is finite, and mask.npy tells which pixels
    hold values.  When the (B, H, W[, C]) maps would exceed DUMP_BYTES in all, every map keeps the same fixed, seeded sample of
    pixels: maps become (B, n[, C]) and the row-major pixel indices into H x W are written as pixel_index.npy (float64).
    Same arguments -> same inputs -> comparable files across builds."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    out = {k: v.float().cpu() for k, v in out.items()}
    maps = {k: v for k, v in out.items() if v.dim() >= 3 and tuple(v.shape[1:3]) == (H, W)}
    if "mask" in maps:
        valid = maps["mask"] > 0
        maps = {k: torch.where(valid if v.dim() == 3 else valid[..., None], v, 0.0) for k, v in maps.items()}
    rest = sum(v.numel() * 4 for k, v in out.items() if k not in maps) + 128 * (len(out) + 1)       # + .npy headers
    n = min(H * W, (DUMP_BYTES - rest) // (sum(v.numel() // (H * W) for v in maps.values()) * 4 + 8))
    if n < H * W:
        idx = torch.randperm(H * W, generator=torch.Generator().manual_seed(0))[:n].sort().values
        np.save(os.path.join(path, "pixel_index.npy"), idx.double().numpy())
        maps = {k: v.flatten(1, 2)[:, idx] for k, v in maps.items()}
    for k, v in {**out, **maps}.items():
        np.save(os.path.join(path, k + ".npy"), v.contiguous().numpy())


def host_threads():
    """Host cores this process may actually use (affinity / cgroup aware), not the machine total."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = max(1, min(n, int(int(q[0]) / int(q[1]))))
    except Exception:
        pass
    return n


def cpu_port_images_per_s(size, res, tokens, n_images, threads):
    """The reference algorithm (oracle port, fp32) on the host cores: images/s over `n_images` single-image infers."""
    from moge_b200.configs import model_config
    from moge_b200.synthetic import make_state_dict, synthetic_images
    from oracle import moge_port
    torch.set_num_threads(threads)
    cfg = model_config(size, True)
    sd = make_state_dict(cfg, 0)
    img = synthetic_images(1, res, res, 0)
    moge_port.infer(cfg, sd, synthetic_images(1, 56, 56, 1), num_tokens=16)      # tiny warm-up (thread pool, allocator)
    t0 = time.perf_counter()
    for _ in range(n_images):
        moge_port.infer(cfg, sd, img, num_tokens=tokens)
    dt = time.perf_counter() - t0
    return n_images / dt, dt


def gpu_baseline(cfg, sd, dev, res, tokens, batch, iters_b1=200, kernels_path=None):
    """Same-box PyTorch-CUDA comparator (SURVEY.md 8d "Reference GPU baseline"): the reference's algorithm as plain PyTorch ops
    (oracle/moge_port.py -> cuBLAS / cuDNN / SDPA kernels, SciPy focal solve on the host exactly like geometry_torch.py:150-166),
    in the reference's two 16-bit modes: (i) `.half()` weights + input, (ii) fp32 weights under torch.autocast(fp16)
    (v2.py:241).  Batch-1 latency (p50 / p90 over `iters_b1` runs, CUDA events, host solve inside) and batch-`batch` images/s."""
    import contextlib
    from oracle import moge_port
    out = {"kind": "oracle port (the reference's algorithm as plain PyTorch ops) on cuda: cuBLAS/cuDNN/SDPA + host SciPy solve",
           "torch": torch.__version__}
    g = torch.Generator().manual_seed(99)
    img = torch.rand(batch, 3, res, res, generator=g).to(dev)
    aspect = 1.0
    for mode in ("half", "autocast"):
        if mode == "half":
            sdd = {k: v.to(dev).half() for k, v in sd.items() if v.is_floating_point()}
            x_all, ctx = img.half(), contextlib.nullcontext
        else:
            sdd = {k: v.to(dev).float() for k, v in sd.items() if v.is_floating_point()}
            x_all, ctx = img, (lambda: torch.autocast("cuda", dtype=torch.float16))

        def run(x):
            with torch.inference_mode():
                with ctx():
                    raw = moge_port.forward(cfg, sdd, x, tokens)
                raw = {k: v.float() for k, v in raw.items()}
                return moge_port.postprocess(raw.get("points"), raw.get("normal"), raw.get("mask"), raw.get("metric_scale"), aspect)

        one = x_all[:1].contiguous()
        for _ in range(10):
            run(one)
        torch.cuda.synchronize()
        lat = []
        for _ in range(iters_b1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(one)
            e1.record()
            torch.cuda.synchronize()
            lat.append(e0.elapsed_time(e1))
        run(x_all)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        nrep = 3
        for _ in range(nrep):
            run(x_all)
        e1.record()
        torch.cuda.synchronize()
        out[mode] = {"batch1_p50_ms": statistics.median(lat), "batch1_p90_ms": sorted(lat)[int(0.9 * len(lat))], "batch1_iters": len(lat),
                     "batch": batch, "images_per_s": batch * nrep / (e0.elapsed_time(e1) / 1e3)}
        if kernels_path and mode == "half":
            from torch.profiler import profile, ProfilerActivity
            with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
                run(one)
                torch.cuda.synchronize()
            rows = [{"kernel": e.key, "calls": e.count, "cuda_us": e.device_time_total} for e in prof.key_averages()
                    if getattr(e, "device_time_total", 0) > 0 and e.device_type.name == "CUDA"]
            rows.sort(key=lambda r: -r["cuda_us"])
            with open(kernels_path, "w") as fh:
                json.dump({"mode": mode, "batch": 1, "launches": sum(r["calls"] for r in rows),
                           "cuda_us_total": sum(r["cuda_us"] for r in rows), "kernels": rows[:60]}, fh, indent=1)
        del sdd
    return out


def workload_name(a, h, w):
    return (f"MoGe-2 {a.size} {a.dtype} infer(), {a.batch} x {a.res}x{a.res} images per GPU, num_tokens={a.tokens} -> {h}x{w} grid "
            f"(BASELINE.json configs[1]/[3] shape; random-init weights)")


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from moge_b200.configs import token_grid
    threads = host_threads()
    h, w = token_grid(a.res, a.res, a.tokens)
    per_step = 1
    # bounded sample: each step = 1 image; warm-up is capped at one image to keep the run within minutes
    ips_w, _ = cpu_port_images_per_s(a.size, a.res, a.tokens, 1, threads) if a.warmup > 0 else (0, 0)
    ips, dt = cpu_port_images_per_s(a.size, a.res, a.tokens, a.steps * per_step, threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": a.gpus,
        "steps": a.steps, "warmup": min(a.warmup, 1), "ms_per_step": 1000.0 * dt / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a, h, w), "sample": "1 image per step on the host cores"},
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": threads, "kind": "port",
                         "sample": f"{a.steps} single-image infer() calls, oracle/moge_port.py fp32, torch CPU {threads} threads"},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_engine(a):
    import torch.distributed as dist
    from moge.model.v2 import MoGeModel
    from moge_b200.configs import model_config, token_grid
    from moge_b200.synthetic import make_state_dict
    from moge_b200 import parallel
    from moge_b200.serving import InferPipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: anything native libraries print (e.g. NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = model_config(a.size, True)
    # ---- weights: rank 0 builds the seeded checkpoint; one NCCL broadcast ships it to every GPU (SURVEY.md 8e)
    t_w = time.perf_counter()
    if world > 1:
        sd = parallel.broadcast_state_dict(make_state_dict(cfg, 0) if rank == 0 else None, dev)
    else:
        sd = make_state_dict(cfg, 0)
    model = MoGeModel(**cfg)
    model.load_state_dict(sd)
    model = model.to(dev).eval()
    if a.dtype == "bf16":
        model = model.bfloat16()
    B, R = a.batch, a.res
    h, w = token_grid(R, R, a.tokens)
    g = torch.Generator().manual_seed(1234 + rank)
    host_in = torch.rand(B, 3, R, R, generator=g).pin_memory()
    dev_in = host_in.to(dev)
    out = model.infer(dev_in, num_tokens=a.tokens)            # builds engine + plan
    torch.cuda.synchronize()
    del sd
    load_s = time.perf_counter() - t_w
    host_out = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in out.items()}
    d2h_bytes = sum(v.numel() * v.element_size() for v in out.values())
    h2d_bytes = host_in.numel() * host_in.element_size()
    n_ops = len(model.engine_ops()) + 2                        # + focal/shift solve + post-processing

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, fence=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if fence is not None:
            fence()                     # the timing stream waits for the pipeline's copy streams
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    last_out = [None]

    def step_dev():
        last_out[0] = model.infer(dev_in, num_tokens=a.tokens)

    def step_e2e():
        x = host_in.to(dev, non_blocking=True)
        o = model.infer(x, num_tokens=a.tokens)
        for k, v in o.items():
            host_out[k].copy_(v, non_blocking=True)

    for _ in range(a.warmup):
        step_dev()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev = timed(step_dev, a.steps)
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump_outputs(last_out[0], a.dump_outputs, R, R)
    last_out[0] = None
    for _ in range(min(a.warmup, 2)):
        step_e2e()
    ms_e2e_serial = timed(step_e2e, a.steps)
    # the serving loop (moge_b200/serving.py): H2D of batch i+1, infer() of batch i and D2H of batch i-1 overlap; every
    # step still copies its own input from pinned host memory and all five outputs back, inside the timed region
    pipe = InferPipeline(model, depth=2, num_tokens=a.tokens)
    host_out2 = [host_out, {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in out.items()}]
    counter = [0]

    def step_pipe():
        pipe.submit(host_in, host_out2[counter[0] & 1])
        counter[0] += 1

    for _ in range(min(a.warmup, 2)):
        step_pipe()
    pipe.join()
    ms_e2e = timed(step_pipe, a.steps, fence=pipe.fence)

    # ---- BASELINE.json configs[3] as defined: "inputs resident on each GPU -> all outputs resident on rank 0".  Every step ends
    #      with a gather of the five output maps into preallocated full-batch buffers on rank 0 (peer-memory pulls, PeerGatherer;
    #      the NCCL isend/irecv form, OutputGatherer, is timed beside it), so the transfer of step i runs under the compute of
    #      step i+1; the timed region ends when the LAST step's outputs are on rank 0.  At N > 1 this is the line's `value`.
    gather = None
    ms_gather = None
    if world > 1:
        def run_gather(gat):
            def step_gather():
                gat.submit(model.infer(dev_in, num_tokens=a.tokens))

            def step_gather_serial():
                gat.submit(model.infer(dev_in, num_tokens=a.tokens))
                gat.fence()

            for _ in range(2):
                step_gather()                                   # first calls set up the channels / buffers
            gat.wait()
            barrier()
            return timed(step_gather, a.steps, fence=gat.fence), timed(step_gather_serial, a.steps, fence=gat.fence)

        # (a) product path: peer-memory gather -- IPC-mapped staging slots pulled by rank 0's copy engines, device-side flags,
        #     no SM time (moge_b200.parallel.PeerGatherer over libmoge_b200's moge_peer_* entry points)
        gat, peer_error = parallel.PeerGatherer([B] * world, dev), None
        try:
            ms_gather, ms_gather_serial = run_gather(gat)
        except parallel.PeerSetupError as ex:          # raised on every rank together (no CUDA IPC / peer access on this box)
            gat, peer_error = None, str(ex)
        # (b) for comparison: the same gather as grouped NCCL isend/irecv on a side stream (copy kernels on both ends)
        gat_nccl = parallel.OutputGatherer([B] * world, device=dev)
        ms_nccl, ms_nccl_serial = run_gather(gat_nccl)
        nccl_api = "moge_b200.parallel.OutputGatherer (grouped NCCL isend/irecv on a side stream)"
        if gat is None:                                # fall back: the NCCL gather is the measured path of this run
            ms_gather, ms_gather_serial = ms_nccl, ms_nccl_serial
        gather = {"bytes_to_rank0_per_step": d2h_bytes * (world - 1), "ms_per_step_pipelined": ms_gather / a.steps,
                  "ms_per_step_serial": ms_gather_serial / a.steps, "ms_per_step_no_gather": ms_dev / a.steps,
                  "api": ("moge_b200.parallel.PeerGatherer.submit(infer(...)) per step, fence() at the end: CUDA-IPC staging slots, "
                          "copy-engine pulls by rank 0, device-side flags; no SM time") if gat is not None
                         else nccl_api + " -- fallback: " + peer_error,
                  "nccl_isend_irecv": {"ms_per_step_pipelined": ms_nccl / a.steps, "ms_per_step_serial": ms_nccl_serial / a.steps,
                                       "api": nccl_api}}
        if gat is not None:
            if gat.debug:
                gather["debug_ms"] = gat.debug_report()
                print(f"[rank {rank}] gather debug (ms): {gather['debug_ms']}", file=sys.stderr, flush=True)
            gat.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- per-launch CUDA-event profile of one step -> roofline of each kernel class (live, same process)
    model.infer(dev_in, num_tokens=a.tokens)
    ops = model.engine_ops()
    prof = [model.engine_profile() for _ in range(3)]
    ms_op = [min(p[i] for p in prof) for i in range(len(ops))]
    pk = peaks()
    if a.dump_ops:
        with open(a.dump_ops, "w") as fh:
            json.dump([{"name": n, "ms": ms_op[i], "flops": f, "bytes": b} for i, (n, f, b) in enumerate(ops)], fh, indent=0)

    def cls(prefixes):
        idx = [i for i, (n, _, _) in enumerate(ops) if n.startswith(prefixes)]
        t = sum(ms_op[i] for i in idx) / 1e3
        return idx, t, sum(ops[i][1] for i in idx), sum(ops[i][2] for i in idx)

    # DRAM traffic of the dominant launch of each class, from the committed `ncu --set full` capture of this workload
    # (profiles/r2_ncu_traffic.json; per launch, like `achieved`); null for any other workload
    traffic = {}
    tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r2_ncu_traffic.json")
    if a.size == "vitl" and B == 32 and R == 518 and a.tokens == 1369 and a.dtype == "fp16" and os.path.exists(tpath):
        with open(tpath) as fh:
            traffic = json.load(fh)

    def traffic_of(key):
        t_ = traffic.get(key)
        return (None, None) if not t_ else (t_["dram_bytes"], {"kernel": t_["kernel"], "algorithmic_bytes": t_["algorithmic_bytes"],
                                                                "ratio_to_algorithmic": t_["dram_bytes"] / t_["algorithmic_bytes"], "source": t_["file"]})

    total_prof_ms = sum(ms_op)
    idx, t, fl, by = cls(("gemm.",))
    roofline = {"kernel": "umma2_kernel (cta_group::2) + umma_kernel<AMODE_ROWS>: encoder linears patch/qkv/proj/fc1/fc2/taps", "bound": "tensor",
                "achieved": fl / t / 1e12, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": fl / t / 1e12 / pk["tflops"],
                "traffic": traffic_of("gemm")[0], "traffic_detail": traffic_of("gemm")[1], "launches": len(idx), "ms_per_step": t * 1e3,
                "share_of_step": t * 1e3 / total_prof_ms, "peak_source": pk["source"]}
    idx, t, fl, by = cls(("conv",))
    dec_bound_s = max(fl / (pk["tflops"] * 1e12), by / (pk["hbm_gbs"] * 1e9))
    # algorithmic bytes: SURVEY.md 8(d) "every tensor that crosses a conv boundary once": 501 760 elements x T per image at 2 bytes
    # (the engine's own per-launch count `by` is LOWER -- its load-time folds removed tensors -- and is reported beside it)
    by_survey = 501760.0 * (h * w) * 2 * B
    roofline_decoder = {"kernel": "umma_kernel<AMODE_TILES> + convh_kernel + conv64_kernel (implicit-GEMM convs)", "bound": "hbm",
                        "achieved": by_survey / t / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": by_survey / t / 1e9 / pk["hbm_gbs"],
                        "bytes_definition": "SURVEY.md 8(d): 501760 * T elements * 2 B per image (conv-boundary tensors once)",
                        "engine_bytes_per_step": by, "frac_engine_bytes": by / t / 1e9 / pk["hbm_gbs"],
                        "tensor_tflops": fl / t / 1e12, "frac_of_max_bound": dec_bound_s / t, "traffic": traffic_of("decoder")[0],
                        "traffic_detail": traffic_of("decoder")[1], "launches": len(idx),
                        "ms_per_step": t * 1e3, "share_of_step": t * 1e3 / total_prof_ms}
    idx, t, fl, by = cls(("attention",))
    roofline_attention = {"kernel": "attention_kernel", "bound": "tensor", "achieved": fl / t / 1e12, "peak": pk["tflops"],
                          "unit": "TFLOP/s", "frac": fl / t / 1e12 / pk["tflops"], "traffic": traffic_of("attention")[0],
                          "traffic_detail": traffic_of("attention")[1], "launches": len(idx), "ms_per_step": t * 1e3,
                          "share_of_step": t * 1e3 / total_prof_ms}
    other_ms = total_prof_ms - roofline["ms_per_step"] - roofline_decoder["ms_per_step"] - roofline_attention["ms_per_step"]

    # ---- batch-1 latency (BASELINE.json configs[1]): p50 / p90 over 200 device-timed single-image infers after 20 warm-ups; every
    #      call gets a fresh input tensor address and fresh output tensors (the graph covers the workspace-only launches)
    one = dev_in[:1].contiguous()
    for _ in range(20):
        model.infer(one, num_tokens=a.tokens)
    lat = []
    for _ in range(200):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        model.infer(one, num_tokens=a.tokens)
        e1.record()
        torch.cuda.synchronize()
        lat.append(e0.elapsed_time(e1))
    latency = {"batch": 1, "p50_ms": statistics.median(lat), "p90_ms": sorted(lat)[int(0.9 * len(lat))], "iters": len(lat)}

    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        threads = host_threads()
        ips, dt = cpu_port_images_per_s(a.size, R, a.tokens, a.cpu_images, threads)
        cpu = {"value": ips, "unit": "images/s", "cores": threads, "kind": "port",
               "sample": f"{a.cpu_images} single-image infer() calls ({dt:.1f} s), oracle/moge_port.py fp32, torch CPU {threads} threads"}

    gpu_base = None
    if world == 1 and not a.no_gpu_baseline:
        gpu_base = gpu_baseline(cfg, make_state_dict(cfg, 0), dev, R, a.tokens, B, kernels_path=a.gpu_baseline_kernels)

    images = B * world * a.steps
    ms_value = ms_gather if ms_gather is not None else ms_dev       # N > 1: the gather to rank 0 is inside the timed region
    line = {
        "metric": METRIC, "value": images / (ms_value / 1e3), "unit": "images/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_value / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": a.dtype, "data": "synthetic",
        "config": {"workload": workload_name(a, h, w), "images_per_gpu": B, "grid": [h, w],
                   "l2": "per-step working set (activation workspace, GBs) far exceeds the 126 MB L2; no explicit flush",
                   "weights": "seeded random init (moge_b200.synthetic), broadcast from rank 0 over NCCL" if world > 1 else "seeded random init"},
        "e2e": {"value": images / (ms_e2e / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                "ms_per_step": ms_e2e / a.steps, "api": "moge_b200.serving.InferPipeline(model).submit(pinned_in, pinned_out) / join()",
                "overlap": "H2D(i+1) | infer(i) | D2H(i-1) on three streams, depth 2",
                "serial": {"value": images / (ms_e2e_serial / 1e3), "ms_per_step": ms_e2e_serial / a.steps,
                           "api": "x = pinned.to(dev); o = model.infer(x); pinned_out.copy_(o) on one stream"}},
        "gpu_launches": n_ops * a.steps,
        "launches_per_step": n_ops,
        "clocks": clocks,
        "roofline": roofline, "roofline_decoder": roofline_decoder, "roofline_attention": roofline_attention,
        "profile_ms": {"sum_of_launches": total_prof_ms, "other_kernels": other_ms},
        "latency": latency,
        "cpu_baseline": cpu,
        "gpu_baseline": gpu_base,
        "load_s": load_s,
    }
    line["value_compute_only"] = images / (ms_dev / 1e3)
    if gather:
        line["gather"] = gather
        line["value_with_gather"] = line["value"]
        line["config"]["value_definition"] = ("N > 1: images/s from inputs resident on each GPU to ALL outputs resident on rank 0 "
                                              "(output gather inside the timed region, overlapped with the next step's compute; "
                                              "transport: see gather.api)")
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _class_times(model, ops_prefixes=("gemm.", "attention", "conv")):
    """One CUDA-event replay of the last forward's launch list -> {class: (seconds, flops, bytes)} (best of 3)."""
    ops = model.engine_ops()
    prof = [model.engine_profile() for _ in range(3)]
    ms = [min(p[i] for p in prof) for i in range(len(ops))]
    out = {}
    for pre in ops_prefixes:
        idx = [i for i, (n, _, _) in enumerate(ops) if n.startswith(pre)]
        out[pre] = (sum(ms[i] for i in idx) / 1e3, sum(ops[i][1] for i in idx), sum(ops[i][2] for i in idx))
    out["all"] = (sum(ms) / 1e3, sum(o[1] for o in ops), sum(o[2] for o in ops))
    return out


def _timed_steps(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def decoder_bytes_survey(c0, tokens, images):
    """SURVEY.md 8(d): conv-boundary tensors once, 2-byte storage: neck 3E0+14E1+14E2+14E3+E4, each head 3E0+12E1+12E2+12E3+5E4."""
    e = [c0, 1024, 2048, 4096, 8192]
    neck = 3 * e[0] + 14 * (e[1] + e[2] + e[3]) + e[4]
    head = 3 * e[0] + 12 * (e[1] + e[2] + e[3]) + 5 * e[4]
    return (neck + 3 * head) * 2.0 * tokens * images


def run_config3(a):
    """BASELINE.json configs[2]: ViT-L-normal bf16, 32 images of ~700 tokens in five aspect ratios on ONE B200 -- encoder tensor-pipe
    roofline.  (a) the reference's only option, same-shape sub-batches (five infer() calls); (b) ragged packing, ONE engine call
    (infer_many): every linear over the concatenated token rows, attention over a ragged work list."""
    from moge.model.v2 import MoGeModel
    from moge_b200.configs import model_config, token_grid
    from moge_b200.synthetic import make_state_dict
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    cfg = model_config("vitl", True)
    model = MoGeModel(**cfg)
    model.load_state_dict(make_state_dict(cfg, 0))
    model = model.to(dev).eval().bfloat16()
    shapes = [(518, 1036, 7), (518, 777, 7), (518, 518, 6), (777, 518, 6), (1036, 518, 6)]      # (H, W, count): grids 19x37 22x32 26x26 32x22 37x19
    tokens = 700
    g = torch.Generator().manual_seed(7)
    batches = [torch.rand(n, 3, H, W, generator=g).to(dev) for (H, W, n) in shapes]
    images = [im for b in batches for im in b]
    grids = [token_grid(H, W, tokens) for (H, W, _) in shapes]
    nimg = len(images)

    def step_bucketed():
        for b in batches:
            model.infer(b, num_tokens=tokens)

    def step_ragged():
        model.infer_many(images, num_tokens=tokens)

    ms_b = _timed_steps(step_bucketed, a.steps, a.warmup)
    ms_r = _timed_steps(step_ragged, a.steps, a.warmup)
    step_ragged()
    cls = _class_times(model)
    pk = peaks()
    enc_t = cls["gemm."][0] + cls["attention"][0]
    enc_f = cls["gemm."][1] + cls["attention"][1]
    # bucketed: sum the classes over the five calls
    enc_tb = enc_fb = 0.0
    for b in batches:
        model.infer(b, num_tokens=tokens)
        c = _class_times(model)
        enc_tb += c["gemm."][0] + c["attention"][0]
        enc_fb += c["gemm."][1] + c["attention"][1]
    line = {
        "metric": "images/sec ViT-L-normal bf16, 32 mixed-aspect ~700-token images (BASELINE.json configs[2])", "value": nimg / (ms_r / 1e3),
        "unit": "images/s", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_r, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "MoGe-2 vitl (normal head) bf16 infer(), 32 images: " + ", ".join(f"{n} x {W}x{H} -> {gh}x{gw}" for (H, W, n), (gh, gw) in zip(shapes, grids))
                               + f" (W x H -> h x w grid), num_tokens={tokens}", "images": nimg},
        "ragged": {"api": "model.infer_many(list of 32 images): ONE engine call, 5 shape groups", "images_per_s": nimg / (ms_r / 1e3), "ms_per_step": ms_r,
                   "encoder": {"tflops": enc_f / enc_t / 1e12, "frac_of_tensor_peak": enc_f / enc_t / 1e12 / pk["tflops"], "ms": enc_t * 1e3,
                               "gemm_tflops": cls["gemm."][1] / cls["gemm."][0] / 1e12, "attention_tflops": cls["attention"][1] / cls["attention"][0] / 1e12}},
        "bucketed": {"api": "five model.infer(same-shape sub-batch) calls (what the reference's API allows)", "images_per_s": nimg / (ms_b / 1e3), "ms_per_step": ms_b,
                     "encoder": {"tflops": enc_fb / enc_tb / 1e12, "frac_of_tensor_peak": enc_fb / enc_tb / 1e12 / pk["tflops"], "ms": enc_tb * 1e3}},
        "roofline": {"bound": "tensor", "achieved": enc_f / enc_t / 1e12, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": enc_f / enc_t / 1e12 / pk["tflops"],
                     "kernel": "encoder (linears + attention) of the ragged call", "traffic": None, "peak_source": pk["source"]},
    }
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)


def run_config5(a):
    """BASELINE.json configs[4]: ViT-B, batch 8 per GPU, long side {256..1024} x aspect {2:1..1:2} x resolution_level {0,5,9}: the
    variable-token encoder + the decoder's HBM roofline.  One row per (H x W, level): (model, dtype, B, HxW, T_req -> h x w), images/s,
    decoder ms and its fraction of the HBM bound by SURVEY.md 8(d)'s byte count."""
    from moge.model.v2 import MoGeModel
    from moge_b200.configs import model_config, token_grid, default_num_tokens
    from moge_b200.synthetic import make_state_dict
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    cfg = model_config("vitb", True)
    model = MoGeModel(**cfg)
    model.load_state_dict(make_state_dict(cfg, 0))
    model = model.to(dev).eval()
    if a.dtype == "bf16":
        model = model.bfloat16()
    pk = peaks()
    B = 8
    rows = []
    g = torch.Generator().manual_seed(11)
    for long_side in (256, 384, 518, 768, 1024):
        for (aw, ah) in ((2, 1), (3, 2), (1, 1), (2, 3), (1, 2)):
            if aw >= ah:
                W, H = long_side, int(round(long_side * ah / aw))
            else:
                H, W = long_side, int(round(long_side * aw / ah))
            x = torch.rand(B, 3, H, W, generator=g).to(dev)
            for level in (0, 5, 9):
                treq = default_num_tokens(cfg["num_tokens_range"], level)
                h, w = token_grid(H, W, treq)
                ms = _timed_steps(lambda: model.infer(x, resolution_level=level), max(2, a.steps // 2), 1)
                c = _class_times(model)
                t_dec, f_dec, b_dec = c["conv"]
                bs = decoder_bytes_survey(768, h * w, B)
                enc_t = c["gemm."][0] + c["attention"][0]
                enc_f = c["gemm."][1] + c["attention"][1]
                rows.append({"model": "vitb", "dtype": a.dtype, "B": B, "HxW": [H, W], "T_req": treq, "grid": [h, w], "images_per_s": B / (ms / 1e3),
                             "ms_per_step": ms, "decoder_ms": t_dec * 1e3, "decoder_gbs_survey_bytes": bs / t_dec / 1e9,
                             "decoder_frac_hbm": bs / t_dec / 1e9 / pk["hbm_gbs"], "decoder_tflops": f_dec / t_dec / 1e12,
                             "decoder_frac_of_max_bound": max(f_dec / (pk["tflops"] * 1e12), bs / (pk["hbm_gbs"] * 1e9)) / t_dec,
                             "encoder_tflops": enc_f / enc_t / 1e12, "encoder_frac": enc_f / enc_t / 1e12 / pk["tflops"]})
            del x
    tot_img = sum(r["B"] for r in rows)
    tot_s = sum(r["ms_per_step"] for r in rows) / 1e3
    dec_t = sum(r["decoder_ms"] for r in rows) / 1e3
    dec_b = sum(decoder_bytes_survey(768, r["grid"][0] * r["grid"][1], r["B"]) for r in rows)
    line = {
        "metric": "images/sec ViT-B resolution/aspect sweep, batch 8 (BASELINE.json configs[4])", "value": tot_img / tot_s, "unit": "images/s", "n_gpus": 1,
        "steps": max(2, a.steps // 2), "warmup": 1, "ms_per_step": 1e3 * tot_s / len(rows), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": a.dtype, "data": "synthetic",
        "config": {"workload": "MoGe-2 vitb* (SURVEY.md 8 test config) infer(), B=8, long side {256,384,518,768,1024} x aspect {2:1,3:2,1:1,2:3,1:2} x "
                               "resolution_level {0,5,9}; value = total images / total time over the 75 rows", "rows": len(rows)},
        "roofline": {"bound": "hbm", "achieved": dec_b / dec_t / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": dec_b / dec_t / 1e9 / pk["hbm_gbs"],
                     "kernel": "decoder conv launches over the whole sweep", "bytes_definition": "SURVEY.md 8(d), 997376 B x T per image", "traffic": None,
                     "peak_source": pk["source"]},
        "rows": rows,
    }
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.config == 3:
        run_config3(args)
    elif args.config == 5:
        run_config5(args)
    else:
        run_engine(args)
