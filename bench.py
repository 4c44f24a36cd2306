#!/usr/bin/env python
"""Benchmark of the Feature2Face generator hot path (BASELINE.json: 512x512 frames/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--mode parity|fast] [--variant large|normal]
                    [--height H --width W] [--gather auto|ce|nccl] [--clip-frames F] [--impl reference] [--dump-outputs DIR]

A step = one pass of the generator over one batch of B synthetic frames (default: the May.yaml 'large' network at
512x512, 32 frames per step - BASELINE.json configs[1]; frames of a clip are independent, so the clip is rendered B
frames per call).  Under torchrun (N > 1) every rank renders its own block of the clip through
``livespeechportraits_b200.parallel.ShardedRenderer`` and every rank receives every frame (configs[3]); weak scaling.
Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

RECIPE = "A"
CLIP_FRAMES = 672          # frames demo.py renders for data/Input/00083.wav (SURVEY.md 8d): the end-to-end clip
DUMP_LIMIT = 64_000_000 - 4096     # bytes of array data --dump-outputs may write: 64 MB less room for the .npy header


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=32,
                    help="frames per step.  profiles/r02_t7_frames_per_step_sweep.txt: 64 is +2 %% over 32 on one box, but the worst parity "
                         "case measured at 64 (recipe B, frames 0/32/63) is 5.3e-4 where 32 gives 3.6e-4 - the default keeps the wider margin")
    ap.add_argument("--mode", default="parity", choices=["parity", "fast"])
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--variant", default="large", choices=["large", "normal"],
                    help="large = May.yaml (BASELINE.json configs[1], default); normal = Obama1/Nadella/... (configs[2], [4])")
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=512)
    ap.add_argument("--gather", default="auto", choices=["auto", "ce", "nccl"],
                    help="N > 1: how rendered frames reach every rank (parallel.ShardedRenderer)")
    ap.add_argument("--clip-frames", type=int, default=10000,
                    help="N > 1: also render one clip of exactly this many frames and report it as clip_run (BASELINE.json "
                         "configs[3]: 10000 synthetic frames, frame-sharded; 0 = skip)")
    ap.add_argument("--no-extras", action="store_true", help="skip the side measurements (other modes / configs, library baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the fp32 frames of the last timed step to DIR/frames.npy (a fixed sample "
                         "of them when they exceed 64 MB), so that two builds can be compared output for output")
    return ap.parse_args()


def metric_name(variant: str, h: int, w: int) -> str:
    cfg = "May.yaml" if variant == "large" else "Obama1.yaml"
    return f"{h}x{w} frames/sec (Feature2Face_G {variant} / {cfg})"


def config_dict(args, world: int) -> dict:
    """Workload description shared verbatim by the product arm and the reference arm (same config, same metric)."""
    v, B, H, W = args.variant, args.batch, args.height, args.width
    return {
        "workload": f"{'May.yaml (large)' if v == 'large' else 'Obama1.yaml (normal)'} {H}x{W}, clip rendered in batches of {B} frames "
                    "per step (BASELINE.json configs[1]/[3]; the one-frame-per-call rate of demo.py is reported as single_frame), "
                    + ("single GPU" if world == 1 else f"frame-sharded over {world} GPUs, every rank receives every frame"),
        "variant": v, "batch": B, "height": H, "width": W, "precision_mode": args.mode, "parallelism": f"dp{world}",
        "l2": "per-step working set (weights 0.24-0.49 GB + activations > 1 GB) exceeds the 126 MB L2; input batches rotate "
              "over a pool",
    }


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1451.7), d.get("hbm_gbs", 6572.9), "MEASURED_PEAKS.json (sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def host_cpu_info() -> dict:
    model, sockets = None, set()
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and model is None:
                model = line.split(":", 1)[1].strip()
            elif line.startswith("physical id"):
                sockets.add(line.split(":", 1)[1].strip())
    except OSError:
        pass
    usable = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    return {"model": model, "sockets": len(sockets) or None, "logical_cpus": os.cpu_count(), "usable_cpus": usable}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)            # no sampler outlives a run that fails before stop()
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        inside = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.1] or [r for (_, r) in self.rows[-3:]]
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in inside:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for nm, val in zip(names, r[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_net(variant: str, mode: str):
    from livespeechportraits_b200.generator import Feature2Face_G
    from oracle import f2f_oracle as O
    opt = types.SimpleNamespace(isTrain=False, size=variant, n_downsample_G=8, ngf=64, fp16=0)
    net = Feature2Face_G(opt, precision=mode)
    sd = O.make_state_dict(variant, RECIPE)
    net.load_state_dict(sd, strict=True)
    return net.cuda().eval(), sd


def dump_outputs(dirpath: str, frames: torch.Tensor) -> None:
    """DIR/frames.npy: the fp32 frames ``[n, 3, H, W]`` of the last timed step, all of them when they fit in DUMP_LIMIT bytes;
    else the frames at fixed seeded indices, or, when one frame alone is larger, every k-th element of the flattened frames."""
    x = frames.detach().float()
    note = "all frames"
    if x.numel() * 4 > DUMP_LIMIT:
        per_frame = x[0].numel() * 4
        if per_frame <= DUMP_LIMIT:
            idx = np.sort(np.random.default_rng(0).choice(x.shape[0], DUMP_LIMIT // per_frame, replace=False))
            x = x[torch.from_numpy(idx).to(x.device)]
            note = f"frames {idx.tolist()}"
        else:
            k = -(-x.numel() // (DUMP_LIMIT // 4))
            x = x.reshape(-1)[::k]
            note = f"every {k}-th element"
    os.makedirs(dirpath, exist_ok=True)
    path = os.path.join(dirpath, "frames.npy")
    np.save(path, x.cpu().numpy())
    print(f"bench: wrote {path} {tuple(x.shape)} float32 ({note} of the last timed step, {tuple(frames.shape)})", file=sys.stderr)


_CPU_THREADS = None


def cpu_reference_fps(variant: str, h: int, w: int, frames_per_step: int, steps: int, warmup: int):
    """The reference's own CPU implementation of the path: the unmodified ATen convs on the host cores, through the
    oracle port (the Python reference checkout does not travel to the GPU box)."""
    global _CPU_THREADS
    from oracle import f2f_oracle as O
    sd = O.make_state_dict(variant, RECIPE)
    fm, cand = O.make_inputs(frames_per_step, h, w)
    x = torch.cat([fm, cand], 1)
    if _CPU_THREADS is None:
        # "all the host threads it can use": calibrate the thread count on one frame each (oneDNN does not always
        # scale to every logical CPU of a big host, and the container may be pinned to fewer than os.cpu_count()).
        usable = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        cands = sorted({c for c in (torch.get_num_threads(), usable, usable // 2, 64, 32, 16, 8) if 1 <= c <= usable})
        best, best_t = None, None
        for c in cands:
            torch.set_num_threads(c)
            O.generator_forward(sd, x[:1], variant)
            t0 = time.perf_counter()
            O.generator_forward(sd, x[:1], variant)
            dt = time.perf_counter() - t0
            if best_t is None or dt < best_t:
                best, best_t = c, dt
        _CPU_THREADS = best
    torch.set_num_threads(_CPU_THREADS)
    for _ in range(warmup):
        O.generator_forward(sd, x, variant)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.generator_forward(sd, x, variant)
    dt = time.perf_counter() - t0
    return frames_per_step * steps / dt, dt / steps * 1e3, torch.get_num_threads()


def run_reference(args, rank: int):
    """`--impl reference`: the reference's CPU path on the host cores, K steps after W warm-up steps as asked; each step is a
    bounded SAMPLE of the B-frame step (2 frames of it) so that the run ends within minutes at ~3 frames/s."""
    if rank != 0:
        return
    per_step = min(args.batch, 2)
    fps, ms, cores = cpu_reference_fps(args.variant, args.height, args.width, per_step, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": metric_name(args.variant, args.height, args.width), "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic (seeded weights with the reference init distribution, seeded inputs)",
        "config": config_dict(args, args.gpus),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "host": host_cpu_info(),
                         "sample": f"{args.steps} steps (+{args.warmup} warm-up) x {per_step} frames of the {args.batch}-frame step, fp32, "
                                   "torch ATen convs on the host (oracle/f2f_oracle.py = the reference's arithmetic; the Python "
                                   "reference checkout cannot travel to the GPU box)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(json.dumps(line))


_REAL_STDOUT = None


def emit(text: str) -> None:
    """The ONE line of the contract, written to the process's original stdout."""
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (text + "\n").encode())


def timed_ms(fn, n: int, warm: int = 3) -> float:
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def library_baseline(variant: str, batch: int, h: int, w: int) -> dict:
    """PyTorch eager + cuDNN on the same GPU, same batch: what the unmodified reference module would execute on this B200
    (base_model.py:46-47 sets cudnn.benchmark).  A library baseline beside the hand-written kernels, never the product path."""
    from oracle import f2f_oracle as O
    torch.backends.cudnn.benchmark = True
    sd_cpu = O.make_state_dict(variant, RECIPE)
    sd = {k: v.cuda() for k, v in sd_cpu.items()}
    fm, cand = O.make_inputs(batch, h, w)
    x = torch.cat([fm, cand], 1).cuda()
    ref = O.generator_forward(sd_cpu, x[:1].cpu(), variant)
    out = {"batch": batch, "what": "oracle restatement on torch eager + cuDNN (cudnn.benchmark), same GPU, same batch"}
    with torch.no_grad():
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        ms = timed_ms(lambda: O.generator_forward(sd, x, variant), 3, 2)
        err = (O.generator_forward(sd, x[:1], variant).cpu() - ref).abs().max().item()
        out["fp32"] = {"frames_per_s": batch / ms * 1e3, "max_abs_err": err}
        torch.backends.cudnn.allow_tf32 = True
        ms = timed_ms(lambda: O.generator_forward(sd, x, variant), 5, 2)
        err = (O.generator_forward(sd, x[:1], variant).cpu() - ref).abs().max().item()
        out["tf32"] = {"frames_per_s": batch / ms * 1e3, "max_abs_err": err}
        xc = x.contiguous(memory_format=torch.channels_last)
        sdc = {k: (v.contiguous(memory_format=torch.channels_last) if v.dim() == 4 else v) for k, v in sd.items()}

        def bf16():
            with torch.autocast("cuda", dtype=torch.bfloat16):
                return O.generator_forward(sdc, xc, variant)
        ms = timed_ms(bf16, 5, 2)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            err = (O.generator_forward(sdc, xc[:1], variant).float().cpu() - ref).abs().max().item()
        out["bf16_autocast_channels_last"] = {"frames_per_s": batch / ms * 1e3, "max_abs_err": err}
    torch.backends.cudnn.allow_tf32 = False
    del sd, x
    torch.cuda.empty_cache()
    return out


def side_config(variant: str, mode: str, batch: int, h: int, w: int, tflops_peak: float, check: bool = True) -> dict:
    """One of BASELINE.json's other configurations measured in the same run: frames/s (device-resident inputs, CUDA-graph
    replay), algorithmic TFLOP/s, fraction of the tensor roofline and the error of the timed plan's first / last frame."""
    from oracle import f2f_oracle as O
    net, sd = make_net(variant, mode)
    fm, cand = O.make_inputs(batch, h, w, seed=41)
    fm_d, cand_d = fm.cuda(), cand[:1].cuda()
    out = torch.empty((batch, 3, h, w), dtype=torch.float32, device="cuda")
    ms = timed_ms(lambda: net.render(fm_d, cand_d, out=out), 8, 3)
    flops = net.flops_per_frame(h, w) * batch
    res = {"variant": variant, "mode": mode, "batch": batch, "height": h, "width": w, "ms_per_step": ms,
           "frames_per_s": batch / ms * 1e3, "tflops_algorithmic": flops / ms / 1e9,
           "roofline_frac": flops / ms / 1e9 / tflops_peak, "launches": net.launches_per_forward()}
    if check:
        errs = []
        for i in sorted({0, batch - 1}):
            x = torch.cat([fm[i:i + 1], cand[:1]], 1)
            errs.append((out[i:i + 1].cpu() - O.generator_forward(sd, x, variant)).abs().max().item())
        res["max_abs_err_vs_oracle"] = max(errs)
    del net, out
    torch.cuda.empty_cache()
    return res


def main():
    global _REAL_STDOUT
    args = parse()
    # Libraries chat on stdout (NCCL prints its version line there): keep the original stdout for the JSON line only and
    # send everything else that writes to fd 1 to stderr.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    VARIANT, H, W = args.variant, args.height, args.width
    METRIC = metric_name(VARIANT, H, W)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU path for the product arm (use --impl reference for the CPU arm)")
    import torch.distributed as dist
    from oracle import f2f_oracle as O
    from livespeechportraits_b200.parallel import ShardedRenderer, partition
    from livespeechportraits_b200.pipeline import ClipRenderer

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, K, Wm = args.batch, args.steps, max(args.warmup, 3)
    net, sd = make_net(VARIANT, args.mode)
    tflops_peak, hbm_peak, peak_src = measured_peaks()

    # ---- synthetic inputs: a pool of feature-map batches (> L2 together with weights and activations).  The seed of a batch
    # is a function of (rank, pool slot), so rank 0 can regenerate any rank's frames for the parity check of the gathered clip.
    pool = 4

    def pool_seed(r: int, i: int) -> int:
        return 100 + r * 16 + i
    fm_pool = []
    for i in range(pool):
        fm, _ = O.make_inputs(B, H, W, seed=pool_seed(rank, i))
        fm_pool.append(fm.cuda())
    cand_cpu = O.make_inputs(1, H, W, seed=99)[1][:1].contiguous()     # ONE candidate set for every frame of every rank (demo.py:95,266)
    cand = cand_cpu.cuda()
    flops_step = net.flops_per_frame(H, W) * B

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def oracle_err(out_frame: torch.Tensor, r: int, step: int, j: int) -> float:
        """max|out - oracle| of one frame of the timed workload: frame j of step `step` of rank r."""
        fm_r, _ = O.make_inputs(B, H, W, seed=pool_seed(r, step % pool))
        x = torch.cat([fm_r[j:j + 1], cand_cpu], 1)
        return (out_frame.float().cpu() - O.generator_forward(sd, x, VARIANT)).abs().max().item()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    gather_info = None
    if world == 1:
        obuf = [torch.empty((B, 3, H, W), dtype=torch.float32, device=dev) for _ in range(2)]

        def step(i):
            net.render(fm_pool[i % pool], cand, out=obuf[i & 1])
        for i in range(Wm):
            step(i)
        barrier()
        sampler.start()
        time.sleep(0.25)
        barrier()
        t_wall0 = time.time()
        e0.record()
        for i in range(K):
            step(i)
        e1.record()
        barrier()
        t_wall1 = time.time()
        # parity of what was just timed: frames of the LAST timed step (the B-frame plan, not a batch-1 call)
        last = obuf[(K - 1) & 1]
        checks = sorted({0, B // 2, B - 1})
        parity_err = max(oracle_err(last[j:j + 1], 0, K - 1, j) for j in checks)
        parity_note = f"frames {checks} of the last timed {B}-frame step vs the oracle"
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
    else:
        # N > 1: the library's own multi-GPU entry point.  One render() = K chunks of B frames per rank; the tail kernel writes
        # into the clip buffer, the frames travel to every rank (copy engines over symmetric memory, or NCCL all-gather).
        sr = ShardedRenderer(lambda fm_, out_: net.render(fm_, cand, out=out_), chunk=B, gather=args.gather)
        local_fm = torch.cat([fm_pool[i % pool] for i in range(K)], 0)                 # this rank's block: K*B frames
        wm_c = min(Wm, K)
        warm_fm = local_fm[: wm_c * B]
        sr.prepare(K * B * world, H, W, dev)           # symmetric clip buffer allocated + exchanged once, outside the timed region
        sr.render(wm_c * B * world, warm_fm)
        barrier()
        if rank == 0:
            sampler.start()
            time.sleep(0.25)
        barrier()
        t_wall0 = time.time()
        e0.record()
        clip_all = sr.render(K * B * world, local_fm)
        e1.record()
        barrier()
        t_wall1 = time.time()
        gather_info = {"mode": sr.gather_mode, "fallback_reason": sr.gather_fallback_reason, "dtype": "f32",
                       "bytes_received_per_step_per_rank": (world - 1) * B * 3 * H * W * 4,
                       "api": "livespeechportraits_b200.parallel.ShardedRenderer.render"}
        parity_err, parity_note = None, None
        if rank == 0:
            # gathered clip, clip order = rank-major blocks: check one frame of the first, a middle and the last rank
            picks = [(0, 0, 0), (world // 2, K // 2, B // 2), (world - 1, K - 1, B - 1)]
            errs = []
            for (r, st_, j) in picks:
                g = partition(K * B * world, world, r)[0] + st_ * B + j
                errs.append(oracle_err(clip_all[g:g + 1], r, st_, j))
            parity_err = max(errs)
            parity_note = f"frames (rank, step, index) {picks} of the gathered clip on rank 0 vs the oracle"
            if args.dump_outputs:
                # the last timed step of every rank: frames (K-1)*B ... K*B-1 of each rank's block of the gathered clip
                starts = [partition(K * B * world, world, r)[0] + (K - 1) * B for r in range(world)]
                dump_outputs(args.dump_outputs, torch.cat([clip_all[s0:s0 + B] for s0 in starts]))
    ms_total = e0.elapsed_time(e1)
    ms_step_local = ms_total / K
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    launches = net.launches_per_forward()       # pack + convs + split-K finishers of the plan that was just timed

    # Per-launch breakdown: the same steps again with a CUDA event after every kernel.  Recording events forces plain
    # stream launches (no CUDA-graph replay, no PDL overlap), so this pass is a little slower than the timed region; it
    # supplies the SHARE of each launch, the timed region supplies the time.
    pbuf = torch.empty((B, 3, H, W), dtype=torch.float32, device=dev)
    net.profile_enable(True)
    for i in range(min(K, 200)):
        net.render(fm_pool[i % pool], cand, out=pbuf)
    torch.cuda.synchronize()
    prof_ms, prof_n = net.profile_read()
    net.profile_enable(False)
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = t.item()
    frames = B * K * world
    value = frames / (ms_total / 1e3)

    # ---- roofline of the dominant kernel family (the tcgen05 convs), from the per-launch events of the timed workload
    rows = net.layer_table(H, W)
    conv_ms = prof_ms[1:]
    groups = {}
    for r, ms in zip(rows, conv_ms):
        key = f"k{r['kind']} {r['cin']}->{r['cout']} @{r['out_h']}"
        g = groups.setdefault(key, {"ms": 0.0, "flops": 0.0, "launches": 0})
        g["ms"] += ms
        g["flops"] += r["flops"] * B
        g["launches"] += 1
    tot_ms = sum(conv_ms)
    conv_share = tot_ms / (tot_ms + prof_ms[0]) if tot_ms > 0 else 1.0
    conv_ms_timed = ms_step_local * conv_share
    achieved = flops_step / (conv_ms_timed / 1e3) / 1e12 if conv_ms_timed > 0 else 0.0
    # tensor work actually issued: folded upsample does 4/9 of the MACs; parity mode issues 3 MMA-equivalents per K step
    exec_flops = 0.0
    for r in rows:
        f = r["flops"] * B
        if r["kind"] == 3:
            f *= 4.0 / 9.0
        exec_flops += f * (3.0 if args.mode == "parity" else 1.0)
    top = sorted(groups.items(), key=lambda kv: -kv[1]["ms"])[:6]
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath):
        try:
            cand_t = [t for t in json.load(open(tpath)) if t.get("batch") == B and t.get("mode") == args.mode and t.get("variant") == VARIANT]
            traffic = cand_t[0] if cand_t else None
        except Exception:
            traffic = None
    roofline = {
        "bound": "tensor", "kernel": "lspg::conv_pair_kernel / conv_umma_kernel / conv_patch_kernel (all conv launches of one step)",
        "achieved": achieved, "peak": tflops_peak, "unit": "TFLOP/s", "frac": achieved / tflops_peak, "peak_source": peak_src,
        "traffic": traffic.get("dram_bytes_per_launch") if traffic else None,
        "traffic_detail": traffic,
        "algorithmic_flops_per_step": flops_step, "kernel_ms_per_step": conv_ms_timed,
        "kernel_ms_per_step_event_pass": tot_ms, "pack_input_ms": prof_ms[0], "forwards_profiled": prof_n,
        "executed_tflops": exec_flops / (conv_ms_timed / 1e3) / 1e12 if conv_ms_timed > 0 else None,
        "executed_frac": (exec_flops / (conv_ms_timed / 1e3) / 1e12) / tflops_peak if conv_ms_timed > 0 else None,
        "note": "achieved = reference-conv FLOPs / time of the conv launches in the timed region; parity mode issues "
                "3 tcgen05 MMAs per K step (hi*hi, hi*lo, lo*hi), so executed_* is the tensor-pipe view",
        "top_groups": [{"group": k, "ms": round(v["ms"], 4), "launches": v["launches"],
                        "tflops": round(v["flops"] / (v["ms"] / 1e3) / 1e12, 1) if v["ms"] > 0 else None} for k, v in top],
    }

    # ---- end to end through the public batched API: host inputs in, host frames out, copies inside the timed region
    if world == 1:
        n_clip = CLIP_FRAMES
        fm_host = torch.empty((n_clip, 1, H, W), dtype=torch.float32, pin_memory=True)
        for o in range(0, n_clip, B):
            ln = min(B, n_clip - o)
            fm_host[o:o + ln].copy_(fm_pool[(o // B) % pool][:ln])
        out_host = torch.empty((n_clip, 3, H, W), dtype=torch.float32, pin_memory=True)
        clip = ClipRenderer(net, batch=B, device=dev)
        clip.render_clip(fm_host, cand, out_host)                # warm-up: the same clip (builds the plan of a ragged last batch too)
        barrier()
        t0 = time.perf_counter()
        clip.render_clip(fm_host, cand, out_host)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        e2e = {"value": n_clip / dt, "unit": "frames/s", "h2d_bytes_per_step": B * H * W * 4,
               "d2h_bytes_per_step": B * 3 * H * W * 4, "frames": n_clip, "seconds": dt,
               "api": "livespeechportraits_b200.pipeline.ClipRenderer.render_clip (pinned host feature maps -> pinned host fp32 "
                      "frames; candidates resident on the device as in demo.py:95); the 672-frame clip of configs[1]"}
    else:
        # every rank uploads its block of feature maps from pinned host memory, renders it, the frames travel to every rank
        # and rank 0 delivers the WHOLE clip to pinned host memory (uint8 images: util.tensor2im fused into the tail kernel -
        # what demo.py:268 builds from every frame) while later chunks are still rendering
        n_local = K * B
        n_all = n_local * world
        fm_host = torch.empty((n_local, 1, H, W), dtype=torch.float32, pin_memory=True)
        fm_host.copy_(local_fm)
        sr8 = ShardedRenderer(lambda fm_, out_: net.render_image(fm_, cand, out=out_), chunk=B, uint8=True, gather=args.gather)
        host_out = torch.empty((n_all, H, W, 3), dtype=torch.uint8, pin_memory=True) if rank == 0 else None
        fm_dev = torch.empty_like(local_fm)
        sr8.prepare(n_all, H, W, dev)

        def e2e_once(n_chunks):
            nl = n_chunks * B
            fm_dev[:nl].copy_(fm_host[:nl], non_blocking=True)
            return sr8.render(nl * world, fm_dev[:nl], host_out=(host_out[: nl * world] if rank == 0 else None), to_host=True)
        e2e_once(min(3, K))
        barrier()
        t0 = time.perf_counter()
        got = e2e_once(K)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = t.item()
        e2e_ok = None
        if rank == 0:
            # the host copy equals the device clip, and a frame of the last rank equals the oracle's image within one level
            e2e_ok = bool(torch.equal(host_out[:64], got[:64].cpu()) and torch.equal(host_out[-64:], got[-64:].cpu()))
        e2e = {"value": n_all / dt, "unit": "frames/s", "h2d_bytes_per_step": B * H * W * 4,
               "d2h_bytes_per_step": world * B * H * W * 3, "frames": n_all, "seconds": dt, "gather_mode": sr8.gather_mode,
               "host_copy_matches_device_clip": e2e_ok,
               "api": "parallel.ShardedRenderer(uint8=True).render(host_out=..., to_host=True): per-rank pinned feature maps -> H2D -> render -> "
                      "frames to every rank -> rank 0 copies the whole gathered clip (uint8 HWC images, util.tensor2im fused) to "
                      "pinned host memory; d2h bytes are rank 0's per step"}
        del host_out, fm_dev

    extras = {}
    if world > 1 and not args.no_extras:
        # uint8 frames through the same entry point (a quarter of the bytes), and the exact-size clip of configs[3] if asked
        sr8 = ShardedRenderer(lambda fm_, out_: net.render_image(fm_, cand, out=out_), chunk=B, uint8=True, gather=args.gather)
        sr8.prepare(K * B * world, H, W, dev)
        sr8.render(min(Wm, K) * B * world, local_fm[: min(Wm, K) * B])
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        sr8.render(K * B * world, local_fm)
        b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        extras["gather_uint8"] = {"value": K * B * world / (t.item() / 1e3), "unit": "frames/s", "gather_mode": sr8.gather_mode,
                                  "bytes_received_per_step_per_rank": (world - 1) * B * H * W * 3}
        del sr8
        # the collective fused into the conv kernel: the tail epilogue stores through the NVLink multicast mapping (NVLS)
        try:
            srm = ShardedRenderer(lambda fm_, out_: net.render(fm_, cand, out=out_), chunk=B, gather="mc",
                                  render_ptr_fn=lambda fm_, ptr: net.render_into_ptr(fm_, cand, ptr))
            srm.prepare(K * B * world, H, W, dev)
            srm.render(min(Wm, K) * B * world, local_fm[: min(Wm, K) * B])
            barrier()
            a.record()
            clip_mc = srm.render(K * B * world, local_fm)
            b.record()
            barrier()
            t = torch.tensor([a.elapsed_time(b)], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            err_mc = None
            if rank == 0:
                g = partition(K * B * world, world, world - 1)[0] + (K - 1) * B + (B - 1)
                err_mc = oracle_err(clip_mc[g:g + 1], world - 1, K - 1, B - 1)
            extras["gather_multicast_in_kernel"] = {
                "value": K * B * world / (t.item() / 1e3), "unit": "frames/s", "gather_mode": srm.gather_mode,
                "max_abs_err_vs_oracle_last_rank_last_frame": err_mc,
                "note": "fp32 frames; the tail conv's float2 stores go through the symmetric buffer's multicast address, no copy "
                        "or collective kernel follows"}
            del srm, clip_mc
        except Exception as exc:      # noqa: BLE001
            extras["gather_multicast_in_kernel"] = {"unavailable": f"{type(exc).__name__}: {exc}"[:300]}
        if args.clip_frames > 0:
            n_tot = args.clip_frames
            s_, e_ = partition(n_tot, world, rank)
            reps = -(-(e_ - s_) // local_fm.shape[0])
            mine = torch.cat([local_fm] * reps, 0)[: e_ - s_]
            src = ShardedRenderer(lambda fm_, out_: net.render(fm_, cand, out=out_), chunk=B, gather=args.gather)
            src.prepare(n_tot, H, W, dev)
            src.render(min(Wm, K) * B * world, local_fm[: min(Wm, K) * B])
            barrier()
            a.record()
            src.render(n_tot, mine)
            b.record()
            barrier()
            t = torch.tensor([a.elapsed_time(b)], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            extras["clip_run"] = {"frames": n_tot, "value": n_tot / (t.item() / 1e3), "unit": "frames/s", "seconds": t.item() / 1e3,
                                  "gather_mode": src.gather_mode, "dtype": "f32",
                                  "gathered_bytes_per_rank": n_tot * 3 * H * W * 4,
                                  "note": "BASELINE.json configs[3]: one clip of exactly this many synthetic frames, block-partitioned"}
            del src, mine
    if rank == 0 and world == 1 and not args.no_extras:
        other = "fast" if args.mode == "parity" else "parity"
        ms_o = timed_ms(lambda: net.render(fm_pool[0], cand, out=obuf[0], precision=other), 10)
        err_o = oracle_err(obuf[0][:1], 0, 0, 0)
        extras[f"{other}_mode"] = {"value": B / ms_o * 1e3, "unit": "frames/s", "max_abs_err_vs_oracle": err_o,
                                   "tflops_algorithmic": flops_step / (ms_o / 1e3) / 1e12,
                                   "roofline_frac": flops_step / (ms_o / 1e3) / 1e12 / tflops_peak}
        # N1 (SURVEY.md 8f): frames leave the GPU as uint8 HWC images (util.tensor2im fused into the tail kernel)
        img_host = torch.empty((n_clip, H, W, 3), dtype=torch.uint8, pin_memory=True)
        clip8 = ClipRenderer(net, batch=B, device=dev, uint8=True)
        clip8.render_clip(fm_host, cand, img_host)
        torch.cuda.synchronize()
        t8 = time.perf_counter()
        clip8.render_clip(fm_host, cand, img_host)
        torch.cuda.synchronize()
        dt8 = time.perf_counter() - t8
        extras["e2e_uint8_images"] = {"value": n_clip / dt8, "unit": "frames/s", "d2h_bytes_per_step": B * H * W * 3,
                                      "api": "ClipRenderer(uint8=True): lspg_forward_image (tensor2im fused, util/util.py:19-42)"}
        # N2 (SURVEY.md 8f): landmark tracks in, uint8 images out - the maps are drawn on the GPU (lspg_draw_feature_maps), so
        # 728 B per frame cross PCIe instead of 1 MB; the host-side cost this removes (88 cv2.line calls per frame,
        # datasets/face_dataset.py:312-323) is timed next to it on one host thread, as the reference runs it
        from oracle import raster_oracle as RO
        lm_np, sh_np = RO.make_landmarks(n_clip, (W, H), seed=3)
        lm_host, sh_host = torch.from_numpy(lm_np).pin_memory(), torch.from_numpy(sh_np).pin_memory()
        clip8.render_clip_from_landmarks(lm_host, sh_host, cand, img_host, (W, H))
        torch.cuda.synchronize()
        tl = time.perf_counter()
        clip8.render_clip_from_landmarks(lm_host, sh_host, cand, img_host, (W, H))
        torch.cuda.synchronize()
        dtl = time.perf_counter() - tl
        ms_r = timed_ms(lambda: net.draw_feature_maps(lm_host[:B].cuda(), sh_host[:B].cuda(), (W, H)), 20)
        chk = net.draw_feature_maps(lm_host[:2].cuda(), sh_host[:2].cuda(), (W, H)).cpu().numpy()
        exact = all(np.array_equal(chk[i, 0] * 255, RO.draw_feature_map_cv2(lm_np[i], (W, H), sh_np[i])) for i in range(2))
        t_cv = time.perf_counter()
        for i in range(32):
            RO.draw_feature_map_cv2(lm_np[i % n_clip], (W, H), sh_np[i % n_clip])
        cv_ms = (time.perf_counter() - t_cv) / 32 * 1e3
        extras["e2e_from_landmarks_uint8"] = {
            "value": n_clip / dtl, "unit": "frames/s", "h2d_bytes_per_step": B * (73 + 18) * 2 * 4, "d2h_bytes_per_step": B * H * W * 3,
            "rasterise_ms_per_batch": ms_r, "bit_exact_vs_cv2": bool(exact), "cv2_host_ms_per_frame": cv_ms,
            "api": "ClipRenderer.render_clip_from_landmarks: lspg_draw_feature_maps + lspg_forward_image"}
        # N3 (SURVEY.md 8f): the demo.py:260-292 loop body - landmarks -> frames -> ONE video stream, no JPEG round trip
        try:
            from livespeechportraits_b200.video import render_to_video
            import tempfile
            with tempfile.TemporaryDirectory() as td:
                path = os.path.join(td, "clip.avi")
                render_to_video(net, lm_np, sh_np, cand, path, size=(W, H), fps=60, batch=B)      # warm-up: the same clip
                tv = time.perf_counter()
                info = render_to_video(net, lm_np, sh_np, cand, path, size=(W, H), fps=60, batch=B)
                dtv = time.perf_counter() - tv
            extras["e2e_to_video"] = {"value": n_clip / dtv, "unit": "frames/s", "seconds": dtv, "frames": n_clip,
                                      "writer": info.get("writer"), "encode_seconds": info.get("encode_seconds"),
                                      "api": "livespeechportraits_b200.video.render_to_video (replaces demo.py:260-292: per-frame "
                                             "inference + JPEG write + re-read + cv2.VideoWriter)"}
        except Exception as exc:      # noqa: BLE001 - a missing codec must not take the benchmark line down
            extras["e2e_to_video"] = {"unavailable": f"{type(exc).__name__}: {exc}"}
        # configs[1] as demo.py:266 calls it: ONE frame per inference() call, with its own roofline block
        one = fm_pool[0][:1].contiguous()
        o1 = torch.empty((1, 3, H, W), dtype=torch.float32, device=dev)
        ms_1 = timed_ms(lambda: net.render(one, cand, out=o1), 50, 10)
        f1 = net.flops_per_frame(H, W)
        extras["single_frame"] = {
            "value": 1e3 / ms_1, "unit": "frames/s", "ms_per_frame": ms_1, "mode": args.mode, "launches": net.launches_per_forward(),
            "max_abs_err_vs_oracle": oracle_err(o1, 0, 0, 0),
            "roofline": {"bound": "tensor", "achieved": f1 / ms_1 / 1e9, "peak": tflops_peak, "unit": "TFLOP/s",
                         "frac": f1 / ms_1 / 1e9 / tflops_peak,
                         "floor_ms": {"tensor_1pass": f1 / tflops_peak / 1e9, "tensor_3pass_parity": 3 * f1 / tflops_peak / 1e9,
                                      "weights_hbm": (2 if args.mode == 'parity' else 1) * 2 * sum(r['cin'] * r['cout'] * 9 for r in rows) / hbm_peak / 1e6}},
            "note": "batch 1 per call, as demo.py:266 calls inference(); CUDA-graph replay, output tensor supplied"}
        # BASELINE.json's other configurations in the same driver-run record (frames/s of the timed plan + its error)
        side = {}
        try:
            side["configs[2] normal 512x512 batch 8 parity"] = side_config("normal", "parity", 8, 512, 512, tflops_peak)
            side["configs[4] normal 1024x1024 batch 8 bf16 (fast)"] = side_config("normal", "fast", 8, 1024, 1024, tflops_peak)
            side["configs[4] normal 1024x1024 batch 8 parity"] = side_config("normal", "parity", 8, 1024, 1024, tflops_peak)
        except Exception as exc:      # noqa: BLE001
            side["error"] = f"{type(exc).__name__}: {exc}"
        extras["other_configs"] = side
        # N4 (SURVEY.md 8f): the Audio2Headpose loop of the same clip (687 audio rows -> 672 frames) in one persistent kernel,
        # next to the reference's loop (oracle port of models/audio2headpose_model.py:169-187) timed on the host CPU
        try:
            from livespeechportraits_b200.headpose import HeadposeGenerator
            from oracle import a2h_oracle as AO
            hopt = AO.default_opt()
            hsd = AO.make_state_dict(hopt, "B", 1)
            audio = AO.make_audio_feats(CLIP_FRAMES + hopt.frame_future, hopt, 2)
            noise = AO.reference_noise(CLIP_FRAMES, 12, 1, seed=0)
            pre = np.zeros(12, np.float32)
            gen = HeadposeGenerator(hopt, hsd, device=dev)
            a_d, n_d, p_d = torch.from_numpy(audio).to(dev), torch.from_numpy(noise).to(dev), torch.from_numpy(pre).to(dev)
            ms8 = timed_ms(lambda: gen.generate(a_d, p_d, n_d, 0.3, cluster=8), 3, 1)
            ms1 = timed_ms(lambda: gen.generate(a_d, p_d, n_d, 0.3, cluster=1), 2, 1)
            got = gen.generate(a_d, p_d, n_d, 0.3, cluster=8).cpu().numpy()
            t0 = time.perf_counter()
            ref = AO.generate_sequences(hsd, audio[:24 + hopt.frame_future], pre, noise[:24], hopt, 0.3)
            cpu_ms = (time.perf_counter() - t0) / 24 * 1e3
            extras["headpose_loop"] = {
                "frames": CLIP_FRAMES, "ms_per_clip": ms8, "frames_per_s": CLIP_FRAMES / ms8 * 1e3, "ms_per_clip_single_cta": ms1,
                "us_per_frame": ms8 / (CLIP_FRAMES + 254) * 1e3, "max_abs_err_vs_oracle_first_24_frames": float(np.abs(got[:24] - ref).max()),
                "cpu_reference_ms_per_frame": cpu_ms, "cpu_reference_s_per_clip_extrapolated": cpu_ms * CLIP_FRAMES / 1e3,
                "api": "livespeechportraits_b200.headpose.HeadposeGenerator.generate (lsph_generate): incremental WaveNet + "
                       "Sample_GMM in one persistent 8-CTA cluster kernel; replaces models/audio2headpose_model.py:169-187"}
            del gen
        except Exception as exc:      # noqa: BLE001
            extras["headpose_loop"] = {"unavailable": f"{type(exc).__name__}: {exc}"}
        try:
            extras["library_baseline"] = library_baseline(VARIANT, B, H, W)
        except Exception as exc:      # noqa: BLE001
            extras["library_baseline"] = {"unavailable": f"{type(exc).__name__}: {exc}"}

    cpu = None
    if rank == 0 and world == 1:
        fps1, ms1, cores = cpu_reference_fps(VARIANT, H, W, 1, 12, 2)
        fps8, ms8, _ = cpu_reference_fps(VARIANT, H, W, 8, 2, 1)
        cpu = {"value": fps1, "unit": "frames/s", "cores": cores, "kind": "port", "host": host_cpu_info(),
               "batch8": {"value": fps8, "unit": "frames/s", "sample": "2 steps (+1 warm-up) of 8 frames"},
               "sample": "12 frames (+2 warm-up), batch 1 (the reference's batch), fp32, all host threads (count calibrated), "
                         "oracle/f2f_oracle.py (torch ATen convs = what the reference executes on CPU)"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.mode == "fast" else "fp16 hi+lo split operands (3 tcgen05 MMAs per K step), fp32 accumulate",
            "data": "synthetic (seeded weights with the reference's init distribution - no checkpoint ships; seeded inputs)",
            "config": config_dict(args, world),
            "max_abs_err_vs_oracle": parity_err, "max_abs_err_note": parity_note,
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches * K,
            "roofline": roofline, "cpu_baseline": cpu, "graph": net.graph_stats(),
        }
        if gather_info:
            line["gather"] = gather_info
        line.update(extras)
        emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
