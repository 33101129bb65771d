#!/usr/bin/env python
"""bench.py — 1920x1024 P-frames/s of the TDVC P-frame coding forward pass on N B200s (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels behind the C-ABI)
    python bench.py --impl reference --steps K --warmup W    # reference arm: the CPU path on the host cores

A "step" is one P-frame (ME + MC + multi-frame fusion + residual codec + bpp + in-loop filter) coded inside a
GOP-12 chain (I-frame raw + 11 P-frames, reference tools/predict.py:51-68) of a synthetic UVG-shaped
1920x1024 sequence.  N>1: one process per GPU (torchrun), GOPs sharded round-robin over ranks (weak scaling:
every rank codes K P-frames), one NCCL all-reduce of the 7 fp64 statistic sums at the end; timing = max over
ranks of CUDA-event time around the K steps, bracketed by barrier + synchronize.

JSON keys beyond the base contract: `e2e` (same metric through VideoCompressor.forward with pinned HOST frames:
H2D of the frame and D2H of the reconstruction + bpp inside the timed region), `roofline` (dominant kernel,
live per-launch CUDA-event timing of an instrumented eager pass of a steady-state chain frame), `cpu_baseline` (oracle on
the host cores: ONE true 1920x1024 P-frame plus the 384x640 sample of round 1), `gpu_eager_baseline` (the same PyTorch
restatement run eagerly on this B200: fp32, TF32 convolutions, autocast fp16), `config5` (multi-frame fusion + in-loop
filter alone), `products_per_mac`, `gpu_launches`, `clocks`, `stats` (bpp / PSNR of the coded frames).  The per-kernel
tables of the instrumented frame (`kernels`, `memory_bound_kernels`) go to stderr as a JSON line of their own, so that the
result line stays short.

--dump-outputs DIR writes what the timed path returned in its last timed step as DIR/<name>.npy (rank 0; float32): the
reconstruction and both bpp of the last P-frame, or for --workload train the five outputs of the training forward and the
loss.  Inputs and weights are generated from fixed seeds, so two builds run with the same arguments can be compared output
for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
import warnings

warnings.filterwarnings("ignore")
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, GOP = 1024, 1920, 12
MACS_PER_PX = 3832051  # SURVEY.md 8(d): MAC per full-resolution pixel of one P-frame
ENABLE_AMP = True   # the reference's shipped evaluation config (reference cfg/predict.yaml: `enable_amp: True`; tools/predict.py:64-65,146)
CPU_SAMPLE = (384, 640)  # 1/8 of the 1920x1024 pixels (secondary CPU sample; the primary one is a full frame)
DUMP_BYTES = 60 * 2 ** 20   # --dump-outputs: data of all files together (64 MB with room for the .npy headers)


def dump_outputs(path, arrays):
    """Writes path/<name>.npy for each tensor of `arrays` in float32 (float64 stays float64).  Should they exceed DUMP_BYTES
    together, every array keeps every n-th element of its flattened form, the same n for all."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    arrays = {k: v.detach().cpu() for k, v in arrays.items()}
    arrays = {k: v if v.dtype == torch.float64 else v.float() for k, v in arrays.items()}
    step = -(-sum(v.numel() * v.element_size() for v in arrays.values()) // DUMP_BYTES)
    for k, v in arrays.items():
        np.save(os.path.join(path, k + ".npy"), (v.reshape(-1)[::step] if step > 1 else v).numpy())


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        if os.environ.get("TDVC_BENCH_SMI_MS") == "0":   # developer A/B switch: no sampling at all
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", os.environ.get("TDVC_BENCH_SMI_MS", "100")],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_oracle_rate(steps, warmup, full=True):
    """Reference CPU path (oracle = restatement pinned bit-exact to the reference code), all host threads.
    Primary sample: `steps` TRUE 1920x1024 P-frames (the workload's own first GOP, frame pair 1) after `warmup` warm-up
    frames at 384x640 (a full-size warm-up would double the minutes for nothing: the first call costs < 1 % of a 35-90 s
    frame).  Secondary: one 384x640 frame (1/8 of the pixels, the round-1 extrapolation base) and BASELINE config 1
    (256x256).  Returns a dict; with `full`, "outputs" holds what the last true-size frame returned."""
    import torch
    from oracle.stats import build_oracle
    from tdvc_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    orc = build_oracle()
    h, w = CPU_SAMPLE
    xs, rs = synth.make_frame_pair(h, w, seed=3)
    out = {"cores": torch.get_num_threads()}
    with torch.no_grad():
        for _ in range(max(warmup, 1)):
            orc(xs, rs, False)
        t0 = time.perf_counter()
        orc(xs, rs, False)
        out["sample_384x640_s"] = time.perf_counter() - t0
        x1, r1 = synth.make_frame_pair(256, 256, seed=4)
        orc(x1, r1, False)
        t0 = time.perf_counter()
        orc(x1, r1, False)
        out["config1_256x256_s"] = time.perf_counter() - t0
        if full:
            g = synth.make_gop(H, W, gop=2, seed=100)
            x, refs = g[1:2], g[0:1].unsqueeze(1).expand(-1, 4, -1, -1, -1).contiguous()
            ts = []
            for _ in range(steps):
                t0 = time.perf_counter()
                recon, bpp_res, bpp_mv = orc(x, refs, False)
                ts.append(time.perf_counter() - t0)
            out["full_s"] = sum(ts) / len(ts)
            out["full_steps"] = steps
            out["outputs"] = {"recon": recon, "bpp_res": bpp_res, "bpp_mv": bpp_mv}
    return out


def _cpu_record(r):
    if "full_s" in r:
        fps = 1.0 / r["full_s"]
        sample = (f"{r['full_steps']} true 1920x1024 P-frame(s) (frame 1 of the bench's first GOP), {r['full_s']:.1f} s each, after a "
                  f"384x640 warm-up; oracle/model.py, torch fp32, {r['cores']} threads")
    else:
        fps = 1.0 / (r["sample_384x640_s"] * (H * W) / (CPU_SAMPLE[0] * CPU_SAMPLE[1]))
        sample = (f"1 P-frame at 384x640 (1/8 of the pixels), {r['sample_384x640_s']:.2f} s, rate scaled by pixel count (extrapolated); "
                  f"oracle/model.py, torch fp32, {r['cores']} threads")
    return {"value": fps, "unit": "P-frames/s", "cores": r["cores"], "kind": "port", "sample": sample,
            "extrapolated": "full_s" not in r, "sample_hw": [H, W] if "full_s" in r else list(CPU_SAMPLE),
            "sample_384x640_s_per_frame": r["sample_384x640_s"],
            "extrapolated_from_384x640_fps": 1.0 / (r["sample_384x640_s"] * (H * W) / (CPU_SAMPLE[0] * CPU_SAMPLE[1])),
            "config1_256x256_s_per_frame": r["config1_256x256_s"]}


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path (the oracle port) on the host cores, TRUE 1920x1024
    frames: K timed steps (35-90 s each)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    r = cpu_oracle_rate(steps, 1, full=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, r["outputs"])
    rec = _cpu_record(r)
    line = {"impl": "reference", "metric": "1920x1024 P-frames/sec", "value": rec["value"], "unit": "P-frames/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": 1, "ms_per_step": 1000.0 / rec["value"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "UVG-shaped synthetic 1920x1024 sequence, GOP 12, P-frame forward, batch 1 "
                                   f"({steps} true-size frame(s) on the host cores)"},
            "cpu_baseline": rec,
            "e2e": {"value": rec["value"], "unit": "P-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def gpu_eager_baseline(dev, hh, ww, iters=3):
    """The PyTorch restatement of the reference forward (oracle/model.py: cuDNN convolutions, torchvision deformable conv)
    run EAGERLY on this GPU - what the reference's own code path costs on a B200 - in exact fp32, with TF32 convolutions,
    and under autocast fp16 (the reference's shipped `enable_amp: True`).  A reported baseline (SURVEY.md 8d)."""
    import torch
    from oracle.stats import build_oracle
    from tdvc_b200 import synth
    out = {}
    try:
        orc = build_oracle().to(dev).eval()
        g = synth.make_gop(hh, ww, gop=2, seed=100).to(dev)
        x, refs = g[1:2], g[0:1].unsqueeze(1).expand(-1, 4, -1, -1, -1).contiguous()
        tf0, tf1 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
        for name, tf32, amp in (("fp32", False, False), ("tf32", True, False), ("autocast_fp16", True, True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.no_grad():
                for _ in range(2):
                    with torch.autocast("cuda", enabled=amp):
                        orc(x, refs, amp)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(iters):
                    with torch.autocast("cuda", enabled=amp):
                        orc(x, refs, amp)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            out[name] = {"ms_per_frame": ms, "fps": 1000.0 / ms}
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf0, tf1
        out["what"] = "oracle/model.py in PyTorch eager mode on this GPU (cuDNN + torchvision deform_conv2d), batch 1, CUDA events"
        del orc
        torch.cuda.empty_cache()
    except Exception as e:  # a baseline leg must never take the bench line down
        out["error"] = f"{type(e).__name__}: {e}"[:300]
    return out


def gpu_eager_training_baseline(dev, batch=8, size=256, iters=3):
    """The same training step on the PyTorch restatement of the reference (oracle/model.py, cuDNN + torchvision deformable
    convolution, torch autograd) run EAGERLY on this GPU: exact fp32, TF32 convolutions (PyTorch's default), autocast fp16 (the
    reference's shipped cfg/train.yaml).  A reported baseline."""
    import torch
    from oracle.stats import build_oracle
    from tdvc_b200 import synth
    out = {}
    try:
        pairs = [synth.make_frame_pair(size, size, seed=500 + i) for i in range(batch)]
        x = torch.cat([p[0] for p in pairs]).to(dev)
        refs = torch.cat([p[1] for p in pairs]).to(dev)
        tf0, tf1 = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
        for name, tf32, amp in (("fp32", False, False), ("tf32", True, False), ("autocast_fp16", True, True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            orc = build_oracle().to(dev).train()
            params = [p for n, p in orc.named_parameters() if not n.endswith(".quantiles")]
            aux_params = [p for n, p in orc.named_parameters() if n.endswith(".quantiles")]
            opt, aux_opt = torch.optim.Adam(params, lr=1e-4), torch.optim.Adam(aux_params, lr=1e-3)
            scaler = torch.amp.GradScaler("cuda", enabled=amp)

            def step():
                with torch.autocast("cuda", enabled=amp):
                    o = orc(x, refs, amp)
                    mse = torch.nn.MSELoss()(o[0], x)
                loss = 2048 * mse + o[1].mean() + o[2].mean()
                opt.zero_grad()
                aux_opt.zero_grad()
                scaler.scale(loss).backward()
                scaler.unscale_(opt)
                torch.nn.utils.clip_grad_norm_(params, 2)
                scaler.step(opt)
                scaler.update()
                (o[3] + o[4]).backward()
                aux_opt.step()

            step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            out[name] = {"ms_per_step": ms, "samples_per_s": batch * 1000.0 / ms}
            del orc, opt, aux_opt
            torch.cuda.empty_cache()
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf0, tf1
        out["what"] = "oracle/model.py training step in PyTorch eager mode on this GPU (cuDNN, torchvision deform_conv2d autograd)"
    except Exception as e:
        out["error"] = f"{type(e).__name__}: {e}"[:300]
    return out


def training_leg(dev, world, steps, warmup, batch=8, size=256, graph=False, amp=None, outputs=None):
    """BASELINE config 4: one training step of reference tools/train.py:125-159 (enable_amp False branch) - forward, rd_loss
    (2048 * MSE + bpp_res + bpp_mv), backward, clip_grad_norm_(2), Adam step, aux_loss backward, aux Adam step - on a
    Vimeo-shaped synthetic batch: `batch` samples of 256x256 with 4 references each PER GPU (the reference splits a global
    batch over DataParallel replicas; one process per GPU with DistributedDataParallel here, NCCL gradient all-reduce).
    CUDA-event timed, max over ranks.  `outputs` (a dict) receives the forward's outputs and the loss of the last timed step,
    on the host."""
    import torch
    import torch.distributed as dist
    from tdvc_b200 import synth
    from tdvc_b200.model import VideoCompressor
    torch.manual_seed(synth.SEED)
    net = VideoCompressor()
    sd = net.state_dict()
    synth.condition_state_dict(sd)
    net.load_state_dict(sd)
    net = net.to(dev).train()
    model = net
    if world > 1:
        # 76 of the 535 tensors get no gradient (layers the forward never runs): the set is the same every step, so DDP is told
        # the graph is static instead of searching for it per step; gradients are views into the all-reduce buckets
        ddp_kw = {"static_graph": True} if os.environ.get("TDVC_BENCH_DDP_DYNAMIC") is None else {"find_unused_parameters": True}
        model = torch.nn.parallel.DistributedDataParallel(net, device_ids=[dev.index], gradient_as_bucket_view=True, **ddp_kw)
    params = [p for n, p in net.named_parameters() if not n.endswith(".quantiles")]
    aux_params = [p for n, p in net.named_parameters() if n.endswith(".quantiles")]
    # reference main/utils/utils.py:90-113 (cfg/train.yaml lr); `capturable` keeps the step counters on the device (graph leg)
    opt = torch.optim.Adam(params, lr=1e-4, capturable=graph)
    aux_opt = torch.optim.Adam(aux_params, lr=1e-3, capturable=graph)
    rank = dist.get_rank() if world > 1 else 0
    pairs = [synth.make_frame_pair(size, size, seed=500 + rank * batch + i) for i in range(batch)]
    x = torch.cat([p[0] for p in pairs]).to(dev)
    refs = torch.cat([p[1] for p in pairs]).to(dev)
    losses = []

    def step():
        out = model(x, refs, ENABLE_AMP if amp is None else amp)   # cfg/train.yaml `amp: True`
        mse = torch.nn.MSELoss()(out[0], x)
        loss = 2048 * mse + out[1].mean() + out[2].mean()
        aux = out[3] + out[4]
        opt.zero_grad()
        aux_opt.zero_grad()
        # one backward pass for both losses: rd_loss does not depend on `.quantiles` and aux_loss depends on nothing else, so
        # the gradients are those of the reference's two passes (DistributedDataParallel ties a forward's outputs to ONE pass)
        (loss + aux).backward()
        torch.nn.utils.clip_grad_norm_(params, 2)
        opt.step()
        aux_opt.step()
        losses.append(loss.detach())
        if outputs is not None:   # (in a captured step these are the graph's output tensors, which every replay rewrites)
            outputs.update({k: v.detach() for k, v in zip(("recon", "bpp_res", "bpp_mv", "mv_aux_loss", "res_aux_loss"), out)},
                           loss=loss.detach())

    torch.cuda.reset_peak_memory_stats(dev)
    mem0 = torch.cuda.memory_allocated(dev)     # what earlier legs of the same process still hold (graphs, caches) is not this leg's
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    run = step
    if graph:
        # the whole step - forward, backward, clipping, both optimiser steps - captured once and replayed: the eager step is
        # bound by the host (autograd + ~3,000 launches per step), not by the GPU
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            step()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize()
        cg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cg):
            step()
        run = cg.replay
        for _ in range(2):
            run()
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        run()
    e1.record()
    torch.cuda.synchronize()
    if outputs is not None:
        outputs.update({k: v.cpu() for k, v in outputs.items()})
    ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms)
    return {"ms_per_step": ms, "samples_per_s": batch * world / (ms / 1e3), "batch_per_gpu": batch, "size": size, "n_gpus": world,
            "steps": steps, "warmup": warmup, "cuda_graph": bool(graph), "loss_first": float(losses[0]), "loss_last": float(losses[-1]),
            "peak_mem_gb": (torch.cuda.max_memory_allocated(dev) - mem0) / 2 ** 30,
            "what": "forward + rd_loss backward + clip + Adam + aux step (reference tools/train.py:125-159); convolutions, GDN, DCN "
                    "and entropy models on tdvc_b200 kernels, torch autograd as the tape with torch glue operators between "
                    "them (DESIGN.md section 7)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=22)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="tdvc_b200")
    ap.add_argument("--conv-impl", type=int, default=0, help="0 auto (tcgen05 where supported), 1 SIMT fp32, 2 force tcgen05")
    ap.add_argument("--precision", default="auto", choices=["auto", "exact", "mixed"],
                    help="auto: as the reference's switch asks - enabled_amp=True (cfg/predict.yaml) relaxes the stages behind the last "
                         "quantiser to one fp16 MMA product; exact: fp32-class everywhere")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cache", action="store_true", help="recompute the per-GOP features every frame (as the reference does)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--cpu-sample", default="full", choices=["full", "small"])
    ap.add_argument("--workload", default="predict", choices=["predict", "train"],
                    help="predict: the headline P-frame coding benchmark; train: BASELINE config 4 (training step) on its own")
    ap.add_argument("--no-train-leg", action="store_true")
    ap.add_argument("--train-exact", action="store_true", help="--workload train: enabled_amp=False (fp32-class weight gradients)")
    ap.add_argument("--train-graph", action="store_true", help="--workload train: capture the whole step in a CUDA graph and replay it (a measurement of the GPU-bound step: replays reuse the captured noise seed and weight scalings)")
    ap.add_argument("--height", type=int, default=H)
    ap.add_argument("--width", type=int, default=W)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from tdvc_b200 import gop as G
    from tdvc_b200 import lib as L
    from tdvc_b200 import synth
    from tdvc_b200.model import VideoCompressor

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (tdvc_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))   # a hang must fail fast
    if args.workload == "train":
        outs = {} if args.dump_outputs else None
        rec = training_leg(dev, world, args.steps, max(args.warmup, 3), graph=args.train_graph and world == 1,
                           amp=False if args.train_exact else None, outputs=outs)
        if rank == 0 and args.dump_outputs:
            dump_outputs(args.dump_outputs, outs)
        if rank == 0 and world == 1 and not args.no_eager_baseline:
            torch.cuda.empty_cache()
            rec["gpu_eager_baseline"] = gpu_eager_training_baseline(dev)
        if rank == 0:
            print(json.dumps({"metric": "training samples/sec (256x256 Vimeo-shaped, batch 8 per GPU)", "value": rec["samples_per_s"],
                              "unit": "samples/s", "n_gpus": world, "steps": rec["steps"], "warmup": rec["warmup"],
                              "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                              "dtype": "f32", "data": "synthetic", "config": {"workload": "BASELINE config 4: " + rec["what"]},
                              "training_step": rec}), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    hh, ww = args.height, args.width
    K, Wm = args.steps, max(args.warmup, 3)
    # one untimed GOP in front of the W warm-up steps: every launch variant of a GOP (which features are cached) is run and
    # captured into its CUDA graph there, so warm-up and timed steps replay graphs only
    Wm_total = Wm + (GOP - 1)

    # ---- model: module default init under the reference seed + deterministic conditioning (synth.py)
    torch.manual_seed(synth.SEED)
    net = VideoCompressor().eval()
    sd = net.state_dict()
    synth.condition_state_dict(sd)
    net.load_state_dict(sd)
    net = net.to(dev)
    net.conv_impl = args.conv_impl
    net.precision = args.precision
    net.use_cuda_graph = not args.no_graph
    net.cache_features = not args.no_cache

    # ---- synthetic sequence: this rank's GOPs (round-robin shard of a global GOP list), pinned on the host
    my_gops = [g * world + rank for g in range(2)]
    host_gops = []
    for g in my_gops:  # two distinct GOPs are generated, then cycled (generation is slow on the host)
        host_gops.append(synth.make_gop(hh, ww, gop=GOP, seed=100 + g).pin_memory())
    dev_gops = [g.to(dev, non_blocking=True) for g in host_gops]
    torch.cuda.synchronize()

    def frame_stream(src):
        """yields (gop, frame index) endlessly, GOP after GOP."""
        gi = 0
        while True:
            g = src[gi % len(src)]
            for t in range(1, GOP):
                yield g, t
            gi += 1

    def run_chain(src, n_warm, n_timed, host_io):
        """Codes n_warm + n_timed P-frames as GOP chains; returns (ms, stats[7], launches, outputs of the last frame)."""
        stats = torch.zeros(7, device=dev, dtype=torch.float64)
        sse = torch.zeros(1, device=dev, dtype=torch.float64)
        it = frame_stream(src)
        refs = None   # tdvc_b200.gop.RefBuffer of the running GOP
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pin_out = torch.empty((1, 3, hh, ww), dtype=torch.float32).pin_memory() if host_io else None
        pin_bpp = torch.empty(2, dtype=torch.float32).pin_memory() if host_io else None
        launches = 0
        for i in range(n_warm + n_timed):
            if i == n_warm:
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                sampler.start()
                ev0.record()
            g, t = next(it)
            if t == 1:
                refs = G.RefBuffer(g[0:1].to(dev, non_blocking=True) if host_io else g[0:1])
            x = g[t:t + 1].to(dev, non_blocking=True) if host_io else g[t:t + 1]
            window, keys = refs.window()
            if host_io:
                # end to end: the reference-facing call exactly as tools/predict.py:64-65 makes it (the feature caches are keyed
                # on the device-side content hash of the reference slices: one host synchronisation per frame)
                recon, bpp_res, bpp_mv = net(x, window, ENABLE_AMP)
            else:
                # resident leg: through the GOP driver's call (tdvc_b200/gop.py), which passes the frame identities it knows
                recon, bpp_res, bpp_mv = net(x, window, ENABLE_AMP, ref_keys=keys)
            if i >= n_warm:
                launches += net.last_launches
            refs.push(recon)
            if host_io:
                pin_out.copy_(recon, non_blocking=True)
                pin_bpp.copy_(torch.cat([bpp_res, bpp_mv]), non_blocking=True)
                torch.cuda.current_stream().synchronize()  # the caller reads the result of every step
            if i >= n_warm:
                sse.zero_()
                G.sq_err_sum(recon, x, sse, 0)
                mse = sse[0] / (3 * hh * ww)
                b = (bpp_res[0] + bpp_mv[0]).double()
                stats += torch.stack([b, bpp_mv[0].double(), bpp_res[0].double(), 10.0 * torch.log10(1.0 / mse),
                                      torch.zeros((), device=dev, dtype=torch.float64), mse,
                                      torch.ones((), device=dev, dtype=torch.float64)])
        ev1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = ev0.elapsed_time(ev1)
        return ms, stats, launches, {"recon": recon, "bpp_res": bpp_res, "bpp_mv": bpp_mv}

    sampler = ClockSampler(local)
    ms, stats, launches, last = run_chain(dev_gops, Wm_total, K, host_io=False)
    clocks = sampler.stop()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    del last
    sampler = ClockSampler(local)
    sampler.start = lambda: None  # clocks are sampled on the device-resident leg only
    ms_e2e, _, _, _ = run_chain(host_gops, Wm_total, K, host_io=True)
    # secondary: the same resident chain with every convolution at fp32-class accuracy (enabled_amp=False semantics)
    ms_exact = None
    if net._precision(ENABLE_AMP) != "exact" and world == 1:   # (run_chain holds collectives: a leg is run by all ranks or none)
        net.precision = "exact"
        ms_exact, _, _, _ = run_chain(dev_gops, GOP - 1, GOP - 1, host_io=False)
        ms_exact /= GOP - 1
        net.precision = args.precision

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        G.reduce_stats(stats)
    ms, ms_e2e = float(t[0]), float(t[1])
    value = world * K / (ms / 1000.0)
    e2e = world * K / (ms_e2e / 1000.0)

    line = None
    if rank == 0:
        peaks, which = _peaks()
        # ---- roofline of the dominant kernel: instrumented eager pass over a steady-state chain frame (frame 7 of a GOP: the
        #      I-frame features and two of the three fusion fronts come from the caches, as in 6 of every 11 frames),
        #      per-launch CUDA events; the hyperprior side stream is serialised so that every launch is timed alone
        net.use_cuda_graph = False
        plan = net._plan(1, hh, ww, dev)
        g = dev_gops[0]
        refs = [g[0:1]]
        prof = None
        for tt in range(1, 8):
            if tt == 7:
                plan.prof = []
            recon, _, _ = net(g[tt:tt + 1], G.reference_window(refs), ENABLE_AMP)
            refs.append(recon)
            if len(refs) > 4:
                refs = [refs[0]] + refs[-3:]
        torch.cuda.synchronize()
        prof, plan.prof = plan.prof, None
        agg = {}
        for label, macs, nbytes, e0, e1, prod in prof:
            a = agg.setdefault(label, [0, 0.0, 0, 0, prod])
            a[0] += 1
            a[1] += e0.elapsed_time(e1)
            a[2] += macs
            a[3] += nbytes
        total_ms = sum(a[1] for a in agg.values())
        mma_macs = sum(a[2] for a in agg.values() if a[4])
        products_per_mac = sum(a[2] * a[4] for a in agg.values() if a[4]) / max(mma_macs, 1)
        top = sorted(agg.items(), key=lambda kv: -kv[1][1])
        dom_label, (cnt, dms, dmacs, dbytes, dprod) = top[0]
        if dmacs > 0 and not dom_label.startswith("dcn"):
            achieved = 2.0 * dmacs / (dms / 1e3) / 1e12
            peak = peaks["bf16_tflops_sustained"]
            traffic = None
            try:  # DRAM bytes per launch of this kernel from the committed ncu --set full capture (profiles/)
                dj = json.load(open(os.path.join(ROOT, "profiles", "r02_dominant.json")))
                if dj["label"] == dom_label:
                    images = dmacs / cnt / (hh * ww * 64 * 64 * 9)
                    traffic = dj["dram_bytes_per_image"] * images
            except Exception:
                pass
            roof = {"kernel": dom_label, "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                    "frac": achieved / peak, "traffic": traffic, "launches": cnt, "avg_launch_ms": dms / cnt,
                    "share_of_frame": dms / total_ms, "peak_source": which + " (sustained bf16)",
                    "products_per_mac": dprod,
                    "mma_equivalent_tflops": dprod * achieved, "mma_equivalent_frac": dprod * achieved / peak,
                    "note": "achieved = algorithmic FLOPs (2*MACs of the convolution); this kernel issues `products_per_mac` fp16 MMA "
                            "products per algorithmic MAC (fp32-class hi/lo split), so tensor-pipe work is that multiple "
                            "(mma_equivalent_*); traffic = ncu dram bytes per launch (profiles/r02_dominant.json)"}
        else:
            achieved = dbytes / (dms / 1e3) / 1e9
            peak = peaks["hbm_gbs"]
            roof = {"kernel": dom_label, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": None, "launches": cnt, "avg_launch_ms": dms / cnt,
                    "share_of_frame": dms / total_ms, "peak_source": which}
        kernels = {k: {"launches": v[0], "ms": round(v[1], 4),
                       "tflops": round(2.0 * v[2] / (v[1] / 1e3) / 1e12, 2) if v[2] and v[1] > 0 else None,
                       "gbs": round(v[3] / (v[1] / 1e3) / 1e9, 1) if v[3] and v[1] > 0 else None,
                       "products_per_mac": v[4] or None} for k, v in top}
        # memory-bound kernels of the frame against the measured HBM peak (SURVEY.md 8d rows: warp, DCN gather, GDN, bits)
        mem_rows = {}
        for k, v in agg.items():
            if v[3] and v[1] > 0 and (not k.startswith("conv") or k.startswith("conv1x1")):
                gbs = v[3] / (v[1] / 1e3) / 1e9
                mem_rows[k] = {"ms": round(v[1], 4), "gbs": round(gbs, 1), "frac_of_hbm_peak": round(gbs / peaks["hbm_gbs"], 3)}
        frame_tflops = 2.0 * MACS_PER_PX * hh * ww / (ms / K / 1e3) / 1e12
        # ---- BASELINE config 5 on its own: multi-frame fusion + in-loop filter with 4 reference frames (nothing cached)
        cfg5 = None
        try:
            p1 = torch.randn(1, 64, hh, ww, device=dev) * 0.5
            rf = torch.randn(1, 64, hh, ww, device=dev) * 0.5
            r4 = G.reference_window([g[0:1], g[1:2], g[2:3], g[3:4]])
            for _ in range(2):
                net.fusion_and_filter(p1, r4, rf, ENABLE_AMP)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                net.fusion_and_filter(p1, r4, rf, ENABLE_AMP)
            e1.record()
            torch.cuda.synchronize()
            c5ms = e0.elapsed_time(e1) / 5
            cfg5 = {"ms_per_call": c5ms, "tflops": 2.0 * 1438138 * hh * ww / (c5ms / 1e3) / 1e12, "launches": net.last_launches,
                    "what": "VideoCompressor.fusion_and_filter: mcfilter + loopfilter at full size, 4 reference frames, no cache, "
                            "eager launches, includes the NCHW<->NHWC conversions of the 64-channel inputs / output"}
            del p1, rf
        except Exception as e:
            cfg5 = {"error": f"{type(e).__name__}: {e}"[:300]}
        # ---- real entropy coding of one frame (`is_compress=True`, reference pnet.py:45-49,69-73): forward + tables (cached) +
        #      both autoregressive passes + host rANS, wall clock around the call; not part of the headline (the reference's
        #      benchmark path estimates bits, cfg/predict.yaml)
        coding = None
        if world == 1:
            try:
                import time
                xg, r4 = g[4:5], G.reference_window([g[0:1], g[1:2], g[2:3], g[3:4]])
                net(xg, r4, ENABLE_AMP, is_compress=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                net(xg, r4, ENABLE_AMP)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                out = net(xg, r4, ENABLE_AMP, is_compress=True)
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                lc = net.last_coded
                coding = {"ms_forward": (t1 - t0) * 1e3, "ms_forward_and_coding": (t2 - t1) * 1e3,
                          "ac_bpp_mv": lc["mv"]["ac_bpp"], "ac_bpp_res": lc["res"]["ac_bpp"],
                          "estimated_bpp_mv": float(out[2]), "estimated_bpp_res": float(out[1]),
                          "bytes": {k: [len(s[0]) for s in v["strings"]] for k, v in lc.items()},
                          "what": "one 1920x1024 P-frame through forward(..., is_compress=True): wavefront autoregressive "
                                  "kernel per coder (two streams) + host rANS (compressai's coder runs on the host too)"}
            except Exception as e:
                coding = {"error": f"{type(e).__name__}: {e}"[:300]}
        train = None
        if world == 1 and not args.no_train_leg:
            try:
                torch.cuda.empty_cache()
                train = training_leg(dev, 1, 4, 3)
            except Exception as e:
                train = {"error": f"{type(e).__name__}: {e}"[:300]}
            torch.cuda.empty_cache()
            if "error" not in train:
                try:   # the same step captured in ONE CUDA graph and replayed (no host work per step)
                    g = training_leg(dev, 1, 4, 3, graph=True)
                    train["cuda_graph_replay"] = {k: g[k] for k in ("ms_per_step", "samples_per_s", "steps", "warmup", "peak_mem_gb")}
                except Exception as e:
                    train["cuda_graph_replay"] = {"error": f"{type(e).__name__}: {e}"[:300]}
                torch.cuda.empty_cache()
                try:   # enabled_amp=False: fp32-class arithmetic everywhere (three-product weight gradients)
                    train["exact_precision_ms_per_step"] = training_leg(dev, 1, 4, 3, amp=False)["ms_per_step"]
                except Exception as e:
                    train["exact_precision_ms_per_step"] = f"{type(e).__name__}: {e}"[:300]
                torch.cuda.empty_cache()
            if not args.no_eager_baseline and "error" not in train:
                train["gpu_eager_baseline"] = gpu_eager_training_baseline(dev)
        eager = None
        if not args.no_eager_baseline and world == 1:
            eager = gpu_eager_baseline(dev, hh, ww)
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cpu = _cpu_record(cpu_oracle_rate(1, 1, full=args.cpu_sample == "full"))
        frame_bytes = 3 * hh * ww * 4
        eff = net._precision(ENABLE_AMP)
        dtype = ("f32 (convolutions: fp32 operands split into fp16 hi+lo, tcgen05 MMA, fp32 accumulation in TMEM"
                 + ("; enabled_amp=True as in the reference's cfg/predict.yaml: one fp16 product - the reference's autocast "
                    "arithmetic - in the stages behind the last quantiser of the frame)" if eff == "mixed" else ")"))
        line = {"metric": "1920x1024 P-frames/sec", "value": value, "unit": "P-frames/s", "n_gpus": world, "steps": K,
                "warmup": Wm_total, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": dtype, "data": "synthetic",
                "config": {"workload": f"UVG-shaped synthetic {ww}x{hh} sequence, GOP 12 (I-frame raw + 11 chained P-frames), "
                                       "inference, batch 1 per GPU, GOP-sharded over ranks",
                           "l2": "per-frame working set >> 126 MB L2 (each full-resolution 64-channel tensor is 503 MB)",
                           "cuda_graph": not args.no_graph, "conv_impl": args.conv_impl, "enabled_amp": ENABLE_AMP,
                           "precision": eff, "feature_cache": not args.no_cache},
                "e2e": {"value": e2e, "unit": "P-frames/s", "h2d_bytes_per_step": frame_bytes,
                        "d2h_bytes_per_step": frame_bytes + 8},
                "gpu_launches": launches, "clocks": clocks,
                "roofline": roof, "frame_tensor_tflops": frame_tflops,
                "frame_tensor_frac_of_sustained_bf16": frame_tflops / peaks["bf16_tflops_sustained"],
                "products_per_mac": products_per_mac, "instrumented_frame_ms": total_ms,
                "config5": cfg5, "entropy_coding": coding, "training_step": train,
                "gpu_eager_baseline": eager, "exact_precision_ms_per_step": ms_exact,
                "cpu_baseline": cpu, "stats": G.summarise(stats)}
        print(json.dumps({"memory_bound_kernels": mem_rows, "kernels": kernels}), file=sys.stderr, flush=True)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
