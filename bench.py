#!/usr/bin/env python
"""bench.py — throughput of the hot path on B200 (one JSON line on stdout, rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Metric (BASELINE.json): 96x96 face-crops/sec through Wav2Lip.forward, B=128, T=5, mel 80x16.
One step = one 5-D generator call `Wav2Lip(indiv_mels (128,5,1,80,16), x (128,6,5,96,96))` = 640 crops
per GPU, eval mode, synthetic seeded inputs, seeded random weights (the reference's default-init
statistics with randomised BatchNorm).  Weak scaling: every rank runs its own 640-crop batch; there is
no data-path collective (eval-mode forward has no cross-sample op), torch.distributed carries only the
barrier and the max-over-ranks time.

  value      crops/s with the inputs resident in HBM, CUDA-event time on the launching stream,
             barrier + synchronize on both sides of EXACTLY K steps, max over ranks.
  e2e        the same metric through the C-ABI host entry points (w2l_generator_submit_host + w2l_host_wait): pinned host
             inputs -> H2D -> forward -> D2H of the (B,3,T,96,96) result, every step.
  roofline   tensor-core bound: algorithmic FLOPs (7.934 GFLOP/crop, SURVEY.md §8d) of the conv kernel
             launches of one step / their summed per-launch CUDA-event durations (measured live, after the
             timed region), against MEASURED_PEAKS.json's sustained bf16 figure (fp16 runs at the same rate).
  cpu_baseline  the oracle port (oracle/w2l_oracle.py, torch CPU fp32 = the reference's own arithmetic) on
             the host cores, N=128 4-D batch (inference.py's default batch), rank 0 at N=1 only.

--dump-outputs DIR writes what rank 0's last timed step returned as DIR/<name>.npy (float32): generator_out.npy,
the (B,3,T,96,96) prediction, or losses.npy for --workload train.  Inputs and weights depend only on the arguments,
so two builds run with the same arguments can be compared array for array.
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
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it

FLOP_PER_CROP = 2 * 3966984192  # SURVEY.md §8(d): 3 966.98 MMAC per 96x96 crop
METRIC = "96x96 face-crops/sec (B=128, T=5, mel 80x16)"
B_DEFAULT, T_DEFAULT = 128, 5
DUMP_BYTES = 64 * 10**6  # --dump-outputs: all arrays together


def dump_outputs(path, arrays):
    """Write each tensor of `arrays` as <path>/<name>.npy in float32.  One that does not fit what is left of DUMP_BYTES
    is cut to a fixed seeded sample of its leading-axis rows (kept in order), the same rows on every run."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    left = DUMP_BYTES - 4096 * len(arrays)  # room for the .npy headers
    for name, t in arrays.items():
        t = t.detach().float().cpu()
        if t.numel() * 4 > left:
            rows = left // (t[0].numel() * 4)
            pick = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values
            t = t[pick]
        left -= t.numel() * 4
        np.save(os.path.join(path, name + ".npy"), t.numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops": float(d["bf16_tflops_sustained"]), "tflops_burst": float(d["bf16_tflops"]),
                "hbm_gbs": float(d["hbm_gbs"]), "src": "measured"}
    return {"tflops": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.lines:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "samples": len(sm),
                "reasons": sorted(reasons)}


def pick_threads(sd, O, torch):
    """torch's CPU conv does not scale to every hardware thread of a large host (128 threads were 8x SLOWER than
    32 on the B200 box): calibrate on a small batch and give the reference arm its best thread count."""
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    mel, face = O.make_generator_inputs(8, 1)
    best, best_t = None, cands[-1]
    for c in cands:
        torch.set_num_threads(c)
        with torch.no_grad():
            O.generator_forward(sd, mel[:2], face[:2])
            t0 = time.perf_counter()
            O.generator_forward(sd, mel, face)
            dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, best_t = dt, c
    torch.set_num_threads(best_t)
    return best_t


def cpu_baseline_run(n, repeats=1):
    """The oracle port (the reference's own CPU arithmetic: torch fp32 conv/BN/ReLU) on the host cores."""
    import torch
    from oracle import w2l_oracle as O
    sd = O.make_state_dict("generator", 0, init="default")
    threads = pick_threads(sd, O, torch)
    mel, face = O.make_generator_inputs(n, 0)
    with torch.no_grad():
        O.generator_forward(sd, mel[:2], face[:2])  # warm the thread pool / primitive cache
        best = None
        for _ in range(repeats):
            t0 = time.perf_counter()
            O.generator_forward(sd, mel, face)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return n / best, best, threads


def measure_extra(dev):
    """SyncNet_color B=256, Wav2Lip_disc_qual B=256 x T=5, audio.melspectrogram 10 k and 1 M frames: CUDA-event
    times of the other entry points of the path (BASELINE configs[2] and [3]); random default-init weights."""
    import numpy as np
    import torch
    from wav2lip_b200 import audio
    from wav2lip_b200.models import SyncNet_color, Wav2Lip_disc_qual
    out = {}

    def timeit(fn, iters):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / iters

    with torch.no_grad():
        torch.manual_seed(2)
        s = SyncNet_color().to(dev).eval()
        mel = (torch.rand((256, 1, 80, 16)) * 8 - 4).to(dev)
        face = torch.rand((256, 15, 48, 96)).to(dev)
        ms = timeit(lambda: s(mel, face), 10)
        out["syncnet"] = {"config": "SyncNet_color.forward B=256 (fp16 operands)", "ms": ms, "windows_per_s": 256 / ms * 1e3,
                          "tflops": 256 / ms * 1e3 * 2 * 1210281984 / 1e12}
        del s
        d = Wav2Lip_disc_qual().to(dev).eval()
        frames = torch.rand((256, 3, 5, 96, 96)).to(dev)
        ms = timeit(lambda: d(frames), 10)
        out["disc"] = {"config": "Wav2Lip_disc_qual.forward B=256, T=5 (1280 frames, fp16 operands)", "ms": ms,
                       "frames_per_s": 1280 / ms * 1e3, "tflops": 1280 / ms * 1e3 * 2 * 1255850496 / 1e12}
        del d, frames
        # scope row f4: the S3FD network on one face_det_batch (inference.py:43: 16 frames) of 720p frames
        try:
            from wav2lip_b200 import _lib as _L
            from wav2lip_b200.face_detection.detection.sfd.net_s3fd import s3fd
            fd = s3fd().to(dev).eval()
            img = (torch.rand((16, 3, 720, 1280)) * 255 - 117).to(dev)
            ms = timeit(lambda: fd(img), 5)
            fl = sum(f for _, _, f in fd._w2l_ctx.profile_plan(_L.NET_S3FD, iters=1))
            out["s3fd"] = {"config": "s3fd.forward, 16 frames of 1280x720 (face_det_batch_size, fp16 operands)", "ms": ms,
                           "frames_per_s": 16 / ms * 1e3, "tflops": fl / ms / 1e9}
            del fd, img
        except Exception as e:
            out["s3fd"] = {"error": repr(e)[:200]}
        # frames in, frames out: the whole inner loop of inference.py in one call (crop, resize, generator, resize, paste)
        try:
            from wav2lip_b200.models import Wav2Lip as _G
            gg = _G().to(dev).eval()
            fr = torch.randint(0, 256, (32, 720, 1280, 3), dtype=torch.uint8, device=dev)
            bx = [[i % 32, 200 + (i % 7), 520 + (i % 5), 500 + (i % 11), 800 + (i % 3)] for i in range(128)]
            mm = (torch.rand((128, 1, 80, 16)) * 8 - 4).to(dev)
            ms = timeit(lambda: gg.infer_frames(mm, fr, bx), 5)
            out["infer_frames"] = {"config": "Wav2Lip.infer_frames: 128 mel chunks + 32 720p frames + boxes -> 128 finished 720p frames "
                                             "(crop, cv2-exact resize, generator, resize, paste; 354 MB of frames written)", "ms": ms,
                                   "frames_per_s": 128 / ms * 1e3}
            del gg, fr
        except Exception as e:
            out["infer_frames"] = {"error": repr(e)[:200]}
        # fused uint8 batch assembly (scope row f): host uint8 crops + fp32 mels in, host uint8 predictions out
        import ctypes as C
        from wav2lip_b200 import _lib
        from wav2lip_b200.models import Wav2Lip
        g = Wav2Lip().to(dev).eval()
        g._ensure(torch.zeros(1, device=dev))
        ctx = g._w2l_ctx
        n = 640
        faces = torch.randint(0, 256, (n, 96, 96, 3), dtype=torch.uint8).pin_memory()
        melh = (torch.rand((n, 1, 80, 16)) * 8 - 4).pin_memory()
        outh = torch.empty((n, 96, 96, 3), dtype=torch.uint8).pin_memory()

        def u8_step():
            _lib.check(ctx.lib.w2l_generator_forward_u8_host(ctx.h, C.c_void_p(melh.data_ptr()), C.c_void_p(faces.data_ptr()),
                                                             C.c_void_p(outh.data_ptr()), n))
        for _ in range(3):
            u8_step()
        t0 = time.perf_counter()
        for _ in range(10):
            u8_step()
        dt = (time.perf_counter() - t0) / 10
        outh2 = torch.empty((n, 96, 96, 3), dtype=torch.uint8).pin_memory()
        outs = [outh, outh2]

        def u8_submit(k):
            _lib.check(ctx.lib.w2l_generator_submit_u8_host(ctx.h, C.c_void_p(melh.data_ptr()), C.c_void_p(faces.data_ptr()),
                                                            C.c_void_p(outs[k & 1].data_ptr()), n))
        for k in range(3):
            u8_submit(k)
            _lib.check(ctx.lib.w2l_host_wait(ctx.h, 1))
        _lib.check(ctx.lib.w2l_host_wait(ctx.h, 0))
        t0 = time.perf_counter()
        for k in range(20):
            u8_submit(k)
            _lib.check(ctx.lib.w2l_host_wait(ctx.h, 1))
        _lib.check(ctx.lib.w2l_host_wait(ctx.h, 0))
        dtp = (time.perf_counter() - t0) / 20
        out["e2e_u8"] = {"config": "640 uint8 96x96x3 crops + fp32 mels from pinned host memory, uint8 predictions back "
                                   "(inference.py:134-140,259-265,269 fused); submit/wait loop with two batches in flight",
                         "ms": dtp * 1e3, "crops_per_s": n / dtp, "h2d_bytes": int(faces.numel() + melh.numel() * 4),
                         "d2h_bytes": int(outh.numel()), "pipelined_equals_sync": bool(torch.equal(outh, outh2)),
                         "synchronous_call": {"api": "w2l_generator_forward_u8_host", "ms": dt * 1e3, "crops_per_s": n / dt}}
        # inference.py's own call shape: one 4-D batch of 128 crops (inference.py:259-263, --wav2lip_batch_size 128)
        mel128 = (torch.rand((128, 1, 80, 16)) * 8 - 4).to(dev)
        face128 = torch.rand((128, 6, 96, 96)).to(dev)
        ms = timeit(lambda: g(mel128, face128), 20)
        out["generator_n128"] = {"config": "Wav2Lip.forward 4-D N=128 (inference.py batch), device-resident", "ms": ms,
                                 "crops_per_s": 128 / ms * 1e3}
        del g, mel128, face128
        # the fp32-faithful precision mode (split fp16 operands, 3 MMAs per product) on the headline workload
        gx = Wav2Lip()
        gx.precision = _lib.PREC_F32X
        gx = gx.to(dev).eval()
        melx = (torch.rand((B_DEFAULT, T_DEFAULT, 1, 80, 16)) * 8 - 4).to(dev)
        facex = torch.rand((B_DEFAULT, 6, T_DEFAULT, 96, 96)).to(dev)
        ms = timeit(lambda: gx(melx, facex), 5)
        out["generator_f32x"] = {"config": "Wav2Lip.forward B=128,T=5 in W2L_PREC_F32X (hi+lo fp16 operands, ~22-bit significands; "
                                           "max-abs error 1.3e-4 on the stress weights vs 3.7e-3 in the default mode)",
                                 "ms": ms, "crops_per_s": B_DEFAULT * T_DEFAULT / ms * 1e3}
        del gx, melx, facex
        for nfr, key in ((10000, "mel_10k"), (1000000, "mel_1M")):
            wav = (0.1 * torch.randn((nfr - 1) * 200, device=dev)).float()
            ms = timeit(lambda: audio.melspectrogram(wav), 10)
            out[key] = {"config": f"audio.melspectrogram, {nfr} frames ({wav.numel()} samples) resident on the device",
                        "ms": ms, "frames_per_s": nfr / ms * 1e3, "algorithmic_GBps": nfr * 1120 / ms / 1e6}
    return out


def measure_train(dev, rank, world, steps, warmup, B=64, T=5, syncnet_wt=0.03, profile_out=None, dump_dir=None):
    """BASELINE configs[4]: one wav2lip_train.py:210-231 iteration per step (generator train-mode forward, get_sync_loss
    through the frozen expert, L1, backward, gradient all-reduce over NCCL when world > 1, Adam), bf16 operands, B=64
    windows x T=5 frames per GPU, everything native (w2l_wav2lip_train_step).  Inputs resident on the device; CUDA-event
    timing, max over ranks."""
    import torch
    import torch.distributed as dist
    from wav2lip_b200 import _lib
    from wav2lip_b200.models import SyncNet_color, Wav2Lip
    from wav2lip_b200.parallel import max_over_ranks
    from wav2lip_b200.training import Wav2LipTrainStep, init_data_parallel
    torch.manual_seed(0)
    model = Wav2Lip().to(dev).train()
    expert = SyncNet_color().to(dev).train()
    step = Wav2LipTrainStep(model, expert, lr=1e-4, syncnet_wt=syncnet_wt)
    if world > 1:
        init_data_parallel(step)
    g = torch.Generator().manual_seed(200 + rank)
    x = torch.rand((B, 6, T, 96, 96), generator=g)
    x[:, 0:3, :, 48:, :] = 0.0
    indiv_mels = torch.rand((B, T, 1, 80, 16), generator=g) * 8 - 4
    mel = torch.rand((B, 1, 80, 16), generator=g) * 8 - 4
    gt = torch.rand((B, 3, T, 96, 96), generator=g)
    x, indiv_mels, mel, gt = (t.to(dev) for t in (x, indiv_mels, mel, gt))

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(3, warmup)):
        losses = step(x, indiv_mels, mel, gt)
    barrier()
    ctx = step.b.ctx
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.current_stream(dev)
    e0.record(stream)
    for _ in range(steps):
        losses = step(x, indiv_mels, mel, gt)
    e1.record(stream)
    torch.cuda.synchronize(dev)
    barrier()
    last_losses = losses.cpu()   # the step reuses its loss buffer: copy the last timed step's before anything else runs
    ms = max_over_ranks(e0.elapsed_time(e1), dev) / steps
    launches = (ctx.launch_count() - l0) // steps
    gen_f = ctx.lib.w2l_train_flops(ctx.h, _lib.NET_GENERATOR)
    syn_f = ctx.lib.w2l_train_flops(ctx.h, _lib.NET_SYNCNET)
    flop = 3.0 * gen_f + 2.0 * syn_f       # forward + dgrad + wgrad of the generator; forward + dgrad of the frozen expert
    lv = [float(v) for v in last_losses]
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {"losses": last_losses})
    n_param = sum(p.numel() for p in model.parameters())
    if profile_out and rank == 0:
        rows = ctx.train_profile(_lib.NET_GENERATOR, iters=3, stream=stream.cuda_stream) + \
            [("expert:" + n, m, f) for n, m, f in ctx.train_profile(_lib.NET_SYNCNET, iters=3, stream=stream.cuda_stream)]
        tot = sum(m for _, m, _ in rows)
        with open(profile_out, "w") as f:
            f.write(f"# per-stage CUDA-event times of one training iteration, B={B} T={T}; {len(rows)} stages, sum {tot:.3f} ms (stages timed warm, back to back)\n")
            for n, m, fl in rows:
                f.write(f"{n:44s} {m * 1e3:10.1f} us {fl / m / 1e9 if m > 0 and fl > 0 else 0:9.1f} TFLOP/s {100 * m / tot:5.1f}%\n")
    return {"config": f"wav2lip_train.py step (gen + L1 + sync loss {syncnet_wt}), bf16 operands / fp32 master+grads, B={B} x T={T} per GPU, "
                      f"{world} GPU(s), gradient all-reduce {'ncclAllReduce(avg) in 3 buckets overlapped with the backward' if world > 1 else 'n/a (1 GPU)'}",
            "ms_per_step": ms, "crops_per_s": world * B * T / ms * 1e3, "windows_per_s": world * B / ms * 1e3,
            "algorithmic_tflop_per_step_per_gpu": flop / 1e12, "tflops_per_gpu": flop / ms / 1e9,
            "kernel_launches_per_step": int(launches), "allreduce_bytes_per_step": int(4 * n_param) if world > 1 else 0,
            "losses_last_step": {"sync": lv[0], "l1": lv[1], "total": lv[3]}}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the reference is
    Python and cannot travel to the GPU box) on all host cores, bounded sample per step."""
    if rank != 0:
        return
    import torch
    B, T = 128, 5  # the metric's own call: one 5-D batch of 128 windows x 5 frames = 640 crops per step (same_config)
    n = B * T
    from oracle import w2l_oracle as O
    sd = O.make_state_dict("generator", 0, init="default")
    cores = pick_threads(sd, O, torch)
    mel, face = O.make_generator_inputs(B, 0, t=T)
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 1))):
            O.generator_forward(sd, mel, face)
        steps = args.steps   # a step takes seconds on the host cores: pass a small --steps for this arm
        t0 = time.perf_counter()
        for _ in range(steps):
            O.generator_forward(sd, mel, face)
        dt = (time.perf_counter() - t0) / steps
    v = n / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "crops/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "Wav2Lip.forward eval, B=128 T=5 (640 crops/GPU/step), 5-D call, fp32 in/out",
                   "global_batch_crops": n,
                   "weights": "seeded random (reference default-init statistics + randomised BatchNorm)"},
        "cpu_baseline": {"value": v, "unit": "crops/s", "cores": cores, "kind": "port",
                         "sample": f"one B=128,T=5 5-D call (640 crops) per step, {steps} steps, torch CPU fp32, best of 8/16/32/64/{os.cpu_count()} threads = {cores}"},
        "e2e": {"value": v, "unit": "crops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=B_DEFAULT, help="B (windows per GPU per step)")
    ap.add_argument("--frames", type=int, default=T_DEFAULT, help="T (frames per window)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the SyncNet / disc / mel side measurements")
    ap.add_argument("--profile-out", default=None, help="write the per-launch table to this file")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default, the driver's mode): --batch windows PER GPU.  strong: --batch is the GLOBAL batch, split over the ranks")
    ap.add_argument("--workload", default="infer", choices=["infer", "train"],
                    help="infer: the headline metric (default).  train: BASELINE configs[4], one training iteration per step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from wav2lip_b200 import _lib
    from wav2lip_b200.models import Wav2Lip
    from wav2lip_b200.parallel import max_over_ranks

    if args.warmup < 3:
        args.warmup = 3
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200; there is no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # keep NCCL's banner / debug lines off stdout: rank 0 prints exactly one JSON line there
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
            os.environ["NCCL_DEBUG"] = "NONE"
        dist.init_process_group("nccl", device_id=dev)
    if args.workload == "train":
        tb = 64 if args.batch == B_DEFAULT else args.batch
        r = measure_train(dev, rank, world, args.steps, args.warmup, B=tb, T=args.frames, profile_out=args.profile_out,
                          dump_dir=args.dump_outputs)
        if rank == 0:
            line = {"metric": "wav2lip_train.py iterations: 96x96 face-crops/sec trained (B=64/GPU, T=5, bf16)", "value": r["crops_per_s"],
                    "unit": "crops/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                    "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                    "config": {"workload": r["config"], "per_gpu_batch": tb * args.frames, "global_batch": tb * args.frames * world,
                               "parallelism": f"dp{world}", "l2": "activations of one step (~10 GB) >> L2"},
                    "gpu_launches": r["kernel_launches_per_step"] * args.steps, "train": r}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    B, T = args.batch, args.frames
    if args.scaling == "strong":
        if args.batch % world != 0:
            raise SystemExit("--scaling strong needs --batch divisible by the number of GPUs")
        B = args.batch // world      # whole T-windows per rank (parallel.shard_range): the t-major flatten stays local
    N = B * T

    # weights + inputs (seeded; every rank its own input seed, identical weights)
    import ctypes as C
    torch.manual_seed(0)
    model = Wav2Lip()  # torch's default Conv2d init == the reference constructor's init statistics
    gen = torch.Generator().manual_seed(1)
    for m in model.modules():  # randomise BatchNorm so that the folded scale/shift are not the identity
        if isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data = torch.rand(m.weight.shape, generator=gen) + 0.5
            m.bias.data = torch.randn(m.bias.shape, generator=gen) * 0.1
            m.running_mean.data = torch.randn(m.running_mean.shape, generator=gen) * 0.1
            m.running_var.data = torch.rand(m.running_var.shape, generator=gen) + 0.5
    model = model.to(dev).eval()
    gin = torch.Generator().manual_seed(100 + rank)
    mel_h = torch.rand((B, T, 1, 80, 16), generator=gin) * 8 - 4           # normalised mel range [-4, 4]
    face_h = torch.rand((B, 6, T, 96, 96), generator=gin)                  # BGR/255
    face_h[:, 0:3, :, 48:, :] = 0.0                                        # masked lower half (inference.py:136-137)
    mel_h, face_h = mel_h.pin_memory(), face_h.pin_memory()
    mel_d, face_d = mel_h.to(dev), face_h.to(dev)
    stream = torch.cuda.current_stream(dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    with torch.no_grad():
        for _ in range(args.warmup):
            out = model(mel_d, face_d)
        ctx = model._w2l_ctx
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
            time.sleep(0.25)
        l0 = ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t_wall0 = time.time()
        e0.record(stream)
        for _ in range(args.steps):
            out = model(mel_d, face_d)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        t_wall1 = time.time()
        last_out = out
        barrier()
        launches = ctx.launch_count() - l0
        ms = e0.elapsed_time(e1)
        per_rank_ms = [ms / args.steps]
        if world > 1:   # every rank's own device time: the spread shows whether a slow step is clocks or code
            box = [None] * world
            dist.all_gather_object(box, ms / args.steps)
            per_rank_ms = [float(v) for v in box]
        ms = max_over_ranks(ms, dev)
        clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
        ms_per_step = ms / args.steps
        value = world * N * args.steps / (ms * 1e-3)

        # ---- e2e: host buffers through the C-ABI host entry point, H2D + forward + D2H every step ----
        e2e = None
        if not args.no_e2e:
            out_h = torch.empty((B, 3, T, 96, 96), dtype=torch.float32).pin_memory()
            out_h2 = torch.empty((B, 3, T, 96, 96), dtype=torch.float32).pin_memory()

            def e2e_step():
                _lib.check(ctx.lib.w2l_generator_forward_host(ctx.h, C.c_void_p(mel_h.data_ptr()), C.c_void_p(face_h.data_ptr()),
                                                              C.c_void_p(out_h.data_ptr()), B, T))
            for _ in range(3):
                e2e_step()
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                e2e_step()  # synchronous: returns after the D2H copy has landed
            torch.cuda.synchronize(dev)
            dt_sync = time.perf_counter() - t0
            dt_sync = max_over_ranks(dt_sync, dev)
            barrier()
            ok = bool(torch.equal(out_h.to(dev), out))

            # the serving loop: submit batch k+1 while batch k is in flight (every step still copies its inputs up and its
            # result down inside the timed region; results land in alternating pinned buffers)
            outs = [out_h, out_h2]

            def submit(k):
                _lib.check(ctx.lib.w2l_generator_submit_host(ctx.h, C.c_void_p(mel_h.data_ptr()), C.c_void_p(face_h.data_ptr()),
                                                             C.c_void_p(outs[k & 1].data_ptr()), B, T))
            for k in range(3):
                submit(k)
                _lib.check(ctx.lib.w2l_host_wait(ctx.h, 1))
            _lib.check(ctx.lib.w2l_host_wait(ctx.h, 0))
            out_h2.zero_()
            barrier()
            t0 = time.perf_counter()
            for k in range(args.steps):
                submit(k)
                _lib.check(ctx.lib.w2l_host_wait(ctx.h, 1))   # batch k-1 is complete in host memory here
            _lib.check(ctx.lib.w2l_host_wait(ctx.h, 0))
            dt = time.perf_counter() - t0
            dt = max_over_ranks(dt, dev)
            barrier()
            ok = ok and bool(torch.equal(out_h.to(dev), out)) and bool(torch.equal(out_h2.to(dev), out))
            e2e = {"value": world * N * args.steps / dt, "unit": "crops/s",
                   "h2d_bytes_per_step": int(mel_h.numel() * 4 + face_h.numel() * 4),
                   "d2h_bytes_per_step": int(out_h.numel() * 4), "result_matches_device_path": ok,
                   "api": "w2l_generator_submit_host + w2l_host_wait(1): pinned host buffers, two batches in flight "
                          "(H2D of step k+1 and D2H of step k-1 overlap the kernels of step k)",
                   "timer": "host wall clock around the whole loop, drained at the end",
                   "synchronous_call": {"value": world * N * args.steps / dt_sync, "unit": "crops/s",
                                        "api": "w2l_generator_forward_host: one blocking call per step, as inference.py:259-265"}}

        # ---- roofline: per-launch CUDA-event timing of the conv kernel family (after the timed region) ----
        out = model(mel_d, face_d)  # make the full-batch plan the profiled one again (the host path runs chunk plans)
        torch.cuda.synchronize(dev)
        peaks = load_peaks()
        prof = ctx.profile_plan(_lib.NET_GENERATOR, iters=3, stream=stream.cuda_stream)
        conv_ms = sum(m for _, m, _ in prof)
        conv_flop = sum(f for _, _, f in prof)
        achieved = conv_flop / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
        roofline = {"bound": "tensor", "kernel": "conv_igemm_kernel<BN,BK> (tcgen05 implicit GEMM, all conv launches of one step)",
                    "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
                    "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['src']}); fp16 operands run at the bf16 rate",
                    "launches_per_step": len(prof), "conv_ms_per_step_isolated": conv_ms,
                    "share_of_step": conv_ms / ms_per_step if ms_per_step > 0 else None,
                    "whole_step_tflops": value / world * FLOP_PER_CROP / 1e12,
                    "traffic": None}
        # DRAM bytes of the same launches from the committed ncu capture (profiles/), valid for the default workload
        tname = next((n for n in ("r2_final_ncu_dram_per_step.json", "r1_final_ncu_dram_per_step.json")
                      if os.path.exists(os.path.join(ROOT, "profiles", n))), None)
        if tname and (B, T) == (B_DEFAULT, T_DEFAULT):
            tj = json.load(open(os.path.join(ROOT, "profiles", tname)))
            roofline["traffic"] = tj["dram_read_bytes"] + tj["dram_write_bytes"]
            roofline["traffic_note"] = ("dram__bytes_read+write summed over the %d conv launches of one step (ncu, profiles/"
                                        "%s); algorithmic conv in+out bytes per step = %.2f GB"
                                        % (tj["launches"], tname, (4.81e6 + 4.49e6) * 2 * N / 1e9))
        if args.profile_out and rank == 0:
            with open(args.profile_out, "w") as f:
                f.write(f"# per-launch CUDA-event times, B={B} T={T} (N={N}), {len(prof)} conv launches, sum {conv_ms:.3f} ms\n")
                for nm, m, fl in prof:
                    f.write(f"{nm:36s} {m * 1e3:10.1f} us {fl / m / 1e9 if m > 0 else 0:9.1f} TFLOP/s {100 * m / conv_ms:5.1f}%\n")

    # ---- the other hot-path entry points (BASELINE configs[2], configs[3]); informational, outside the timed region ----
    extra = None
    if rank == 0 and world == 1 and not args.no_extra:
        extra = measure_extra(dev)
        try:
            extra["train_step"] = measure_train(dev, 0, 1, steps=5, warmup=3)
        except Exception as e:  # the training row must not take the headline line down
            extra["train_step"] = {"error": repr(e)[:300]}

    # ---- CPU baseline (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, dt, cores = cpu_baseline_run(128)
        cpu = {"value": v, "unit": "crops/s", "cores": cores, "kind": "port",
               "sample": f"one N=128 4-D batch (inference.py batch) = {dt:.2f} s of oracle/w2l_oracle.py (torch CPU fp32; "
                         f"{cores} threads = the fastest of 8/16/32/64/{os.cpu_count()} on this host)"}

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"generator_out": last_out})

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "crops/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f16", "data": "synthetic", "per_rank_ms_per_step": per_rank_ms,
            "config": {"workload": f"BASELINE configs[1] at the metric's B={B}, T={T}: Wav2Lip.forward eval, {N} crops/GPU/step, fp32 NCHW in/out",
                       "per_gpu_batch": N, "global_batch": N * world, "parallelism": f"replicas x{world}, batch-sharded, no collective",
                       "weights": "seeded random (reference default-init statistics + randomised BatchNorm)",
                       "l2": "inputs larger than L2 (141 MB face + activations >> 126 MB), no explicit flush",
                       "precision": "fp16 operands / fp32 accumulate+epilogue (TF32-class mantissa)"},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "extra": extra,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
