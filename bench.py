#!/usr/bin/env python
"""bench.py -- C-ViViT encode frames/s (headline, BASELINE.json configs[1]) + MaskGIT sample tokens/s.

    python bench.py --gpus N --steps K --warmup W            # this framework (libphk.so, sm_100a)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port), rank 0

A "step" is one pass of the hot path over one batch of synthetic input: one
``CViViT(video, return_only_codebook_ids=True)`` on (8,3,17,256,256) per GPU (weak scaling: every rank
encodes its own 8 videos, no collective on the data path).  One JSON line on rank 0.
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

CFG2 = dict(dim=512, codebook_size=65536, image_size=256, patch_size=32, temporal_patch_size=2, spatial_depth=4,
            temporal_depth=4, dim_head=64, heads=8, use_vgg_and_gan=False)
VIDEO = (8, 3, 17, 256, 256)
CFG3 = dict(dim=512, num_tokens=65536, max_seq_len=1024, dim_context=768, depth=6)
CFG3_RUN = dict(batch=4, num_frames=17, steps=18, ctx_len=16, cond_scale=3.0)
# SURVEY.md 8(d): algorithmic FLOPs (2*M*N*K per product, UNPADDED dims)
ENCODE_GFLOP = 264.8        # whole encode call
ENCODE_GEMM_GFLOP = 259.28  # its nn.Linear products: patch embed 27.38 + 2 x (projections 38.66 + feed-forward 77.29)
MASKGIT_FWD_GFLOP = 277.1   # one MaskGit forward at b=4, N=576, L=16 (head 154.6, FF 58.0, self 45.3, cross 15.6, ...)
MASKGIT_HEAD_GFLOP = 154.6  # to_logits over all b*N rows, one forward
# algorithmic operand + output bytes of the encode's 33 GEMM launches, MB (M = 4608 tokens, dim 512, bf16 operands):
#   8 x out-proj  (A 4.7 + W 0.5 + fp32 residual in 9.4 + out 9.4)      = 24.0 each
#   8 x FF2       (A 13.0 + W 1.4 + residual in 9.4 + out 9.4)         = 33.2
#   8 x FF1+GEGLU (A 4.7 + W 2.9 + bf16 out 12.6)                      = 20.2
#   8 x q / k,v   (A 2 x 4.7 + W 1.6 + bf16 out 14.2)                  = 25.2
#   1 x patch embeddings (A 50.3 + 3.1, W 6.3 + 3.1, fp32 out 9.4)     = 72.2
ENCODE_GEMM_ALGORITHMIC_MB_PER_LAUNCH = (8 * 24.0 + 8 * 33.2 + 8 * 20.2 + 8 * 25.2 + 72.2) / 33


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"],
                    src="MEASURED_PEAKS.json")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: an NVML polling thread (2 ms period -- the timed
    region is only tens of milliseconds), `nvidia-smi -lms` as the fallback when NVML cannot be loaded."""
    SMI_Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines, self.samples = index, None, [], []
        self.stop_flag, self.thread, self.nvml, self.handle, self.window = False, None, None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
        except Exception:
            self.nvml = None

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if index < len(ids) and ids[index].isdigit():
                return int(ids[index])
        return index

    def _poll(self):
        n = self.nvml
        get_reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        power, i = 0.0, 0
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                reasons = get_reasons(self.handle)
                if i % 8 == 0:  # the power query is the slow one (milliseconds)
                    power = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                self.samples.append((sm, reasons, power, time.perf_counter()))
                i += 1
            except Exception:
                pass
            time.sleep(0.003)  # (a 1 ms poll took a measurable share of a core from the launching thread)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.SMI_Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def report(self, window):
        """Clock record of one timed window (a perf_counter pair) while the poller keeps running (NVML path only)."""
        if self.nvml is None:
            return None
        return self._nvml_summary(list(self.samples), window)

    def _nvml_summary(self, samples, window):
        n = self.nvml
        # keep the samples taken inside the timed window (the poller starts during warm-up so that its first, slow NVML
        # calls are over); if the window was shorter than one polling period keep the nearest ones
        inside = [x for x in samples if window[0] <= x[3] <= window[1]] if window else []
        if len(inside) < 3 and samples and window:
            mid = 0.5 * (window[0] + window[1])
            inside = sorted(samples, key=lambda x: abs(x[3] - mid))[:3]
        samples = [x[:3] for x in (inside or samples)]
        if not samples:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        bits = {"hw_slowdown": getattr(n, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted(k for k, b in bits.items() if any(r & b for _, r, _ in samples))
        try:
            mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        except Exception:
            mx = None
        return dict(sm_mhz=statistics.median(s for s, _, _ in samples), sm_max_mhz=mx,
                    power_w_max=max(p for _, _, p in samples), samples=len(samples), reasons=reasons,
                    source="nvml, ~4 ms period")

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1)
            return self._nvml_summary(self.samples, self.window)
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), power_w_max=max(power), samples=len(sm),
                    reasons=sorted(reasons), source="nvidia-smi -lms 100")


def tune_cpu_threads(fn, candidates=None):
    """The host may expose far more hardware threads than the eager ATen path can use (128 on the GPU boxes: oversubscribed
    GEMMs run ~10x slower than with 16-32 threads).  Times one call per candidate and keeps the fastest."""
    import torch
    n = os.cpu_count() or 1
    cands = sorted({c for c in (candidates or [8, 16, 32, 64, n]) if 1 <= c <= n})
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        fn()
        t0 = time.perf_counter()
        fn()
        fn()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def _cfg2_state():
    import torch
    import phenaki_pytorch_b200 as P
    torch.manual_seed(0)
    return {k: v.detach() for k, v in P.CViViT(**CFG2).state_dict().items()}


def cpu_encode_baseline(seconds_budget=12.0, batch=2):
    """The reference's CPU path (oracle port: same ATen ops, all host threads) on a BOUNDED sample of the
    same workload: `batch` video(s) of cfg2 per call."""
    import torch
    from oracle import phenaki_oracle as O
    sd = _cfg2_state()
    video = torch.randn(batch, *VIDEO[1:])
    with torch.no_grad():
        cores = tune_cpu_threads(lambda: O.cvivit_codebook_ids(video, sd, (256, 256), (32, 32)))
        t0, n = time.perf_counter(), 0
        while True:
            O.cvivit_codebook_ids(video, sd, (256, 256), (32, 32))
            n += 1
            dt = time.perf_counter() - t0
            if dt > seconds_budget or n >= 400:
                break
    fps = n * batch * VIDEO[2] / dt
    return dict(value=fps, unit="frames/s", cores=cores, kind="port",
                sample=f"{n} x oracle C-ViViT cfg2 encode of ({batch},3,17,256,256) fp32, torch {torch.__version__} "
                       f"CPU eager, {torch.get_num_threads()} threads (best of 8/16/32/64/{os.cpu_count()}), {dt:.1f}s")


def cpu_maskgit_baseline(loop_steps=2):
    """The reference's demasking loop on the host cores (oracle port), bounded: the first `loop_steps` of the 18
    iterations at the full b=4 (each iteration = 2 MaskGit forwards + the V-wide gumbel / softmax / top-k tail)."""
    import torch
    from oracle import phenaki_oracle as O
    import phenaki_pytorch_b200 as P
    torch.manual_seed(1)
    sd = {k: v.detach() for k, v in P.MaskGit(**CFG3).state_dict().items()}
    b, L = CFG3_RUN["batch"], CFG3_RUN["ctx_len"]
    ctx = torch.randn(b, L, 768)

    class Stop(Exception):
        pass

    class StopAfter(list):  # the oracle appends one trace record per finished iteration
        def __init__(self, n):
            super().__init__()
            self.n = n

        def append(self, rec):
            super().append(rec)
            if len(self) >= self.n:
                raise Stop()

    def run(steps_run):
        # the schedule depends on the total step count: run the FIRST iterations of the 18-step loop (the last one
        # stops before its confidence scores, a few percent of an iteration in the CPU's favour)
        try:
            O.sample_token_ids(sd, num_tokens=576, patch_shape=(9, 8, 8), batch=b, steps=CFG3_RUN["steps"],
                               text_embeds=ctx, cond_scale=CFG3_RUN["cond_scale"],
                               noise_fn=lambda shape, tag: torch.zeros(shape).uniform_(0, 1), trace=StopAfter(steps_run))
        except Stop:
            pass

    with torch.no_grad():
        torch.set_num_threads(min(32, os.cpu_count() or 1))
        run(1)  # warm-up (allocator, thread pool)
        t0 = time.perf_counter()
        run(loop_steps)
        dt = time.perf_counter() - t0
    return dict(value=b * 576 * loop_steps / dt, unit="tokens/s", cores=torch.get_num_threads(), kind="port",
                s_per_decode_step=dt / loop_steps,
                sample=f"first {loop_steps} of 18 demasking iterations at b={b}, N=576, V=65536, cond_scale 3 (oracle port of "
                       f"Phenaki.sample, CPU fp32 eager ATen, {torch.get_num_threads()} threads), {dt:.1f}s")


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (oracle port), rank 0 only, on the FULL
    configs[1] batch (8 videos per step)."""
    if rank != 0:
        return
    per_step = VIDEO[0]
    import torch
    from oracle import phenaki_oracle as O
    sd = _cfg2_state()
    video = torch.randn(per_step, *VIDEO[1:])
    small = video[:2].contiguous()
    with torch.no_grad():
        cores = tune_cpu_threads(lambda: O.cvivit_codebook_ids(small, sd, (256, 256), (32, 32)))
        for _ in range(args.warmup):
            O.cvivit_codebook_ids(video, sd, (256, 256), (32, 32))
        steps = min(args.steps, 100)
        t0 = time.perf_counter()
        for _ in range(steps):
            O.cvivit_codebook_ids(video, sd, (256, 256), (32, 32))
        dt = time.perf_counter() - t0
    fps = steps * per_step * VIDEO[2] / dt
    sample = (f"{steps} steps x the full ({per_step},3,17,256,256) cfg2 batch, oracle port of the reference (CPU fp32 "
              f"eager ATen, {cores} threads = best of 8/16/32/64/{os.cpu_count()})")
    out = {
        "impl": "reference", "metric": "cvivit_encode_frames_per_s", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": dt / steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[1]: CViViT(dim=512,image=256,patch=32,pt=2,depth=4+4,heads=8,"
                               "codebook=65536) encode+LFQ ids of (8,3,17,256,256) fp32 per GPU, random-init weights",
                   "batch_per_gpu": per_step, "frames": VIDEO[2],
                   "note": "host CPU, oracle port of the reference modules (kind: port -- /root/reference is not on the "
                           "GPU box), thread count auto-tuned"},
        "cpu_baseline": dict(value=fps, unit="frames/s", cores=cores, kind="port", sample=sample),
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if not args.no_maskgit:
        try:
            out["maskgit"] = cpu_maskgit_baseline()
        except Exception as ex:
            out["maskgit"] = {"error": repr(ex)}
    print(json.dumps(out))


def _timed(fn, iters, barrier):
    """CUDA-event time of `iters` calls on the current stream, bracketed by barrier + synchronize."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    out = None
    for _ in range(iters):
        out = fn()
    e1.record()
    _timed.host_enqueue_ms = (time.perf_counter() - t0) * 1e3  # how long the host took to ISSUE the work (no sync inside)
    barrier()
    return e0.elapsed_time(e1), (t0, time.perf_counter()), out


def bench_maskgit(dev, prec, world, barrier, sampler, samples_timed=6):
    """configs[2]: MaskGit(dim=512, depth=6, seq=1024, ctx=768) 18-step demasking loop, b=4 per GPU, 17 frames.
    Device-resident `value`, `e2e` through Phenaki.sample (pinned host text embeddings in, host ids out), roofline on
    algorithmic and on executed FLOPs, launches per iteration."""
    import torch
    import phenaki_pytorch_b200 as P
    from phenaki_pytorch_b200 import _lib as L
    from phenaki_pytorch_b200 import sharding as S
    lib = L.lib()
    torch.manual_seed(1)
    cv = P.CViViT(**CFG2).to(dev)
    mg = P.MaskGit(**CFG3).to(dev)
    cv.precision = mg.precision = prec
    ph = P.Phenaki(cvivit=cv, maskgit=mg, steps=CFG3_RUN["steps"], text_embed_dim=768).eval()
    ph.cvivit.precision = prec
    if os.environ.get("PHK_FUSED_HEAD") is not None:   # A/B: fused logits-head kernel vs head GEMM + sampling kernel
        ph.fused_head = os.environ["PHK_FUSED_HEAD"] != "0"
    b, Lc, steps = CFG3_RUN["batch"], CFG3_RUN["ctx_len"], CFG3_RUN["steps"]
    host_ctx = torch.randn(b, Lc, 768)
    host_ctx[1, Lc // 2:] = 0
    host_ctx = host_ctx.pin_memory()
    ctx = host_ctx.to(dev)
    n = cv.num_tokens_per_frames(CFG3_RUN["num_frames"])
    shape = cv.get_video_patch_shape(CFG3_RUN["num_frames"])
    run = lambda: ph.sample_token_ids(num_tokens=n, patch_shape=shape, batch_size=b, text_embeds=ctx,
                                      cond_scale=CFG3_RUN["cond_scale"])
    for _ in range(3):  # warm-up: tables, caches, (one-launch mode) eager call + capture + first replay
        run()
    l0 = lib.phk_launch_count()
    ms_total, window, ids = _timed(run, samples_timed, barrier)
    launches = lib.phk_launch_count() - l0
    ms = S.max_over_ranks(ms_total, dev) / samples_timed
    assert int((ids == mg.mask_id).sum()) == 0
    # e2e: the public call, host buffers in and out every sample
    e2e_fn = lambda: ph.sample(num_frames=CFG3_RUN["num_frames"], text_embeds=host_ctx, cond_scale=CFG3_RUN["cond_scale"],
                               return_token_ids=True).cpu()
    e2e_fn()
    barrier()
    t0 = time.perf_counter()
    for _ in range(samples_timed):
        e2e_fn()
    torch.cuda.synchronize()
    e2e_ms = S.max_over_ranks((time.perf_counter() - t0) * 1e3, dev) / samples_timed
    tokens = b * n * steps
    pk = peaks()
    alg_gflop = 2 * MASKGIT_FWD_GFLOP * steps
    # executed: the logits head only on the still-masked rows (576, k_1, ..., k_17 of 576 per sequence) and the first
    # layer's PEG + self-attention once for the CFG pair -- DESIGN 4.3
    ks = [n] + P.phenaki.demask_counts(n, steps)
    head_rows = sum(ks) / (n * steps)
    exec_gflop = alg_gflop - 2 * MASKGIT_HEAD_GFLOP * steps * (1 - head_rows) - steps * (45.3 / 6 / 2 + 0.4 / 6 / 2)
    graphs = int(launches) <= samples_timed * steps  # one cudaGraphLaunch per iteration counted as its kernels by the library
    out = dict(metric="maskgit_sample_tokens_per_s", value=world * tokens / ms * 1e3, unit="tokens/s", ms_per_sample=ms,
               ms_per_decode_step=ms / steps, samples_timed=samples_timed, n_gpus=world,
               config=dict(workload=f"BASELINE.json configs[2]: MaskGit(dim=512,depth=6,V=65536,ctx=768) {steps}-step "
                                    f"Phenaki.sample demasking loop, b={b} per GPU, N={n}, L={Lc}, cond_scale=3 (2 forwards "
                                    f"per step as one batch of {2 * b}), in-kernel Philox gumbel noise",
                           one_launch_per_iteration=bool(getattr(ph, "iteration_call", False)),
                           fused_head=bool(ph.fused_head)),
               e2e=dict(value=world * tokens / e2e_ms * 1e3, unit="tokens/s", ms_per_sample=e2e_ms,
                        h2d_bytes_per_step=int(host_ctx.numel() * 4), d2h_bytes_per_step=int(b * n * 8),
                        api="Phenaki.sample(text_embeds=<pinned host tensor>, return_token_ids=True).cpu(): text embeddings "
                            "H2D, text keys/values, 18 iterations, ids D2H inside the timed region"),
               roofline=dict(bound="tensor", kernel="whole demasking iteration", unit="TFLOP/s",
                             achieved=alg_gflop / ms, peak=pk["tf_sustained"], frac=alg_gflop / ms / pk["tf_sustained"],
                             achieved_on_executed_flops=exec_gflop / ms,
                             frac_on_executed_flops=exec_gflop / ms / pk["tf_sustained"],
                             algorithmic_gflop_per_sample=alg_gflop, executed_gflop_per_sample=exec_gflop,
                             peak_source=pk["src"] + " (sustained bf16)", traffic=None,
                             note="algorithmic = SURVEY 8d (all rows, both CFG halves, every layer: 554.1 GFLOP per "
                                  "iteration); executed = head on the still-masked rows only, first layer's PEG + "
                                  "self-attention once per CFG pair"),
               gpu_launches=int(launches), kernels_per_iteration=launches / (samples_timed * steps),
               launches_per_iteration=1 if getattr(ph, "iteration_call", False) else launches / (samples_timed * steps),
               launch_scheme=("one cudaGraphLaunch per demasking iteration (phk_maskgit_demask_iteration: re-mask, CFG-pair "
                              "forward, logits head on the masked rows, noise-counter advance = kernels_per_iteration kernels "
                              "inside the graph)" if getattr(ph, "iteration_call", False) else "one PDL-chained launch sequence per iteration"),
               clocks=sampler.report(window) if sampler is not None else None)
    return out


def bench_train(dev, prec, world, barrier, sampler, steps_timed=5):
    """BASELINE configs[3] (SURVEY 8f-2): Phenaki.forward + backward (C-ViViT tokenises the raw videos, MaskGit masked-token
    cross entropy, hand-written backward kernels), 4 videos of (3,17,256,256) per GPU, data parallel: the flat fp32
    gradient bucket is averaged over the ranks by ONE NCCL all-reduce per step (what the reference gets from DDP)."""
    import torch
    import torch.distributed as dist
    import phenaki_pytorch_b200 as P
    from phenaki_pytorch_b200 import sharding as S
    torch.manual_seed(2)
    cv = P.CViViT(**CFG2).to(dev)
    mg = P.MaskGit(**CFG3).to(dev)
    cv.precision = mg.precision = prec
    ph = P.Phenaki(cvivit=cv, maskgit=mg, steps=CFG3_RUN["steps"], text_embed_dim=768).to(dev).train()
    ph.cvivit.precision = prec
    b = 4
    videos = torch.randn((b, 3, 17, 256, 256), device=dev)
    ctx = torch.randn((b, CFG3_RUN["ctx_len"], 768), device=dev)

    def step():
        for p_ in mg.parameters():
            p_.grad = None
        loss = ph(videos, text_embeds=ctx)
        loss.backward()   # hands out the gradients the C call computed; averages the bucket over the ranks (NCCL)
        return loss

    for _ in range(2):
        loss = step()
    ms_total, window, loss = _timed(step, steps_timed, barrier)
    ms = S.max_over_ranks(ms_total, dev) / steps_timed
    nparams = sum(p_.numel() for p_ in mg.parameters())
    out = dict(metric="phenaki_train_tokens_per_s", value=world * b * 576 / ms * 1e3, unit="tokens/s", ms_per_step=ms,
               videos_per_s=world * b / ms * 1e3, steps_timed=steps_timed, loss=float(loss), n_gpus=world,
               config=dict(workload="BASELINE.json configs[3]: Phenaki forward+backward (C-ViViT encode of the raw videos, "
                                    f"MaskGit(dim=512,depth=6,V=65536) masked CE), {b} x (3,17,256,256) per GPU, bf16 products",
                           global_batch=b * world, parallelism=f"dp{world}: one flat fp32 gradient bucket, NCCL all-reduce (mean) launched slice by slice while the backward runs"),
               approx_tflops=3 * MASKGIT_FWD_GFLOP * b / 4 / ms,
               maskgit_parameters=nparams, peak_mem_gb=torch.cuda.max_memory_allocated(dev) / 2 ** 30,
               clocks=sampler.report(window) if sampler is not None else None)
    if world > 1:  # the collective alone: bus bandwidth of the bucket all-reduce
        flat = torch.zeros(nparams, dtype=torch.float32, device=dev)
        for _ in range(2):
            dist.all_reduce(flat)
        ar_ms, _, _ = _timed(lambda: dist.all_reduce(flat), 5, barrier)
        ar_ms = S.max_over_ranks(ar_ms, dev) / 5
        out["all_reduce"] = dict(bytes=nparams * 4, ms=ar_ms, algbw_gbs=nparams * 4 / ar_ms / 1e6,
                                 busbw_gbs=nparams * 4 / ar_ms / 1e6 * 2 * (world - 1) / world,
                                 share_of_step=ar_ms / ms)
        out["overlap"] = ("sliced all-reduce on a side stream as the backward finishes each gradient group"
                          if "_overlap_cache" in mg.__dict__ else "one all-reduce of the whole bucket after the step")
    return out


def bench_make_video(dev, prec, world, barrier, sampler, chains_timed=3, b=2):
    """BASELINE configs[4]: Phenaki.sample with a TokenCritic and cond_scale 5, sliding-window scene chain of
    3 scenes x (17, 14, 14) frames primed with the last 5 frames of the previous scene (make_video,
    phenaki_pytorch.py:692-714), `b` prompts per GPU (batch-sharded over the GPUs, no collective)."""
    import torch
    import phenaki_pytorch_b200 as P
    from phenaki_pytorch_b200 import sharding as S
    torch.manual_seed(3)
    cv = P.CViViT(**CFG2).to(dev)
    mg = P.MaskGit(**CFG3).to(dev)
    cr = P.TokenCritic(dim=512, num_tokens=65536, max_seq_len=1024, has_cross_attn=True, depth=6, dim_context=768).to(dev)
    cv.precision = mg.precision = cr.precision = prec
    ph = P.Phenaki(cvivit=cv, maskgit=mg, critic=cr, steps=CFG3_RUN["steps"], text_embed_dim=768).eval()
    ph.cvivit.precision = prec
    frames, prime = (17, 14, 14), 5
    embeds = [torch.randn((b, CFG3_RUN["ctx_len"], 768), device=dev) for _ in frames]

    def chain():
        scenes, pf = [], None
        for nf, e in zip(frames, embeds):
            video = ph.sample(text_embeds=e, prime_frames=pf, num_frames=nf, cond_scale=5.0)
            scenes.append(video)
            pf = video[:, :, -prime:].contiguous()
        return torch.cat(scenes, dim=2)

    video = chain()
    assert tuple(video.shape) == (b, 3, sum(frames), 256, 256) and bool(torch.isfinite(video).all())
    chain()  # second warm-up: every workspace / weight table / bias table of the three scene shapes exists
    ms_total, window, _ = _timed(chain, chains_timed, barrier)
    host_ms = _timed.host_enqueue_ms / chains_timed
    ms = S.max_over_ranks(ms_total, dev) / chains_timed
    new_tokens = sum(cv.num_tokens_per_frames(nf, include_first_frame=(i == 0)) for i, nf in enumerate(frames))
    return dict(metric="make_video_tokens_per_s", value=world * b * new_tokens * CFG3_RUN["steps"] / ms * 1e3, unit="tokens/s",
                ms_per_chain=ms, videos_per_s=world * b / ms * 1e3, frames_per_s=world * b * sum(frames) / ms * 1e3,
                chains_timed=chains_timed, n_gpus=world, host_enqueue_ms_per_chain=host_ms,
                config=dict(workload=f"BASELINE.json configs[4]: 3-scene chain x {frames} frames, prime {prime}, TokenCritic "
                                     f"(cross-attn, depth 6), cond_scale 5, 18 steps per scene, {b} prompts per GPU; each "
                                     "scene = tokenise prime frames + demasking loop (MaskGit + critic CFG pairs) + C-ViViT decode",
                            prompts_per_gpu=b, global_prompts=b * world, new_tokens_per_video=new_tokens,
                            parallelism=f"dp{world}: prompts batch-sharded, no data-path collective"),
                clocks=sampler.report(window) if sampler is not None else None)


def reference_gpu_leg(dev, maskgit=True):
    """SURVEY 2a / 8d: the reference's own PyTorch path on this B200 (oracle port on CUDA, eager fp32 and autocast
    bf16) -- the same-box bar the build must beat."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import ref_gpu_bench as R
    out = dict(encode=R.encode_leg(dev))
    if maskgit:
        out["maskgit"] = R.maskgit_leg(dev, iters=1)
    return out


def dump_outputs(directory, **arrays):
    """Writes each array as `directory/<name>.npy` in float64 so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().cpu().double().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--prec", default=os.environ.get("PHK_PREC", "bf16"), choices=["f32", "bf16", "bf16x3"])
    ap.add_argument("--no-maskgit", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-refgpu", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the configs[3] training-step block")
    ap.add_argument("--no-makevideo", action="store_true", help="skip the configs[4] make_video block")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the token ids of the last timed encode step to DIR/codebook_ids.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import ctypes as C
    import phenaki_pytorch_b200 as P
    from phenaki_pytorch_b200 import _lib as L
    from phenaki_pytorch_b200 import sharding as S

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps
    prec = {"bf16": L.PREC_BF16, "f32": L.PREC_F32, "bf16x3": getattr(L, "PREC_BF16X3", L.PREC_F32)}[args.prec]
    lib = L.lib()

    torch.manual_seed(0)
    model = P.CViViT(**CFG2).to(dev).eval()
    model.precision = prec
    B, Cc, F, H, Wd = VIDEO
    # three distinct input buffers (3 x 107 MB > 126 MB L2) so no timed step finds its video in L2
    host = [torch.randn(VIDEO, generator=torch.Generator().manual_seed(100 + rank * 10 + i)).pin_memory()
            for i in range(3)]
    vids = [h.to(dev, non_blocking=True) for h in host]
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # setup, untimed: the library captures one CUDA graph per (input buffer, shape) on the second call with that key
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()   # polls from here on (the first NVML calls take ~10 ms); only samples inside the timed window are reported
    for v in vids:
        for _ in range(3):
            model(v, return_only_codebook_ids=True)
    for i in range(W):
        ids = model(vids[i % 3], return_only_codebook_ids=True)
    barrier()
    launches0 = lib.phk_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_window = time.perf_counter()
    e0.record()
    t_submit = time.perf_counter()
    for i in range(K):
        ids = model(vids[i % 3], return_only_codebook_ids=True)
    t_submit = time.perf_counter() - t_submit   # host time to enqueue the K steps (launch-bound if close to the GPU time)
    e1.record()
    barrier()
    enc_window = (t_window, time.perf_counter())
    sampler.window = enc_window
    ms_total = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, codebook_ids=ids)
    launches = lib.phk_launch_count() - launches0
    clocks = (sampler.report(enc_window) or None) if rank == 0 else None
    ms_total = S.max_over_ranks(ms_total, dev)   # the job is as slow as its slowest rank
    ms_step = ms_total / K
    value = world * B * F * K / (ms_total / 1e3)

    # the K-step window is tens of milliseconds (power and clocks have not settled): also a long run of the same loop
    KS = 1500
    e0.record()
    t_sus = time.perf_counter()
    for i in range(KS):
        model(vids[i % 3], return_only_codebook_ids=True)
    e1.record()
    barrier()
    sus_window = (t_sus, time.perf_counter())
    sus_ms = S.max_over_ranks(e0.elapsed_time(e1), dev) / KS
    sustained = dict(steps=KS, ms_per_step=sus_ms, value=world * B * F / sus_ms * 1e3, unit="frames/s",
                     step_frac_of_tensor_peak=ENCODE_GFLOP / sus_ms / peaks()["tf_sustained"],
                     clocks=(sampler.report(sus_window) or None) if rank == 0 else None)

    # ---- e2e: the C-ABI call with HOST buffers (pinned), H2D + encode + D2H inside the timed region ----
    KE = min(K, 40)
    table = model._table()
    tp, hh, ww = model.get_video_patch_shape(F)
    host_ids = torch.empty((B, tp, hh, ww), dtype=torch.int64).pin_memory()
    dev_ids = torch.empty((B, tp, hh, ww), dtype=torch.int64, device=dev)
    stage = torch.empty(VIDEO, dtype=torch.float32, device=dev)
    nbytes = lib.phk_cvivit_workspace_bytes(C.byref(table), B, F, prec)
    ws = model._ws.get(nbytes, dev)
    bias = model._spatial_bias(table, dev)

    def e2e_step(i):
        L.check(lib.phk_cvivit_encode_host(C.byref(table), L.ptr(host[i % 3]), B, F, L.ptr(host_ids), L.ptr(stage),
                                           L.ptr(dev_ids), L.ptr(ws), ws.numel(), prec, L.ptr(bias), L.stream_ptr()),
                "phk_cvivit_encode_host")

    for i in range(3):
        e2e_step(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(KE):
        e2e_step(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert torch.equal(host_ids, model(vids[(KE - 1) % 3], return_only_codebook_ids=True).cpu())
    e2e_sync_value = world * B * F * KE / S.max_over_ranks(e2e_s, dev)

    # the same through the public streaming API (CViViT.encode_host_iter -> phk_encode_pipe_*): every step still does
    # its own H2D from pinned memory and D2H of the ids, but batch i+1's copy overlaps batch i's encode
    for _ in model.encode_host_iter((host[i % 3] for i in range(3)), device=dev):
        pass
    barrier()
    t0 = time.perf_counter()
    last = None
    for last in model.encode_host_iter((host[i % 3] for i in range(KE)), device=dev):
        pass
    torch.cuda.synchronize()
    e2e_pipe_s = time.perf_counter() - t0
    assert torch.equal(last, host_ids)
    e2e_value = world * B * F * KE / S.max_over_ranks(e2e_pipe_s, dev)

    # ---- per-kernel-family device time (CUDA events on the launching stream) over 3 more steps ----
    lib.phk_prof_enable(1)
    PROF_STEPS = 3
    for i in range(PROF_STEPS):
        model(vids[i % 3], return_only_codebook_ids=True)
    torch.cuda.synchronize()
    lib.phk_prof_enable(0)
    fam = L.profile_collect()
    tot = sum(v[0] for v in fam.values()) or 1.0
    shares = {k: round(v[0] / tot, 4) for k, v in sorted(fam.items(), key=lambda kv: -kv[1][0])}
    pk = peaks()
    dom = max(fam, key=lambda k: fam[k][0])
    dms, dcalls, dwork = fam[dom]
    if dom.startswith("gemm") or dom == "attention":
        # the family's ALGORITHMIC FLOPs: unpadded 2*M*N*K of the reference's nn.Linear products (the kernels multiply
        # the zero-padded 1365 -> 1408 feed-forward width as well; that padding is not counted as work)
        alg = ENCODE_GEMM_GFLOP * 1e9 * PROF_STEPS if dom.startswith("gemm") and prec != L.PREC_F32 else dwork
        achieved = alg / (dms * 1e-3) / 1e12
        roof = dict(bound="tensor", kernel=dom, achieved=achieved, peak=pk["tf_sustained"], unit="TFLOP/s",
                    frac=achieved / pk["tf_sustained"], traffic=None,
                    per_launch=dict(flops=alg / dcalls, executed_flops_incl_padding=dwork / dcalls, ms=dms / dcalls),
                    peak_source=pk["src"] + " (sustained bf16)")
    else:
        achieved = dwork / (dms * 1e-3) / 1e9
        roof = dict(bound="hbm", kernel=dom, achieved=achieved, peak=pk["hbm"], unit="GB/s", frac=achieved / pk["hbm"],
                    traffic=None, per_launch=dict(bytes=dwork / dcalls, ms=dms / dcalls), peak_source=pk["src"])
    # DRAM bytes per launch of the dominant family, from the committed `ncu --set full` capture (not measured live)
    for tname in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if os.path.exists(tpath):
            tj = json.load(open(tpath)).get(dom)
            if tj:
                roof["traffic"], roof["traffic_source"] = tj["dram_bytes_per_launch"], tj["source"]
                if dom == "gemm_bf16":  # what the same launches move algorithmically: traffic above it = wasted re-reads
                    roof["algorithmic_bytes_per_launch"] = ENCODE_GEMM_ALGORITHMIC_MB_PER_LAUNCH * 1e6
                break
    roof["family_share_of_step"] = shares
    roof["family_launches_per_step"] = {k: v[1] // PROF_STEPS for k, v in fam.items()}
    roof["step_tflops"] = ENCODE_GFLOP / ms_step  # whole-step algorithmic FLOPs / device time
    roof["step_frac_of_tensor_peak"] = roof["step_tflops"] / pk["tf_sustained"]
    roof["step_frac_of_burst_peak"] = roof["step_tflops"] / pk["tf_burst"]

    out = {
        "metric": "cvivit_encode_frames_per_s", "value": value, "unit": "frames/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.prec, "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[1]: CViViT(dim=512,image=256,patch=32,pt=2,depth=4+4,heads=8,"
                               "codebook=65536) encode+LFQ ids of (8,3,17,256,256) fp32 per GPU, random-init weights",
                   "batch_per_gpu": B, "global_batch": B * world, "frames": F,
                   "parallelism": f"dp{world}: batch-sharded, one process per GPU, no data-path collective",
                   "l2": "inputs rotate over 3 device buffers (3 x 107 MB > 126 MB L2)",
                   "precision_mode": {"f32": "PHK_PREC_F32 (fp32 FFMA GEMMs, parity mode)",
                                      "bf16": "PHK_PREC_BF16 (tcgen05 bf16 GEMMs, fp32 accumulate/residual/LN/softmax)",
                                      "bf16x3": "PHK_PREC_BF16X3 (tcgen05, split-bf16 operands: fp32-grade products)"}[args.prec]},
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": B * Cc * F * H * Wd * 4,
                "d2h_bytes_per_step": B * tp * hh * ww * 8, "steps": KE,
                "api": "CViViT.encode_host_iter -> phk_encode_pipe_submit/wait (C ABI; pinned host video -> host int64 "
                       "ids every step, the H2D of step i+1 overlaps the encode of step i)",
                "sync_call_value": e2e_sync_value,
                "sync_call_api": "phk_cvivit_encode_host (one blocking call per step: H2D, encode, D2H, sync)"},
        "gpu_launches": int(launches), "host_submit_ms_per_step": t_submit / K * 1e3,
        "roofline": roof,
        "clocks": clocks,
        "sustained": sustained,
    }
    if rank == 0 and world == 1 and not args.no_cpu:
        out["cpu_baseline"] = cpu_encode_baseline(batch=2)
    if not args.no_maskgit:
        try:
            mres = bench_maskgit(dev, prec, world, barrier, sampler if rank == 0 else None)
            if rank == 0 and world == 1 and not args.no_cpu:
                mres["cpu_baseline"] = cpu_maskgit_baseline()
            out["maskgit"] = mres
            out["extra"] = {"maskgit_sample": {k: mres[k] for k in ("metric", "value", "unit", "ms_per_sample",
                                                                   "ms_per_decode_step")}}
        except Exception as ex:  # the headline line must still print
            out["maskgit"] = {"error": repr(ex)}
    # BASELINE configs[3] / configs[4] ("next" rows of SURVEY 8f): every rank takes part (the training step all-reduces).
    # The headline above is complete at this point: a watchdog thread prints it if one of these blocks ever hangs
    # (a rank-asymmetric failure inside a collective), so the extras can never cost the line.
    printed = threading.Event()

    def emit():
        if rank == 0 and not printed.is_set():
            printed.set()
            print(json.dumps(out), flush=True)

    def watchdog(deadline_s=420.0):
        if not printed.wait(deadline_s):
            out.setdefault("extras_watchdog", f"a block after the headline did not finish within {deadline_s:.0f} s")
            emit()
            os._exit(0)

    threading.Thread(target=watchdog, daemon=True).start()
    if prec == L.PREC_BF16:
        for key, fn, skip in (("train_step", bench_train, args.no_train), ("make_video", bench_make_video, args.no_makevideo)):
            if skip:
                continue
            try:
                torch.cuda.empty_cache()
                out[key] = fn(dev, prec, world, barrier, sampler if rank == 0 else None)
            except Exception as ex:
                out[key] = {"error": repr(ex)}
    if rank == 0 and world == 1 and not args.no_refgpu:
        try:
            out["reference_gpu"] = reference_gpu_leg(dev, maskgit=not args.no_maskgit)
            out["reference_gpu"]["encode_speedup_vs_autocast_bf16"] = value / out["reference_gpu"]["encode"]["autocast_bf16"]["value"]
            if "maskgit" in out["reference_gpu"] and "value" in out.get("maskgit", {}):
                out["reference_gpu"]["maskgit_speedup_vs_autocast_bf16"] = (
                    out["maskgit"]["value"] / out["reference_gpu"]["maskgit"]["autocast_bf16"]["value"])
        except Exception as ex:
            out["reference_gpu"] = {"error": repr(ex)}
    if rank == 0:
        sampler.stop()
    emit()
    printed.set()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
