#!/usr/bin/env python
"""bench.py — StyleSinger ph -> mel -> wav hot path on B200 (driver contract; see the task statement).

    python bench.py --gpus 1 --steps K --warmup W [--workload utt10s|batch64] [--T 100]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # CPU arm: the UNMODIFIED reference where tools/ref_import.py finds its
                                              # sources, else the oracle port; host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's outputs as DIR/<name>.npy
    python bench.py --workload sweep          # BASELINE.json configs[4]: T sweep, persistent vs per-launch mel sampler

A "step" is one pass of the whole hot path (encoder, style adaptor + RVQ, two F0/UV diffusions, FFT
decoder, T-step mel diffusion, HiFi-GAN-NSF) over one batch of seeded synthetic utterances
(SURVEY.md §8d) with synthetic (seed 0) checkpoints.  `value` = mel frames of all ranks / step time with
the inputs resident in HBM; `e2e` = the same pass through StyleSingerInfer.infer_packed with pinned HOST
inputs (H2D inside the timed region) and the waveform copied back to the host (D2H inside).
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = "mel_frames_per_sec_ph2wav_T100"
UNIT = "frames/s"

# ALGORITHMIC FLOPs per frame-step of the mel denoiser (SURVEY.md section 8d: 26.43 MFLOP as the reference executes it).
# This implementation hoists the step-invariant conditioner projection out of the T loop (20 x 2 x 256 x 512 = 5.24 MFLOP per
# frame ONCE per sampler call instead of per step): MEL_STEP_FLOPS_EXECUTED is what the tensor cores actually do per step.
MEL_STEP_FLOPS = 2 * 80 * 256 + 20 * (2 * 768 * 512 + 2 * 256 * 512 + 2 * 256 * 512) + 2 * 256 * 256 + 2 * 256 * 80  # 26.43 MFLOP
MEL_STEP_FLOPS_EXECUTED = MEL_STEP_FLOPS - 20 * 2 * 256 * 512                                                       # 21.18 MFLOP
MEL_HOIST_FLOPS = 20 * 2 * 256 * 512  # executed once per frame and sampler call
# HBM bytes one frame streams per reverse step in this layout (DESIGN.md section 3), per residual layer: y planes in (1024)
# + hoisted conditioner addend, fp32 (2048) + gate output planes out / in (2 x 1024) + y planes read-modify-write (2 x 1024)
# + skip read-modify-write (2048) = 9216; heads ~4 KB
MEL_STEP_STREAM_BYTES = 20 * 9216 + 4096


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "src": "fallback"}


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_workload(name, rank, world, describe_only=False):
    from stylesinger_b200 import synth
    from stylesinger_b200.sharding import lpt_assign  # plain Python: the reference arm must not load the CUDA library
    if name == "utt10s":
        desc = "single 10 s utterance per GPU (BASELINE.json configs[1])"
        return desc if describe_only else ([synth.make_utterance(10.0, utt_idx=rank)], desc)
    n_per = {"batch64": 64, "batch8": 8}[name]
    if describe_only:
        return f"{n_per} variable-length (2-15 s) utterances per GPU, LPT-sharded (BASELINE.json configs[2]/[3])"
    secs = synth.batch_seconds(n_per * world, seed=1234)
    mine = lpt_assign(secs, world)[rank]
    utts = [synth.make_utterance(float(secs[i]), utt_idx=i) for i in mine]
    return utts, f"{n_per} variable-length (2-15 s) utterances per GPU, LPT-sharded (BASELINE.json configs[2]/[3])"


# ---------------------------------------------------------------------------------------------------
class CpuArm:
    """The reference's own implementation of the path on the host cores.  kind "reference": the unmodified reference
    (baseline/ref_harness.py drives its StyleSingerInfer, model and vocoder built by the reference's own loaders from
    checkpoint directories in its on-disk format); kind "port": the oracle restatement, used only when tools/ref_import.py
    finds no copy of the reference.  Neither touches libstylesinger_b200.so."""

    def __init__(self, T, threads):
        self.T, self.threads = T, threads
        torch.set_num_threads(threads)
        sys.path.insert(0, os.path.join(REPO, "baseline"))
        self.runner = None
        try:
            import ref_harness
            if ref_harness.available():
                cwd = os.getcwd()
                with contextlib.redirect_stdout(sys.stderr):  # the reference prints while loading: keep stdout to the JSON line
                    self.runner = ref_harness.ReferenceRunner(T=T, device="cpu", threads=threads)
                os.chdir(cwd)
        except Exception as e:  # reference copy broken: say so and fall back to the port
            print(f"[bench] reference harness unavailable ({type(e).__name__}: {e}); using the oracle port", file=sys.stderr)
            self.runner = None
        self.kind = "reference" if self.runner is not None else "port"

    def describe(self):
        return ("unmodified reference (inference/StyleSinger.py:41-64 with explicit mel2ph; StyleSinger + HifiGAN_NSF from its "
                "own loaders)" if self.kind == "reference" else "CPU oracle port of the reference (no reference copy found)")

    def one_pass(self, seconds, utt_idx=0):
        if self.runner is not None:
            with contextlib.redirect_stdout(sys.stderr):
                return self.runner.timed_pass(seconds, utt_idx=utt_idx)
        return self._port_pass(seconds, utt_idx)

    def _port_pass(self, seconds, utt_idx):
        from oracle import stylesinger_oracle as O
        from stylesinger_b200 import synth
        from stylesinger_b200.hparams import DEFAULT_VOCODER_CONFIG, resolve
        hp = resolve(timesteps=self.T, K_step=self.T, f0_timesteps=self.T)
        if not hasattr(self, "sd"):
            self.sd = synth.acoustic_state_dict(hp, seed=0)
            self.vsd = synth.vocoder_state_dict(DEFAULT_VOCODER_CONFIG, seed=0)
        u = synth.make_utterance(seconds, utt_idx=utt_idx)
        ns = O.NoiseSource(0)
        t0 = time.perf_counter()
        with torch.no_grad():
            r = O.stylesinger_forward(self.sd, hp, u["txt_tokens"][None], u["note"][None], u["note_dur"][None],
                                      u["note_type"][None], u["spk_embed"][None], u["emo_embed"][None], u["ref_mels"][None],
                                      u["ref_f0"], ns, mel2ph=u["mel2ph"][None])
            mel, f0 = O.postprocess_mel(r["mel_out"][0].numpy(), r["f0_denorm"][0].numpy(), hp)
            O.spec2wav(mel, f0, self.vsd, DEFAULT_VOCODER_CONFIG, ns)
        return int(u["mel2ph"].shape[0]), time.perf_counter() - t0

    def close(self):
        if self.runner is not None:
            self.runner.close()


def cpu_threads():
    """Threads for the CPU arm.  The reference's PyTorch CPU path gets SLOWER beyond ~16 threads on the GPU
    box's 128 logical cores (probe, 94 frames x 20 steps: 8 thr 0.74 s, 16 thr 0.70 s, 32 thr 1.50 s, 64 thr 3.59 s;
    128 thr did not finish in 15 min), so "all the threads it can use" is capped where it is fastest;
    tools/baseline_arms.py records the os.cpu_count() and 1-thread figures BASELINE.md section 3 asks for."""
    return max(1, min(os.cpu_count() or 1, 16))


def cpu_sample_seconds(args):
    """Utterance length of one CPU-arm step.  BASELINE.json configs[1] (10 s) whenever the whole --steps run then stays
    within a few minutes (~18 s per pass), else configs[0]'s length (4 s); --cpu-sample-seconds overrides."""
    if args.cpu_sample_seconds > 0:
        return args.cpu_sample_seconds
    return 10.0 if args.steps <= 8 else 4.0


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = cpu_threads()
    sample_s = cpu_sample_seconds(args)
    arm = CpuArm(args.T, threads)
    arm.one_pass(0.5)  # warm-up (thread pools, allocator, lazy inits); further --warmup passes would only burn CPU minutes
    times, frames = [], 0
    for i in range(args.steps):
        frames, dt = arm.one_pass(sample_s, utt_idx=0)
        times.append(dt)
    arm.close()
    ms = 1000.0 * float(np.mean(times))
    val = frames / (ms / 1000.0)
    line = {"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "ms_per_step_median": 1000.0 * float(np.median(times)), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            # same workload naming as the b200 arm; each step is a bounded sample of it (the metric is per frame)
            "config": {"workload": f"{args.workload}: {make_workload(args.workload, 0, 1, describe_only=True)}; T={args.T} mel + "
                                   f"2x{args.T} F0 steps; full ph->mel->wav",
                       "sample": f"one {sample_s:g} s utterance of that workload per step (B=1, as the reference's own inference "
                                 f"path runs: tasks/StyleSinger/stylesinger.py:168 asserts B=1); {arm.describe()}",
                       "parallelism": f"{threads} host threads (torch intra-op) of {os.cpu_count()} logical cores"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "host_logical_cores": os.cpu_count(), "kind": arm.kind,
                             "sample": f"{sample_s:g} s utterance ({frames} frames), full ph->wav, T={args.T}, mean of {args.steps} passes"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


DUMP_BYTES = 60 << 20  # with the .npy headers, under 64 MB


def dump_outputs(outdir, arrays, budget=None):
    """Write each array as <outdir>/<name>.npy (float64 for integer arrays, float32 otherwise).  When together they exceed
    `budget` bytes (default DUMP_BYTES), every array with more than 4096 rows keeps the same fraction of its rows, chosen by
    np.random.default_rng(0) and sorted (so equal row counts give equal rows), and those row indices go to
    <name>_rows.npy."""
    budget = DUMP_BYTES if budget is None else budget
    os.makedirs(outdir, exist_ok=True)
    host = {}
    for k, a in arrays.items():
        a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
        host[k] = a.astype(np.float64 if a.dtype.kind in "iub" else np.float32)
    big = [k for k, a in host.items() if a.shape[0] > 4096]
    small_bytes = sum(a.nbytes for k, a in host.items() if k not in big)
    big_bytes = sum(host[k].nbytes + 8 * host[k].shape[0] for k in big)  # values + float64 row index
    keep = min(1.0, (budget - small_bytes) / max(big_bytes, 1))
    for k, a in host.items():
        if k in big and keep < 1.0:
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], int(a.shape[0] * keep), replace=False))
            np.save(os.path.join(outdir, k + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(outdir, k + ".npy"), a)


# ---------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist
    from stylesinger_b200 import synth
    from stylesinger_b200._lib import lib
    from stylesinger_b200.engine import pack_batch
    from stylesinger_b200.hparams import DEFAULT_VOCODER_CONFIG, resolve
    from stylesinger_b200.infer import StyleSingerInfer

    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    T = args.T
    hp = resolve(timesteps=T, K_step=T, f0_timesteps=T)
    eng = StyleSingerInfer(hp, dev, synth.acoustic_state_dict(hp, seed=0),
                           synth.vocoder_state_dict(DEFAULT_VOCODER_CONFIG, seed=0), DEFAULT_VOCODER_CONFIG)
    utts, wl_desc = make_workload(args.workload, rank, world)
    pb_host = pack_batch(utts, use_mel2ph=True, pin=True)
    pb_dev = pb_host.to(dev)
    frames = pb_host.total_frames
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for s in range(steps):
            flush.zero_()  # flush L2 between timed iterations (outside the event pair)
            evs[s][0].record()
            fn(s)
            evs[s][1].record()
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs) / steps
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up
    for s in range(args.warmup):
        eng.run_device(pb_dev, seed=s)
    torch.cuda.synchronize(dev)

    # ---- value: device-resident inputs
    last = {}

    def value_step(s):
        out = eng.run_device(pb_dev, seed=100 + s)
        if s == args.steps - 1:
            last["out"] = out

    clocks = ClockSampler(local_rank)
    clocks.start()
    l0 = lib.ssb_launch_count()
    ms = timed(value_step, args.steps)
    launches = int(lib.ssb_launch_count() - l0)
    clk = clocks.stop()
    if args.dump_outputs:
        mel, f0, wav, fo_v = last["out"]
        hop = eng.vocoder.hop
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"),
                     {"mel_out": mel, "f0_denorm": f0, "wav": wav.reshape(-1, hop), "wav_frame_offsets": fo_v},
                     budget=DUMP_BYTES // world)  # every rank writes its own shard
    del last

    # ---- e2e: host buffers in, host waveform out
    wav_bytes = frames * 256 * 4
    ms_e2e = timed(lambda s: eng.infer_packed(pb_host, seed=200 + s), args.steps)

    # ---- e2e including the only collective the design has (SURVEY 8e / BASELINE.json configs[3] "NCCL scatter/gather"):
    # rank 0 owns the whole 64*N-utterance request on the host; every timed step scatters the ragged inputs over NCCL
    # (GPU -> GPU, NVLink), runs the shard, and gathers the waveforms back to rank 0's pinned host memory.
    sg = None
    if world > 1 and not args.no_collective:
        from stylesinger_b200.dist import gather_waveforms_device, scatter_utterances
        all_utts = None
        n_total = 0
        if rank == 0:
            secs = synth.batch_seconds(len(utts) * world, seed=1234) if args.workload != "utt10s" else [10.0] * world
            all_utts = [synth.make_utterance(float(secs[i]), utt_idx=i) for i in range(len(secs))]
            n_total = len(all_utts)
        nt = torch.tensor([n_total], dtype=torch.int64, device=dev)
        dist.broadcast(nt, src=0)
        n_total = int(nt.item())

        def sg_step(s):
            pb, idx = scatter_utterances(all_utts, src=0, device=dev, keep_on_device=True)
            if pb.B > 0:
                _, _, wav, fo_v = eng.run_device(pb, seed=400 + s)
            else:
                wav, fo_v = torch.zeros(0, device=dev), np.zeros(1, np.int32)
            return gather_waveforms_device(wav, fo_v, eng.vocoder.hop, idx, n_total, dst=0)

        sg_step(0)
        ms_sg = timed(sg_step, args.steps)
        sg = {"ms_per_step": ms_sg, "steps": args.steps}

    # ---- latency regime: BASELINE.json configs[1] (one 10 s utterance) through the same public API
    lat = None
    if args.workload != "utt10s" and not args.no_latency:
        u10, _ = make_workload("utt10s", rank, world)
        pb10 = pack_batch(u10, use_mel2ph=True, pin=True)
        for s_ in range(2):
            eng.infer_packed(pb10, seed=s_)
        ms10 = timed(lambda s: eng.infer_packed(pb10, seed=300 + s), args.steps)
        f10 = pb10.total_frames
        lat = {"workload": "utt10s: one 10 s utterance (BASELINE.json configs[1]), host buffers in/out", "frames": f10,
               "ms": ms10, "frames_per_s": f10 / (ms10 / 1000.0), "rtf": (ms10 / 1000.0) / (f10 * 256 / 48000.0)}

    # ---- roofline of the dominant kernel (mel denoiser GEMMs), timed live on the stream
    out = eng.model.forward(pb_dev, seed=1, skip_mel_diffusion=True, want=("coarse_mel", "diff_cond"))
    cond, coarse = out["diff_cond"], out["coarse_mel"]
    eng.model.mel_diffusion(cond, coarse, pb_dev.frame_offsets, seed=2)
    l1 = lib.ssb_launch_count()
    ms_mel = timed(lambda s: eng.model.mel_diffusion(cond, coarse, pb_dev.frame_offsets, seed=3 + s), args.steps)
    n_mel = int(lib.ssb_launch_count() - l1) // args.steps
    pk = peaks()
    traffic = None  # dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    tpath = os.path.join(REPO, "profiles", "traffic.json")  # ncu --set full capture of this workload (profiles/*.md)
    if os.path.exists(tpath) and args.workload == "batch64" and T == 100:
        try:
            traffic = json.load(open(tpath))
        except Exception:
            traffic = None
    flops = frames * T * MEL_STEP_FLOPS  # algorithmic (reference) FLOPs; executed: see executed_tflops below
    achieved = flops / (ms_mel / 1000.0) / 1e12
    executed = frames * (T * MEL_STEP_FLOPS_EXECUTED + MEL_HOIST_FLOPS) / (ms_mel / 1000.0) / 1e12
    gemm_launches = T * (2 * hp["residual_layers"] + 3) + 1
    roof = {"bound": "tensor", "achieved": achieved, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
            "frac": achieved / pk["bf16_tflops"], "traffic": (traffic or {}).get("bytes_per_launch"),
            "traffic_detail": traffic, "peak_source": pk["src"] + " (cuBLAS bf16, sustained)",
            "kernel": "conv_gemm_tc2r_kernel<128, GATE> (tcgen05 cta_group::2, tap reuse; 90.6 %% tensor pipe active under ncu) + "
                      "conv_gemm_tc2_kernel<128, RES_SKIP>; mel denoiser stage: %d launches per sampler call, of which %d residual-layer GEMMs"
                      % (n_mel, 2 * T * hp["residual_layers"]),
            "avg_launch_us": 1000.0 * ms_mel / max(n_mel, 1), "stage_ms": ms_mel,
            "note": "useful FLOPs (26.43 MFLOP per frame-step, SURVEY 8d) over the CUDA-event time of the mel-diffusion stage; "
                    "the step-invariant conditioner projection is hoisted out of the T loop (executed_tflops counts what the tensor "
                    "cores really do: 21.18 MFLOP per frame-step + 5.24 MFLOP per frame once); the GEMMs run as 3 tcgen05 fp16 MMAs "
                    "per product (hi/lo split) for fp32-class accuracy, so the issued-MMA rate is 3x executed_tflops and the "
                    "effective ceiling of this precision scheme is peak/3",
            "executed_tflops": executed, "issued_mma_tflops": 3.0 * executed,
            # the same stage against the HBM roofline under the per-layer-streamed byte model of THIS layout
            # (DESIGN.md section 3: fp32 residual stream + fp16 hi/lo operand planes, nothing stays in L2 at this size)
            "hbm_streamed": {"bytes_per_frame_step": MEL_STEP_STREAM_BYTES,
                             "achieved_gbs": frames * T * MEL_STEP_STREAM_BYTES / (ms_mel / 1000.0) / 1e9,
                             "peak_gbs": pk["hbm_gbs"]}}

    tot = torch.tensor([float(frames)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    total_frames = float(tot.item())

    if rank == 0:
        cpu, gpu_ref = None, None
        if world == 1 and not args.no_cpu_baseline:
            threads = cpu_threads()
            cwd = os.getcwd()
            sample_s = args.cpu_sample_seconds if args.cpu_sample_seconds > 0 else 10.0  # BASELINE.json configs[1]
            arm = CpuArm(T, threads)
            arm.one_pass(0.5)
            f, dt = arm.one_pass(sample_s)
            arm.close()
            cpu = {"value": f / dt, "unit": UNIT, "cores": threads, "host_logical_cores": os.cpu_count(), "kind": arm.kind,
                   "sample": f"{sample_s:g} s utterance ({f} frames, B=1), full ph->wav, T={T}, 1 pass ({dt:.1f} s); {arm.describe()}"}
            # ---- the denominator of north_star's >= 10x target: the reference's own PyTorch path on this GPU (eager, default
            # backend flags = cuDNN TF32 convs on), B=1 as its inference driver runs, same 10 s utterance as latency_utt10s
            if arm.kind == "reference" and not args.no_torch_gpu_baseline:
                try:
                    import ref_harness
                    with contextlib.redirect_stdout(sys.stderr):
                        g = ref_harness.ReferenceRunner(T=T, device="cuda")
                        g.timed_pass(1.0)
                        passes = [g.timed_pass(10.0) for _ in range(3)]
                        g.close()
                    fg = passes[0][0]
                    tg = float(np.median([p_[1] for p_ in passes]))
                    gpu_ref = {"value": fg / tg, "unit": UNIT, "ms": 1000.0 * tg, "kind": "reference",
                               "sample": f"10 s utterance ({fg} frames, B=1), full ph->wav, T={T}, median of 3 passes, eager PyTorch "
                                         f"{torch.__version__} on cuda:0, default flags (cudnn.allow_tf32={torch.backends.cudnn.allow_tf32}, "
                                         f"matmul.allow_tf32={torch.backends.cuda.matmul.allow_tf32})"}
                except Exception as e:
                    gpu_ref = {"unavailable": f"{type(e).__name__}: {e}"}
            os.chdir(cwd)
        val = total_frames / (ms / 1000.0)
        audio_s = total_frames * 256 / 48000.0
        line = {"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "impl": "b200",
                "config": {"workload": f"{args.workload}: {wl_desc}; T={T} mel + 2x{T} F0 steps; full ph->mel->wav",
                           "frames_per_step": total_frames, "utterances_per_gpu": len(utts), "parallelism": f"dp{world} (utterance sharding; no collective inside the computation, scatter/gather timed in e2e_scatter_gather)",
                           "l2": "256 MiB flush between timed iterations", "rtf": (ms / 1000.0) / audio_s},
                "clocks": clk,
                "e2e": {"value": total_frames / (ms_e2e / 1000.0), "unit": UNIT, "h2d_bytes_per_step": pb_host.h2d_bytes(),
                        "d2h_bytes_per_step": int(wav_bytes), "ms_per_step": ms_e2e},
                "gpu_launches": launches, "roofline": roof}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if lat is not None:
            line["latency_utt10s"] = lat
        if sg is not None:
            line["e2e_scatter_gather"] = {"value": total_frames / (sg["ms_per_step"] / 1000.0), "unit": UNIT, **sg,
                                          "what": "rank 0 owns the request on the host: NCCL scatter of the ragged inputs + compute + "
                                                  "NCCL gather of the waveforms to rank 0's pinned memory, all inside the timed region"}
        if gpu_ref is not None:
            line["torch_gpu_baseline"] = gpu_ref
            if "value" in gpu_ref and lat is not None:
                line["target_10x"] = {"utt10s_b200_e2e_over_reference_gpu": lat["frames_per_s"] / gpu_ref["value"],
                                      "batch_b200_e2e_over_reference_gpu_b1": line["e2e"]["value"] / gpu_ref["value"],
                                      "note": "reference = its own B=1 inference path on the same GPU; see profiles/ for the "
                                              "padded-batch and allow_tf32=False variants (tools/baseline_arms.py)"}
        print(json.dumps(line), flush=True)


def run_sweep(args, rank, world, local_rank):
    """BASELINE.json configs[4]: T in {25, 50, 100, 200, 500} at batch 64 on one B200, mel sampler only (the F0 loops stay at
    100 steps and are not part of the timed stage): one launch per GEMM vs the persistent single-launch kernel run over
    groups of <= 48 row tiles (ssb_model_set_persistent_groups)."""
    from stylesinger_b200 import synth
    from stylesinger_b200._lib import lib
    from stylesinger_b200.engine import pack_batch
    from stylesinger_b200.hparams import DEFAULT_VOCODER_CONFIG, resolve
    from stylesinger_b200.infer import StyleSingerInfer
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    hp = resolve(timesteps=100, K_step=100, f0_timesteps=100)
    eng = StyleSingerInfer(hp, dev, synth.acoustic_state_dict(hp, seed=0),
                           synth.vocoder_state_dict(DEFAULT_VOCODER_CONFIG, seed=0), DEFAULT_VOCODER_CONFIG)
    utts, wl_desc = make_workload("batch64", rank, world)
    pb_dev = pack_batch(utts, use_mel2ph=True, pin=True).to(dev)
    frames = pb_dev.total_frames
    out = eng.model.forward(pb_dev, seed=1, skip_mel_diffusion=True, want=("coarse_mel", "diff_cond"))
    cond, coarse = out["diff_cond"], out["coarse_mel"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    pk = peaks()

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        torch.cuda.synchronize(dev)
        for s_ in range(steps):
            flush.zero_()
            evs[s_][0].record()
            fn(s_)
            evs[s_][1].record()
        torch.cuda.synchronize(dev)
        return sum(a.elapsed_time(b) for a, b in evs) / steps

    clocks = ClockSampler(local_rank)
    clocks.start()
    rows = []
    for T in [int(t) for t in args.sweep_T.split(",")]:
        eng.model.set_timesteps(T, None)
        row = {"T": T}
        for arm, grp in (("per_launch", False), ("persistent_groups", True)):
            eng.model.set_persistent_groups(grp)
            eng.model.mel_diffusion(cond, coarse, pb_dev.frame_offsets, seed=2)  # warm-up
            l0 = lib.ssb_launch_count()
            ms = timed(lambda s_: eng.model.mel_diffusion(cond, coarse, pb_dev.frame_offsets, seed=3 + s_), args.steps)
            tf = frames * T * MEL_STEP_FLOPS / (ms / 1000.0) / 1e12
            row[arm] = {"ms": ms, "launches": int(lib.ssb_launch_count() - l0) // args.steps, "frames_per_s": frames / (ms / 1000.0),
                        "useful_tflops": tf, "frac_of_bf16_peak": tf / pk["bf16_tflops"],
                        "hbm_streamed_gbs": frames * T * MEL_STEP_STREAM_BYTES / (ms / 1000.0) / 1e9}
        rows.append(row)
    eng.model.set_persistent_groups(False)
    clk = clocks.stop()
    r100 = next((r for r in rows if r["T"] == 100), rows[0])
    line = {"metric": "mel_frames_per_sec_mel_diffusion_stage", "value": r100["per_launch"]["frames_per_s"], "unit": UNIT, "n_gpus": 1,
            "steps": args.steps, "warmup": 1, "ms_per_step": r100["per_launch"]["ms"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "b200",
            "config": {"workload": f"sweep (BASELINE.json configs[4]): {wl_desc}; mel diffusion stage only, T in {args.sweep_T}",
                       "frames_per_step": frames, "l2": "256 MiB flush between timed iterations"},
            "clocks": clk, "peak_tflops": pk["bf16_tflops"], "peak_hbm_gbs": pk["hbm_gbs"], "sweep": rows}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="batch64", choices=["utt10s", "batch64", "batch8", "sweep"])
    ap.add_argument("--T", type=int, default=100)
    ap.add_argument("--cpu-sample-seconds", type=float, default=0.0, help="0: 10 s (configs[1]) when it fits a few minutes, else 4 s")
    ap.add_argument("--no-torch-gpu-baseline", action="store_true")
    ap.add_argument("--no-collective", action="store_true", help="N>1: skip the scatter/gather e2e measurement")
    ap.add_argument("--sweep-T", default="25,50,100,200,500")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's mel_out, f0_denorm, wav (rows of one hop) and "
                         "wav_frame_offsets as DIR/<name>.npy (DIR/rank<r>/ per rank when N>1; at most 64 MB over all "
                         "ranks, a fixed seeded row sample when larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "sweep"):
        ap.error("--dump-outputs writes the outputs of the b200 ph -> wav pass; --impl reference and --workload sweep "
                 "do not run it")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        os.environ["CUDA_VISIBLE_DEVICES"] = ""  # CPU arm: nothing of it may touch the GPU (set before any CUDA init)
        if args.workload == "sweep":
            args.workload = "batch64"
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    try:
        if args.workload == "sweep":
            run_sweep(args, rank, world, local_rank)
        else:
            run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
