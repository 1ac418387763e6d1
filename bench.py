#!/usr/bin/env python
"""Benchmark of the MagicPose DDIM denoising hot path on B200 (contract: see the task statement).

    python bench.py --gpus 1 --steps 50 --warmup 3            # ours, one frame, full 50-step chain
    torchrun --nproc-per-node N ... bench.py --gpus N ...     # frames sharded over N GPUs
    python bench.py --impl reference --steps K --warmup W     # the reference's path on the host CPUs

A "step" is one p_sample_ddim (ddim.py:518-645) for the per-GPU batch of frames: the pose
ControlNet, the UNet in 'read' mode with the appearance bank, the unconditional UNet, CFG combine
and DDIM update.  The appearance ('write') pass runs once per timestep per SEQUENCE: the timesteps
are dealt over the ranks and exchanged with one all-gather per slot row before / while the steps run
(SURVEY §8e); that work and the exchange are inside the timed region.

What one run reports (rank 0 prints ONE JSON line):
  value / ms_per_step   B = 1 frame per GPU (BASELINE.json configs[1] at N = 1), inputs resident in HBM, the
                        captured step / bank graphs driven directly (pipeline.GraphedDenoiser)
  e2e                   the same chain through the reference-facing API exactly as test_tiktok.py:261-268 calls it:
                        create_model(yaml) -> model.sample_log(cond, ..., x_T) with HOST (pinned) tensors; H2D of
                        the inputs, the bank build for a NEW reference image, a D2H of pred_x0 every step
                        (img_callback) and of the final latent are inside the timed region
  batch8                (N = 1) the same two measurements at eight frames per GPU = configs[2], with its own roofline
  config4               (N > 1) configs[3]: 8 frames per GPU of one sequence, bank sharded over the ranks
  multi_gpu_check       (N > 1) a probe frame every rank computes with the gathered bank: bit-equal across ranks,
                        and within fp16 tolerance of rank 0's chain with a locally built bank
  gpu_eager_baseline    (N = 1) the reference's modules as eager PyTorch (cuDNN/cuBLAS/SDPA, fp16 autocast) on this GPU
  cpu_baseline          (N = 1) the oracle port of the same step on the host cores
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
YAML = os.path.join(REPO, "model_lib", "ControlNet", "models", "cldm_v15_reference_only_pose.yaml")

METRIC = "denoise-steps/sec @512x512 50-step DDIM"
UNIT = "frame-steps/s"
# algorithmic FLOPs (SURVEY §8d / BASELINE.md §2, torch FlopCounterMode on the reference modules)
GF_FRAME_STEP = 2037.9   # pose ControlNet + UNet-read + UNet-uncond, per frame per step
GF_REF_STEP = 803.18     # appearance 'write' pass, per reference per timestep
GF_REF_AS_EXECUTED = 3124.4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1, help="frames per GPU of the headline measurement")
    ap.add_argument("--latent", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-batch8", action="store_true", help="skip the configs[2] sub-record (N = 1)")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the torch-eager GPU baseline (N = 1)")
    ap.add_argument("--no-config4", action="store_true", help="skip the configs[3] sub-record and the probe (N > 1)")
    ap.add_argument("--nvtx", action="store_true", help="wrap the LAST step of the steady-state run in an NVTX range "
                    "'mdb_step' (ncu --nvtx --nvtx-include 'mdb_step/' then profiles exactly one step)")
    ap.add_argument("--tune", default="", help="experiments: launch heuristics as k=v[,k=v] (keys of ops.tuning)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write x_prev and pred_x0 of the last timed step (rank 0's frames of "
                         "the headline run) as DIR/<name>.npy in float32, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 64 * 2 ** 20


def dump_outputs(path, arrays):
    """name -> tensor, written as path/<name>.npy (float32).  Past DUMP_BYTES in all (headers included), each array is
    replaced by the same fixed, seeded sample of its flattened elements, so that dumps of one configuration compare."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    budget = DUMP_BYTES - 256 * len(arrays)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > budget:
            keep = a.size * budget // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
        except Exception:  # noqa: BLE001
            self.proc = None
            return self
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def host_threads():
    """usable host cores: CPU affinity, capped by the cgroup CPU quota when one is set"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p) + 0.5)))
    except Exception:  # noqa: BLE001
        pass
    return n


def cpu_port_step_seconds(sd, latent, steps, warmup, torch):
    """Times the oracle port of p_sample_ddim (oracle/restatement.py) on the host cores: the mean step time and the
    x_prev / pred_x0 of the last step."""
    from oracle import restatement as R  # the ONE place bench.py executes oracle/: the CPU baseline
    from magicdance_b200 import synth
    import numpy as np
    inp = synth.synth_inputs(1, latent, seed=0, shared_reference=True)
    sched = R.ddim_schedule(R.make_schedule()["alphas_cumprod"].astype(np.float32).astype(np.float64))
    x = inp["x"]
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            index = 49 - (i % 50)
            t = torch.full((1,), int(sched["timesteps"][index]), dtype=torch.long)
            t0 = time.perf_counter()
            # as executed by the reference: appearance + pose + UNet-read, then pose (discarded) + UNet-uc
            x_prev, pred_x0, _, _ = R.p_sample_ddim(sd, x, t, index, inp["context"], inp["pose"], inp["ref"], sched,
                                                    scale=7.0)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
            x = x_prev
    return sum(times) / len(times), {"x_prev": x_prev, "pred_x0": pred_x0}


def run_reference(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from magicdance_b200 import synth
    torch.set_grad_enabled(False)
    torch.set_num_threads(host_threads())
    sd = synth.synth_state_dict(seed=0)
    steps = args.steps
    warm = 1 if args.warmup > 0 else 0
    sec, outputs = cpu_port_step_seconds(sd, args.latent, steps, warm, torch)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    val = 1.0 / sec
    sample = (f"{steps} timed p_sample_ddim step(s) of the 50-step chain (+{warm} warm-up), B=1, fp32, latent "
              f"{args.latent}x{args.latent}; per-step time extrapolates linearly to the chain")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "512x512, 50-step DDIM, batch 1, appearance-control + OpenPose ControlNet (CPU)",
                   "latent": args.latent, "frames_per_gpu": 1, "cfg_scale": 7.0},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------
def roofline_probe(torch, ops, trace, peaks, frames_per_gpu=1):
    """Replays every distinct tensor-core GEMM/conv launch of one step standalone, L2 flushed before
    each launch, CUDA-event timed; achieved = sum(2MNK) / sum(avg duration x count)."""
    from collections import Counter
    cnt = Counter(trace)
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device="cuda")
    tot_fl, tot_t, rows = 0.0, 0.0, []
    for (m, n, k, conv, epi, splits, k2), c in cnt.items():
        w = torch.randn(n, k, device="cuda", dtype=torch.float16) * k ** -0.5
        if conv is not None:
            a = torch.randn(conv[0] * conv[1] * conv[2], conv[3], device="cuda", dtype=torch.float16)
            kw = dict(conv=conv[:4], conv_stride=conv[4] if len(conv) > 4 else 1)
        elif k2:
            a = torch.randn(m, k - k2, device="cuda", dtype=torch.float16)
            kw = dict(a2=torch.randn(m, k2, device="cuda", dtype=torch.float16))
        else:
            a = torch.randn(m, k, device="cuda", dtype=torch.float16)
            kw = {}
        reps, ts = 5, []
        for r in range(reps + 1):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ops.gemm(a, w, epilogue=epi, splits=splits, **kw)
            e1.record()
            torch.cuda.synchronize()
            if r:
                ts.append(e0.elapsed_time(e1) * 1e-3)
        t = sum(ts) / len(ts)
        fl = 2.0 * m * n * k
        tot_fl += fl * c
        tot_t += t * c
        rows.append((fl * c, t * c, (m, n, k, conv is not None, splits), c))
    rows.sort(key=lambda r: -r[1])
    peak = peaks.get("bf16_tflops", 1590.0)
    ach = tot_fl / tot_t / 1e12
    top = [{"shape_mnk_conv_splits": list(map(int, r[2][:3])) + [bool(r[2][3]), int(r[2][4])], "count": r[3],
            "ms_total": r[1] * 1e3, "tflops": r[0] / r[1] / 1e12} for r in rows[:6]]
    # DRAM bytes per launch of the family (dram__bytes_read.sum + dram__bytes_write.sum, ncu): a committed
    # capture of the step (profiles/traffic.json, keyed by frames per GPU); no capture -> null
    traffic, traffic_detail = None, None
    try:
        with open(os.path.join(REPO, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        traffic_detail = tj.get(f"gemm_tc_kernel_b{frames_per_gpu}") or (tj.get("gemm_tc_kernel") if frames_per_gpu == 1 else None)
        if traffic_detail is not None:
            traffic = float(traffic_detail["dram_bytes_per_launch_avg"])
    except Exception:  # noqa: BLE001
        traffic, traffic_detail = None, None
    return {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 GEMM + 3x3 implicit-GEMM conv)",
            "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst)" if "bf16_tflops" in peaks else "fallback 1590",
            "traffic": traffic, "traffic_detail": traffic_detail, "gemm_gflop_per_step": tot_fl / 1e9,
            "gemm_ms_per_step_isolated": tot_t * 1e3, "launches_per_step": int(sum(cnt.values())), "top_by_time": top}


class Bench:
    """one process per GPU: the model (reference-facing drop-in), its engine, and the measurements over them"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from magicdance_b200 import synth
        from model_lib.ControlNet.cldm.model import create_model  # the repo's drop-in of the reference's dotted path
        self.torch, self.dist, self.args = torch, dist, args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        torch.set_grad_enabled(False)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        self.peaks = {}
        try:
            with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
                self.peaks = json.load(f)
        except Exception:  # noqa: BLE001
            pass
        dev = f"cuda:{self.local}"
        model = create_model(YAML).to(dev).eval()
        sd = synth.synth_state_dict(seed=0, device=dev)  # random-init weights, generated on the GPU
        missing, unexpected = model.load_state_dict(sd, strict=False)
        assert not unexpected, unexpected
        del sd
        self.model = model
        self.eng = model.engine(dev)  # the DenoiseEngine over the modules' lazily packed fp16 weights
        torch.cuda.empty_cache()
        from magicdance_b200.pipeline import DenoisePipeline
        self.pipe = DenoisePipeline(self.eng, ddim_steps=50, scale=7.0, eta=0.0)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        t = self.torch.tensor([v], device="cuda", dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident chain over the captured graphs --------------------------------------------------------
    def measure(self, B, K, W, seed=None, e2e=True, steady=True, sequence_frames=False):
        """bank build (this rank's share) -> per-slot all-gathers -> K steps of B frames on this GPU.
        Returns the record of this batch size (timings are max over ranks, CUDA events on the launching stream)."""
        torch, ops = self.torch, __import__("magicdance_b200.ops", fromlist=["ops"])
        from magicdance_b200 import parallel, synth
        from magicdance_b200.pipeline import GraphedDenoiser
        world, rank, L, eng, pipe = self.world, self.rank, self.args.latent, self.eng, self.pipe
        inp = synth.synth_inputs(B, L, seed=(100 + rank) if seed is None else seed, shared_reference=True)
        if sequence_frames:  # one sequence: every rank shares the reference / prompt / x_T of rank 0's seed
            shared = synth.synth_inputs(B, L, seed=100, shared_reference=True)
            inp["x"], inp["ref"], inp["context"] = shared["x"], shared["ref"], shared["context"]
        x_T = inp["x"][:1].expand(B, -1, -1, -1).contiguous()  # same x_T for every frame (test_tiktok.py:225)
        pin = lambda t: t.contiguous().pin_memory()
        x_host, pose_host = pin(x_T), pin(inp["pose"])
        ref_host, ctx_host = pin(inp["ref"]), pin(inp["context"])
        ref = ref_host[:1].cuda(non_blocking=True)
        ctx = ctx_host[:1].cuda(non_blocking=True)
        uniq_n = min(K, 50)
        chunk = parallel.bank_chunk_size(uniq_n, world)
        gd = GraphedDenoiser(pipe, B, (L, L), ctx, bank_chunk=chunk)
        gd.ref.copy_(ref)
        gd.capture()
        layout = gd.layout
        slots = (uniq_n + world - 1) // world
        storage = parallel.bank_storage(slots, layout, eng.device, world)  # no cudaMalloc while timing
        build_fn = lambda indices, out: gd.build_bank(indices, ref, out)
        timing = {}

        def run(n_steps, prebuilt=None):
            idxs = [49 - (i % 50) for i in range(n_steps)]
            uniq = list(dict.fromkeys(idxs))
            if prebuilt is None:
                st = storage if (len(uniq) + world - 1) // world == slots else None
                bank = parallel.build_and_gather_bank(uniq, layout, build_fn, eng.device, world, rank, chunk=chunk,
                                                      storage=st, timing=timing)
            else:
                bank = prebuilt
            x = x_host.cuda(non_blocking=True)
            pose = pose_host.cuda(non_blocking=True)
            gd.hint.copy_(pipe.hint(pose, frame_key=None))
            gd.x.copy_(x)
            for j, ix in enumerate(idxs):
                bank.wait(ix)
                mark = self.args.nvtx and prebuilt is not None and j == len(idxs) - 1
                if mark:
                    torch.cuda.synchronize()
                    torch.cuda.nvtx.range_push("mdb_step")
                gd.step(ix, bank[ix])
                if mark:
                    torch.cuda.synchronize()
                    torch.cuda.nvtx.range_pop()
            run.last_bank = bank
            return gd.x_prev

        run(max(W, 1))  # warm-up (untimed)
        self.barrier()
        clocks = ClockSampler(self.local).start()
        l0 = ops.launch_count() + gd.replayed_launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        x_final = run(K)
        e1.record()
        self.barrier()
        launches = ops.launch_count() + gd.replayed_launches - l0
        # what the last timed step hands its caller (the runs below overwrite these buffers)
        self.outputs = {"x_prev": gd.x_prev.clone(), "pred_x0": gd.pred_x0.clone()}
        sec = self.max_over_ranks(e0.elapsed_time(e1)) * 1e-3
        clk = clocks.stop()
        bank_ms = self.max_over_ranks(timing["build0"].elapsed_time(timing["build1"]))
        finite = bool(torch.isfinite(x_final).all())
        fp = [float(x_final.float().abs().mean()), float(x_final.float().flatten()[::997].sum())]
        rec = {"frames_per_gpu": B, "value": world * B * K / sec, "unit": UNIT, "ms_per_step": sec * 1e3 / K, "steps": K,
               "bank_build_ms": bank_ms, "bank_chunk": chunk, "gpu_launches": int(launches), "clocks": clk,
               "finite": finite, "x_final_fingerprint": fp, "step_launches": int(gd.step_launches),
               "bank_launches": int(gd.bank_launches)}
        gflop = GF_FRAME_STEP * B * K * world + GF_REF_STEP * uniq_n
        peak_s = self.peaks.get("bf16_tflops_sustained", 1400.0)
        rec["step_roofline"] = {"algorithmic_gflop": gflop, "achieved_tflops": gflop / sec / 1e3,
                                "peak_tflops_per_gpu": peak_s, "frac": gflop / sec / 1e3 / (world * peak_s)}
        if world > 1:
            # the exchange alone (no build, nothing overlapping it): what it would cost if it were serialised
            self.barrier()
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record()
            gb = parallel.build_and_gather_bank(list(range(49, 49 - uniq_n, -1)), layout, lambda i_, o_: None, eng.device,
                                                world, rank, chunk=chunk, storage=storage)
            gb.wait()
            eb.record()
            self.barrier()
            rec["allgather_ms"] = self.max_over_ranks(ea.elapsed_time(eb))
            rec["allgather_bytes_per_rank"] = int(slots * world * layout.numel * 2)
            rec["allgather_note"] = ("%d all_gather_into_tensor calls (one per slot row, consumption order); in the timed "
                                     "run only the first row is exposed, the rest overlaps the first steps" % slots)
            # (the probe re-gathered the very slots the timed run built: run.last_bank still holds the right data)
        if steady:
            # steady state of a multi-frame video: the bank of this reference is already built and gathered
            self.barrier()
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record()
            run(K, prebuilt=run.last_bank)
            eb.record()
            self.barrier()
            sec_ss = self.max_over_ranks(ea.elapsed_time(eb)) * 1e-3
            rec["steady_state"] = {"value": world * B * K / sec_ss, "unit": UNIT, "ms_per_step": sec_ss * 1e3 / K,
                                   "what": "same K steps with the appearance bank of the reference already built "
                                           "(every frame after the first of a multi-frame video)"}
        self._last = dict(gd=gd, run=run, x_host=x_host, pose_host=pose_host, ref_host=ref_host, ctx_host=ctx_host,
                          ref=ref, ctx=ctx, x_final=x_final.clone())
        if e2e:
            rec["e2e"] = self.measure_e2e(B, K, x_host, pose_host, ref_host, ctx_host)
        return rec

    # ---- the reference-facing call, host buffers ---------------------------------------------------------------
    def measure_e2e(self, B, K, x_host, pose_host, ref_host, ctx_host):
        """model.sample_log as test_tiktok.py:261-268 calls it, from pinned HOST tensors; a NEW reference image in
        the timed call (so the appearance bank is rebuilt inside it), pred_x0 read back every step."""
        torch, model = self.torch, self.model
        L = self.args.latent
        model.image_size = L
        if self.world > 1:
            model.bank_process_group = self.dist.group.WORLD  # one sequence sharded over the ranks (INTEGRATION.md)
        gen = torch.Generator().manual_seed(123)
        uc_ctx = torch.randn(1, 77, 768, generator=gen).expand(B, -1, -1).contiguous().pin_memory()
        ref_b = (ref_host * 0.75).contiguous().pin_memory()  # another reference image: bank rebuilt in the timed call
        p0_host = torch.empty((B, 4, L, L), dtype=torch.float32).pin_memory()
        out_host = torch.empty((B, 4, L, L), dtype=torch.float32).pin_memory()

        def img_callback(pred_x0, i):
            p0_host.copy_(pred_x0, non_blocking=True)
            torch.cuda.synchronize()  # the step's result is on the host before the next step is issued

        def call(ref_h):
            c = {"c_concat": [pose_host], "c_crossattn": [ctx_host], "image_control": [ref_h], "wonoise": True,
                 "overlap_sampling": False}
            uc = {"c_concat": [pose_host], "c_crossattn": [uc_ctx], "wonoise": True, "overlap_sampling": False}
            s, _ = model.sample_log(cond=c, batch_size=B, ddim=True, ddim_steps=K, eta=0.0, unconditional_guidance_scale=7,
                                    unconditional_conditioning=uc, inpaint=None, x_T=x_host, img_callback=img_callback)
            out_host.copy_(s, non_blocking=True)
            torch.cuda.synchronize()
            return s

        call(ref_host)  # untimed: captures the drop-in's graphs, builds the bank of reference A
        self.barrier()
        t0 = time.perf_counter()
        s = call(ref_b)
        self.barrier()
        sec = self.max_over_ranks(time.perf_counter() - t0)
        h2d = sum(t.numel() * t.element_size() for t in (x_host, pose_host, ref_b, ctx_host))
        return {"value": self.world * B * K / sec, "unit": UNIT, "ms_per_step": sec * 1e3 / K,
                "h2d_bytes_per_step": int(h2d / K), "d2h_bytes_per_step": int(p0_host.numel() * 4 + out_host.numel() * 4 / K),
                "api": "model_lib.ControlNet.cldm.model.create_model(yaml) -> model.sample_log(cond, batch_size, ddim=True, "
                       f"ddim_steps={K}, eta=0, unconditional_guidance_scale=7, unconditional_conditioning=uc, x_T=host "
                       "tensor, img_callback=D2H of pred_x0) — test_tiktok.py:261-268; cond tensors on the (pinned) host",
                "includes": "H2D of x_T / pose maps / reference latent / prompt context, appearance-bank build for a new "
                            "reference image, K graph-replayed DDIM steps, D2H of pred_x0 every step and of the sample",
                "timing": "host wall clock between device synchronisations, max over ranks",
                "finite": bool(torch.isfinite(s).all())}

    def roofline(self, B):
        torch, ops = self.torch, __import__("magicdance_b200.ops", fromlist=["ops"])
        st = self._last
        hint_ = self.pipe.hint(st["pose_host"].cuda())
        bank_ = self.pipe.reference_bank(st["ref"], st["ctx"], 49, first_only=True)
        self.pipe.step(st["x_host"].cuda(), 49, st["ctx"], hint_, bank_)  # untraced: fills the per-prompt text K/V cache
        ops.TRACE = []  # the per-step kernel mix: pose ControlNet + paired cond/uncond UNet
        self.pipe.step(st["x_host"].cuda(), 49, st["ctx"], hint_, bank_)
        torch.cuda.synchronize()
        trace, ops.TRACE = ops.TRACE, None
        self.pipe.clear_caches()
        return roofline_probe(torch, ops, trace, self.peaks, frames_per_gpu=B)

    # ---- N > 1: every rank computes a probe frame with the GATHERED bank --------------------------------------
    def multi_gpu_check(self, K):
        """bank slot routing under NCCL: all ranks run rank 0's frame over the gathered bank -> bit-equal across
        ranks; rank 0 reruns it over a bank it builds alone -> equal to fp16 tolerance (the batched appearance
        passes of a 1-GPU and an N-GPU build differ in GEMM split-K, i.e. in summation order only)."""
        torch, dist = self.torch, self.dist
        from magicdance_b200 import parallel
        st = self._last
        gd, run = st["gd"], st["run"]
        # same inputs on every rank (rank 0's), through the bank the timed run gathered
        probe = __import__("magicdance_b200.synth", fromlist=["synth"]).synth_inputs(gd.batch, self.args.latent, seed=100,
                                                                                     shared_reference=True)
        x_T = probe["x"][:1].expand(gd.batch, -1, -1, -1).contiguous().cuda()
        hint = self.pipe.hint(probe["pose"].cuda())
        idxs = [49 - (i % 50) for i in range(K)]

        def chain(bank):
            gd.hint.copy_(hint)
            gd.x.copy_(x_T)
            for ix in idxs:
                bank.wait(ix)
                gd.step(ix, bank[ix])
            return gd.x_prev.clone()

        got = chain(run.last_bank)
        allx = [torch.empty_like(got) for _ in range(self.world)]
        dist.all_gather(allx, got)
        bit_equal = all(bool(torch.equal(allx[0], a)) for a in allx)
        res = {"probe": "rank 0's frame(s), K=%d steps, computed by every rank over the gathered bank" % K,
               "cross_rank_bit_equal": bit_equal}
        if self.rank == 0:
            uniq = list(dict.fromkeys(idxs))
            local = parallel.build_and_gather_bank(uniq, gd.layout, lambda ix, out: gd.build_bank(ix, st["ref"], out),
                                                   self.eng.device, 1, 0, chunk=gd.bank_chunk)
            alone = chain(local)
            res["vs_single_gpu_bank_rel_l2"] = float((got.double() - alone.double()).norm() / alone.double().norm())
            res["ok"] = bool(bit_equal and res["vs_single_gpu_bank_rel_l2"] <= 5e-3)
        return res


def run_ours(args):
    if args.tune:
        from magicdance_b200 import ops
        ops.tuning(**{k: int(v) for k, v in (kv.split("=") for kv in args.tune.split(","))}).__enter__()
    b = Bench(args)
    torch, dist = b.torch, b.dist
    world, rank = b.world, b.rank
    K, W, B = args.steps, args.warmup, args.batch
    # N > 1: the ranks hold frames of ONE sequence (shared reference image / prompt / x_T, own pose maps)
    main = b.measure(B, K, W, e2e=not args.no_e2e, sequence_frames=world > 1)
    outputs = b.outputs
    roof = None
    if rank == 0 and not args.no_roofline:
        roof = b.roofline(B)
    check = cfg4 = None
    if world > 1 and not args.no_config4:
        check = b.multi_gpu_check(K)
        if B != 8:
            b._last = None
            torch.cuda.empty_cache()
            # BASELINE configs[3]: one sequence, 8 frames per GPU (64 over 8 GPUs), bank sharded + gathered in the timer
            cfg4 = b.measure(8, K, W, e2e=not args.no_e2e, sequence_frames=True)
    batch8 = None
    if world == 1 and B != 8 and not args.no_batch8:
        b._last = None
        torch.cuda.empty_cache()
        batch8 = b.measure(8, K, W, e2e=not args.no_e2e)
        if not args.no_roofline:
            batch8["roofline"] = b.roofline(8)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)

    line = {
        "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(W, 1),
        "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": "512x512, 50-step DDIM, batch %d/GPU, appearance-control + OpenPose ControlNet, "
                               "CFG 7 (BASELINE.json configs[%d])" % (B, 1 if B == 1 else 2),
                   "latent": args.latent, "frames_per_gpu": B, "cfg_scale": 7.0, "ddim_steps": 50,
                   "bank": "appearance pass once per timestep per sequence (timesteps batched %d at a time, sharded "
                           "over ranks + one all-gather per slot row, overlapped with the first steps), inside the "
                           "timed region" % main["bank_chunk"],
                   "l2": "no flush needed: each step streams >4 GB of fp16 weights (L2 is 126 MB)",
                   "weights": "random init (seeded), fp16 storage, fp32 accumulate",
                   "cuda_graph": True, **({"tune": args.tune} if args.tune else {})},
        "gpu_launches": main["gpu_launches"], "clocks": main["clocks"], "finite": main["finite"],
        "x_final_fingerprint": main["x_final_fingerprint"], "step_roofline": main["step_roofline"],
        "launches_per_step": main["step_launches"], "bank_build_ms": main["bank_build_ms"],
    }
    for k in ("steady_state", "e2e", "allgather_ms", "allgather_bytes_per_rank", "allgather_note"):
        if k in main:
            line[k] = main[k]
    if roof is not None:
        line["roofline"] = roof
    if batch8 is not None:
        batch8["config"] = "512x512, 50-step DDIM, batch 8, fp16, 1xB200 (BASELINE.json configs[2])"
        line["batch8"] = batch8
    if cfg4 is not None:
        cfg4["config"] = ("%d-frame pose sequence, shared reference image, 8 frames per GPU over %d GPUs, bank sharded "
                          "+ gathered inside the timed region (BASELINE.json configs[3])" % (8 * world, world))
        ss = cfg4.get("steady_state", {}).get("value")
        if ss:
            cfg4["fraction_of_steady_state"] = cfg4["value"] / ss
        line["config4"] = cfg4
    if check is not None:
        line["multi_gpu_check"] = check
    if world == 1 and not args.no_gpu_baseline:
        line["gpu_eager_baseline"] = gpu_eager_baseline(args)
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(host_threads())
        sd = {k: v.detach().float().cpu() for k, v in b.model.state_dict().items()
              if k.startswith(("model.diffusion_model.", "appearance_control_model.", "pose_control_model."))}
        csec, _ = cpu_port_step_seconds(sd, args.latent, 1, 0, torch)
        line["cpu_baseline"] = {"value": 1.0 / csec, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                "sample": "1 p_sample_ddim step (index 49) of the same chain, B=1, fp32, as executed "
                                          "by the reference (incl. its discarded 2nd pose pass), no warm-up"}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    if check is not None and not check.get("ok", False):
        raise SystemExit("multi-GPU probe frame differs between ranks or from the single-GPU bank: %r" % (check,))


def gpu_eager_baseline(args):
    """BASELINE.md §3's secondary baseline, same box, same run: tests/torch_gpu_baseline.py in its own process (it
    executes the oracle restatement as eager PyTorch on the GPU, which only tests/ may do)."""
    cmd = [sys.executable, os.path.join(REPO, "tests", "torch_gpu_baseline.py"), "--batch", "1,8", "--steps", "5",
           "--warmup", "2", "--algorithmic", "--latent", str(args.latent)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=REPO)
        lines = [ln for ln in out.stdout.strip().splitlines() if ln.startswith("{")]
        if not lines:
            return {"unavailable": f"rc {out.returncode}: " + out.stderr.strip()[-600:]}
        res = json.loads(lines[-1])
        res["cmd"] = " ".join(cmd[1:])
        return res
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}


_RESULT_FD = None


def claim_stdout():
    """stdout carries exactly ONE line, the JSON result: point fd 1 at stderr for the duration of the run
    (NCCL prints its version banner to stdout from C, libraries may print warnings) and keep the real stdout
    aside for emit()."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    payload = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(payload.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_RESULT_FD, payload)


def main():
    args = parse()
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
