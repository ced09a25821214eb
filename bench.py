#!/usr/bin/env python
"""bench.py — propagated frames/sec of the mask-propagation hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--config cfg2|cfg3|cfg4|cfg5]     (ours; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W [--config ...]    (reference algorithm, host cores)

Workloads (BASELINE.json configs[1..4], SURVEY.md §8d; synthetic DAVIS-shaped clips, seeded random
weights in the reference's checkpoint format, mem_freq 5):
  cfg2 (default, the configuration the metric is quoted on)  480x854 (-> 480x864), 1 object, top-k 20,
        101-frame clip, interaction on frame 0: bank grows 1 -> 21 frames
  cfg3  480x854, 3 objects, top-k 50, 251-frame clip (bank 1 -> 51)
  cfg4  480x854, 2 objects, top-k 50, 61-frame clip, interactions on frames 0 then 60: 59 frames through
        fuse_one_frame / FusionNet (inference_core.py:190-217)
  cfg5  720x1280, 5 objects, top-k 50, 501-frame clip (bank 1 -> 101; 4.6 GB of bank per clip)
ONE STEP = the interaction(s) of the configuration on every clip a GPU holds: `--clips-per-gpu` concurrent
lanes (own network object, CUDA stream, Python thread) x `--lockstep` clips per lane advanced as one
batch (mivos_b200.LockstepSession).  The JSON line carries, measured in the same run:
  value / e2e                    the headline configuration (fp16 operands; cfg2: 3 lanes x 4 lock-step clips; measured
                                 on B200, profiles/r02c9_bench_c*_l4.json: 3 x 4 1060 frames/s, 2 x 4 1038)
                                 value: clips resident in HBM; e2e: clips in PINNED HOST memory, every frame
                                 copied H2D inside the timed region, u8 masks copied D2H at the end
  single_session                 the same metric through ONE InferenceCore.interact (1 lane x 1 clip): what
                                 the unchanged reference callers get (eval_interactive_davis.py:76-83)
  tf32                           the headline configuration with fp32 storage / TF32 MMAs (the path that is
                                 fp32-comparable with the reference's DAVIS evaluation), with its own roofline
  reference_cuda_eager           the reference's PyTorch ops (oracle port, torch eager -> cuDNN / cuBLAS) on
                                 the SAME GPU and clip: the library kernels this repository replaces
  cpu_baseline                   the reference's PyTorch ops on the host cores, bounded sample (below)
  roofline / roofline_memory_read   event-bracketed launches of the dominant kernel family (conv implicit
                                 GEMM) and of the memory read, on the unit of the timed workload
Reference arm / cpu_baseline sample: `interact()` over the first `--ref-frames` frames of the same clip
with the memory bank PRE-FILLED to the mean bank size a frame of the full clip sees (cfg2: 11.3 frames;
the per-frame cost of the reference is linear in the bank size, so the sample's frames cost what the
average frame of the full clip costs) — same shapes, same top-k, same per-frame work as `config`.
`--dump-outputs DIR` writes what the timed steps hand to their caller (the u8 masks interact() returns), from
the last headline step, as float32 .npy files (dump_outputs); inputs and weights are seeded, so the same
arguments give the same inputs and two builds can be compared output for output.
Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
Every step reads a whole clip (503 MB at cfg2) plus >200 MB of weights: inputs exceed the 126 MB L2.
Multi-GPU: clips shard across ranks (weak scaling, no data-path collective); NCCL only for the barrier
and the max/sum reductions of the timings.
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MEM_FREQ = 5
METRIC = "propagated frames/sec, 480p, 1 object (mask propagation)"
DEFAULT_ACT = "fp16"
ACT_DTYPE = torch.float32  # set from --act in main()

# lanes / lockstep: clips a GPU propagates at a time in the headline measurement of each configuration;
# ref_frames / ref_bank: the bounded CPU sample (frames of the sub-clip, pre-filled certain bank frames)
CONFIGS = {
    "cfg2": dict(H=480, W=854, K=1, top_k=20, frames=101, inter=(0,), lanes=3, lockstep=4, ref_frames=11, ref_bank=10,
                 metric=METRIC, label="cfg2: DAVIS-shaped 480p (480x854 -> 480x864), 1 object, 101-frame clip, mem_freq 5, "
                                      "bank 1->21 frames, top-k 20"),
    "cfg3": dict(H=480, W=854, K=3, top_k=50, frames=251, inter=(0,), lanes=2, lockstep=1, ref_frames=4, ref_bank=25,
                 metric="propagated frames/sec, 480p, 3 objects (mask propagation)",
                 label="cfg3: DAVIS-shaped 480p, 3 objects, 251-frame clip, mem_freq 5, bank 1->51 frames, top-k 50"),
    "cfg4": dict(H=480, W=854, K=2, top_k=50, frames=61, inter=(0, 60), lanes=2, lockstep=1, ref_frames=5, ref_bank=6,
                 metric="propagated frames/sec, 480p, 2 objects, bidirectional propagation + FusionNet",
                 label="cfg4: DAVIS-shaped 480p, 2 objects, 61-frame clip, interactions on frames 0 then 60 (59 fused frames), "
                       "mem_freq 5, top-k 50"),
    "cfg5": dict(H=720, W=1280, K=5, top_k=50, frames=501, inter=(0,), lanes=1, lockstep=1, ref_frames=3, ref_bank=50,
                 metric="propagated frames/sec, 720p, 5 objects (mask propagation)",
                 label="cfg5: synthetic 720p, 5 objects, 501-frame clip, mem_freq 5, bank 1->101 frames, top-k 50"),
}
# module-level views of the default configuration (tests/test_bench_cpu.py)
H, W, K_OBJ, TOP_K = 480, 854, 1, 20
DUMP_BYTES = 60_000_000  # --dump-outputs: at most this much on disk (a cfg2 step returns 12 x 41 MB of masks)


def dump_outputs(out_dir, outputs, rank=0):
    """Write the masks of one step, {(clip, interaction): u8 [T, H, W]}, as float32 `masks_clip<c>_inter<j>.npy`.
    If they exceed DUMP_BYTES, every array keeps the same fixed, seeded sample of flat positions, written as
    float64 `masks_sample_index.npy` (by rank 0: every rank draws the same one)."""
    os.makedirs(out_dir, exist_ok=True)
    numel = next(iter(outputs.values())).size
    n = min(numel, DUMP_BYTES // (4 * len(outputs) + 8))
    idx = None
    if n < numel:
        idx = np.sort(np.random.default_rng(0).choice(numel, n, replace=False))
        if rank == 0:
            np.save(os.path.join(out_dir, "masks_sample_index.npy"), idx.astype(np.float64))
    for (c, j), m in sorted(outputs.items()):
        a = m.reshape(-1)[idx] if idx is not None else m
        np.save(os.path.join(out_dir, f"masks_clip{c:03d}_inter{j}.npy"), a.astype(np.float32))


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def _measured_traffic(fp16: bool):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from THIS round's
    `ncu --set full` capture (profiles/r02_traffic.json, written by tools/ncu_summary.py traffic); null when no
    capture of the current kernels is committed."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p)).get("fp16" if fp16 else "tf32")
    return (d["bytes"], d["launch"]) if d else (None, None)


def _workload_config(cfgd, name):
    """The `config` object of the JSON line: the WORKLOAD only, identical in both arms."""
    T = cfgd["frames"]
    return {"workload": cfgd["label"], "name": name, "size": [cfgd["H"], cfgd["W"]], "objects": cfgd["K"], "top_k": cfgd["top_k"],
            "mem_freq": MEM_FREQ, "clip_frames": T, "interactions": list(cfgd["inter"]),
            "l2": f"inputs larger than L2 ({T * 3 * cfgd['H'] * cfgd['W'] * 4 / 1e6:.0f} MB clip + 215 MB weights per clip-step)"}


def propagated_frames(T, inter):
    """Frames written by do_pass over the interactions of a configuration (host arithmetic)."""
    from mivos_b200 import schedule
    seen, n, nc = set(), 0, 0
    for idx in inter:
        seen.add(idx)
        nc += 1
        for fwd in (True, False):
            n += len(schedule.plan_pass(T, seen, idx, fwd, MEM_FREQ, nc).frames)
    return n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe).  One looping
    `nvidia-smi -lms` child, 500 ms period: every NVML query briefly stalls concurrent launches
    (measured: an in-process pynvml thread at 200 ms cost 15 % of `value`; the e2e region, which is
    not sampled, shows the unperturbed rate)."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", os.environ.get("MIVOS_BENCH_SMI_MS", "500")], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _best_cpu_threads(psd, frame):
    """The reference runs `torch` CPU ops on however many threads PyTorch is given.  On a many-core
    host oversubscription can make it SLOWER (measured: 128 threads are >10x slower than 16 on the
    GPU box), so give the CPU side its best case: time one query-encoder call (73 GFLOP of convs)
    at a few thread counts and keep the fastest.  MIVOS_CPU_THREADS overrides."""
    from oracle import stm_oracle as O
    env = os.environ.get("MIVOS_CPU_THREADS")
    if env:
        torch.set_num_threads(int(env))
        return int(env)
    ncpu = os.cpu_count() or 1
    # (PyTorch CPU convolutions stop scaling long before 64 threads; the sweep itself is bounded)
    cands = sorted({c for c in (min(ncpu, 64), 32, 16, 8) if 1 <= c <= ncpu}, reverse=True)
    best, best_t = cands[-1], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        O.get_query_values(psd, frame)  # warm the thread pool
        t0 = time.perf_counter()
        O.get_query_values(psd, frame)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def _dist():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------- CPU sample (both arms)
class CpuSample:
    """The bounded CPU sample of a configuration: `interact()` of the reference algorithm (oracle port,
    oracle/stm_oracle.py — the reference itself is Python and cannot travel to the GPU box, DESIGN.md)
    over the first `ref_frames` frames of the configuration's clip, with `ref_bank - 1` earlier frames
    already in the certain memory (memorised from the clip's own frames outside the timed region), so
    that the frames of the sample see the MEAN bank size of the full clip.  cfg4 adds the second
    interaction on the sample's last frame (every frame of its backward pass is fused)."""

    def __init__(self, cfgd, ref_frames=None):
        from oracle import stm_oracle as O
        from mivos_b200 import synth
        self.O, self.cfgd = O, cfgd
        self.n = int(ref_frames or cfgd["ref_frames"])
        self.psd = synth.make_prop_state_dict()
        self.fsd = synth.make_fusion_state_dict() if len(cfgd["inter"]) > 1 else None
        Hh, Ww, K = cfgd["H"], cfgd["W"], cfgd["K"]
        images, self.mask = synth.synthetic_clip(self.n + cfgd["ref_bank"], Hh, Ww, K, seed=1234)
        self.images = images[:, :self.n].contiguous()
        self.mask2 = synth.second_interaction_mask(K, Hh, Ww) if self.fsd is not None else None
        self.cores = _best_cpu_threads(self.psd, O.pad_divide_by(images[:, 0], 16)[0])
        # certain memory of ref_bank - 1 earlier interactions: keys / values of OTHER frames of the clip
        pm = O.pad_divide_by(self.mask, 16)[0]
        ks, vs = [], []
        for j in range(cfgd["ref_bank"] - 1):
            k_, v_ = O.memorize(self.psd, O.pad_divide_by(images[:, self.n + j], 16)[0], pm[1:])
            ks.append(k_); vs.append(v_)
        self.pre_k = torch.cat(ks, 2) if ks else None
        self.pre_v = torch.cat(vs, 2) if vs else None
        self.frames = self._count()

    def _count(self):
        from mivos_b200 import schedule
        n, nc, seen = 0, self.cfgd["ref_bank"] - 1, set()
        for idx in self._inter():
            seen.add(idx); nc += 1
            for fwd in (True, False):
                n += len(schedule.plan_pass(self.n, seen, idx, fwd, MEM_FREQ, nc).frames)
        return n

    def _inter(self):
        return (0,) if self.fsd is None else (0, self.n - 1)

    def run(self):
        """One sample: returns (seconds, u8 masks)."""
        cfgd = self.cfgd
        core = self.O.OracleInferenceCore(self.psd, self.fsd, self.images, cfgd["K"], mem_freq=MEM_FREQ, top_k=cfgd["top_k"])
        core.certain_mem_k, core.certain_mem_v = self.pre_k, self.pre_v
        t0 = time.perf_counter()
        out = core.interact(self.mask, 0)
        if self.fsd is not None:
            out = core.interact(self.mask2, self.n - 1)
        return time.perf_counter() - t0, out

    def describe(self, dt):
        b = self.cfgd["ref_bank"]
        return (f"oracle interact() on the first {self.n} frames ({self.frames} propagated) of the same clip with the bank "
                f"pre-filled to {b} frames (mean bank a frame of the full clip sees), {dt:.1f} s, {self.cores} torch threads "
                f"(fastest of a sweep up to {os.cpu_count()} host cores)")


def run_reference(args, cfgd, cfg_name):
    """The reference's algorithm on the host cores, each step one bounded sample of `config` (CpuSample)."""
    rank, world, _ = _dist()
    if rank != 0:
        return
    torch.set_grad_enabled(False)
    sample = CpuSample(cfgd, args.ref_frames)
    times = []
    for i in range(args.warmup + args.steps):
        dt, _ = sample.run()
        if i >= args.warmup:
            times.append(dt)
    total = sum(times)
    fps = sample.frames * len(times) / total
    print(json.dumps({
        "impl": "reference", "metric": cfgd["metric"], "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": _workload_config(cfgd, cfg_name),
        "frames_per_step": sample.frames,
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": sample.cores, "host_cores": os.cpu_count(), "kind": "port",
                         "sample": sample.describe(total / len(times)), "torch": torch.__version__},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


# ------------------------------------------------------------------------------------- our arm
def _bracketed_pass(mivos_b200, ops, net, clips, masks, dev, fuse=None, inter=(0,), masks2=None):
    """One extra EAGER pass over `clips` (one clip, or several in lock-step) with CUDA events around
    every convolution and memory-read call on the launching stream.  Returns (records, GPU ms of the pass).
    Graph replay is switched off for the pass (per-launch events need eager launches: same kernels, same
    order) and restored afterwards."""
    rec = {"conv": [], "memread": []}
    orig_conv, orig_mr = ops.conv_gemm, ops.memory_read

    def conv_prof(x, pc, n, h, w, out, **kw):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = orig_conv(x, pc, n, h, w, out, **kw)
        b.record()
        rec["conv"].append((a, b, 2.0 * n * h * w * pc.ksize * pc.ksize * pc.cin * pc.cout))
        return r

    def mr_prof(bank_k, bank_v, slots, qk, top_k, out, **kw):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = orig_mr(bank_k, bank_v, slots, qk, top_k, out, **kw)
        b.record()
        if kw.get("dyn_slots") is not None:  # graph-style step: `slots` is the capacity, the live count is on the device
            slots = int(kw["dyn_slots"][0])
        kk, hw = bank_k.shape[0], qk.shape[-2]
        rec["memread"].append((a, b, 2.0 * 128 * slots * hw * kk + 2.0 * top_k * 512 * hw * kk,
                               4.0 * (kk * slots * 128 + kk * top_k * hw * 512 + hw * 128 + kk * hw * 512)))
        return r

    eng = net.engine()
    lock_steps = list(eng.__dict__.get("_lock_steps", {}).values())
    saved_flags = [st.use_graph for st in lock_steps]
    saved_env = os.environ.get("MIVOS_GRAPH")
    # the batched query pass normally runs on the network's side stream, concurrently with the frame loop: a
    # bracket around a launch of one stream would then include whatever the other stream's kernels took from it
    # (r02c9: the same memory read bracketed at 457 us and at 885 us in two runs).  For this pass the query pass
    # is issued on the launching stream, so every bracket times its own launch only.
    saved_qs = eng.__dict__.get("_qstream")
    eng._qstream = torch.cuda.current_stream(dev)
    ops.conv_gemm, ops.memory_read = conv_prof, mr_prof
    os.environ["MIVOS_GRAPH"] = "0"
    for st in lock_steps:
        st.use_graph = False
    try:
        k_obj = masks[0].shape[0] - 1
        cores = [mivos_b200.InferenceCore(net, fuse, im, k_obj, mem_profile=0, mem_freq=MEM_FREQ, device=dev) for im in clips]
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        pe0.record()
        for j, idx in enumerate(inter):
            ms = masks if j == 0 else masks2
            if len(cores) == 1:
                cores[0].interact(ms[0], idx)
            else:
                mivos_b200.LockstepSession(cores).interact(ms, idx)
        pe1.record()
        torch.cuda.synchronize()
        prof_ms = pe0.elapsed_time(pe1)  # GPU time of this pass: the denominator of the shares
    finally:
        ops.conv_gemm, ops.memory_read = orig_conv, orig_mr
        eng._qstream = saved_qs
        if saved_env is None:
            os.environ.pop("MIVOS_GRAPH", None)
        else:
            os.environ["MIVOS_GRAPH"] = saved_env
        for st, flag in zip(lock_steps, saved_flags):
            st.use_graph = flag
    return rec, prof_ms


def _roofline_dicts(rec, prof_ms, peaks, peak_src, fp16, what):
    conv_ms = sum(a.elapsed_time(b) for a, b, _ in rec["conv"])
    conv_fl = sum(f for _, _, f in rec["conv"])
    tf32_peak = peaks["bf16_tflops_sustained"] / 2.0
    conv_peak = peaks["bf16_tflops_sustained"] if fp16 else tf32_peak
    ach = conv_fl / (conv_ms / 1e3) / 1e12
    traffic, traffic_launch = _measured_traffic(fp16)
    roof = {"kernel": f"conv_gemm_persistent_kernel (tcgen05 kind::{'f16' if fp16 else 'tf32'} implicit GEMM, all conv layers of the step)",
            "bound": "tensor", "achieved": ach, "peak": conv_peak, "unit": "TFLOP/s", "frac": ach / conv_peak,
            # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel from this round's
            # `ncu --set full` capture (profiles/r02_traffic.json); null when no capture of the current kernels exists
            "traffic": traffic, "traffic_launch": traffic_launch,
            "launches": len(rec["conv"]), "avg_launch_us": 1e3 * conv_ms / max(1, len(rec["conv"])),
            "share_of_step": conv_ms / prof_ms, "measured_on": what,
            "peak_source": (f"{peak_src}: sustained dense bf16 {peaks['bf16_tflops_sustained']:.0f} (kind::f16 issues at the bf16 rate)" if fp16 else
                            f"{peak_src}: TF32 dense = sustained bf16 {peaks['bf16_tflops_sustained']:.0f} / 2 (kind::tf32 issues at half the bf16 rate)"),
            "note": "event-bracketed eager launches, the batched query pass issued on the launching stream for this pass "
                    "(no cross-stream contention inside a bracket): durations include launch gaps, so this is a lower bound; "
                    "share_of_step = bracketed time / GPU time of the same pass"}
    mr_ms = sum(a.elapsed_time(b) for a, b, _, _ in rec["memread"])
    mr_fl = sum(f for _, _, f, _ in rec["memread"])
    mr_by = sum(by for _, _, _, by in rec["memread"])
    roof_mr = {"kernel": "memory_read (candidate pass on tcgen05 + exact selection / read-out)", "bound": "tensor",
               "achieved": mr_fl / (mr_ms / 1e3) / 1e12, "peak": tf32_peak, "unit": "TFLOP/s",
               "frac": mr_fl / (mr_ms / 1e3) / 1e12 / tf32_peak, "hbm_gbs": mr_by / (mr_ms / 1e3) / 1e9,
               "hbm_frac": mr_by / (mr_ms / 1e3) / 1e9 / peaks["hbm_gbs"], "launches": len(rec["memread"]),
               "avg_call_us": 1e3 * mr_ms / max(1, len(rec["memread"])), "share_of_step": mr_ms / prof_ms, "measured_on": what}
    return roof, roof_mr


def _cuda_eager(cfgd, dev, frames_cap=101):
    """The reference's own PyTorch ops (oracle port) with every tensor on the GPU: eager launches into
    cuDNN / cuBLAS / ATen — the library kernels this repository's hand-written path replaces, on the same
    box, same clip, same weights.  fp32 with PyTorch's default flags (cuDNN convolutions may use TF32,
    matmuls do not) and under torch.autocast(fp16) as the reference GUI runs (interactive_gui.py:990);
    cudnn.benchmark is switched ON (the eager path's best case; the reference's inference scripts leave it
    off).  Clips longer than `frames_cap` are truncated (the oracle caches every frame's features)."""
    from oracle import stm_oracle as O
    from mivos_b200 import synth
    T = min(cfgd["frames"], frames_cap)
    inter = tuple(i if i < T else T - 1 for i in cfgd["inter"])
    images, mask = synth.synthetic_clip(T, cfgd["H"], cfgd["W"], cfgd["K"], seed=1234)
    mask2 = synth.second_interaction_mask(cfgd["K"], cfgd["H"], cfgd["W"]) if len(inter) > 1 else None
    psd = {k: v.to(dev) for k, v in synth.make_prop_state_dict().items()}
    fsd = {k: v.to(dev) for k, v in synth.make_fusion_state_dict().items()} if len(inter) > 1 else None
    images, mask = images.to(dev), mask.to(dev)
    mask2 = None if mask2 is None else mask2.to(dev)
    nfr = propagated_frames(T, inter)
    out = {"frames": nfr, "clip_frames": T, "flags": "cudnn.benchmark=True; fp32: torch defaults (cudnn.allow_tf32=True, matmul fp32)"}
    old = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    try:
        for tag, ctx in (("fp32", None), ("autocast_fp16", torch.float16)):
            def once():
                core = O.OracleInferenceCore(psd, fsd, images, cfgd["K"], mem_freq=MEM_FREQ, top_k=cfgd["top_k"], device=dev)
                for j, idx in enumerate(inter):
                    core.interact(mask if j == 0 else mask2, idx)
                return core
            best = None
            for rep in range(2):  # first repetition warms cuDNN's autotuner and the allocator
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                if ctx is None:
                    once()
                else:
                    with torch.autocast("cuda", dtype=ctx):
                        once()
                e1.record()
                torch.cuda.synchronize()
                best = e0.elapsed_time(e1)
            out[tag] = {"value": nfr / (best / 1e3), "unit": "frames/s", "ms": best}
            gc.collect(); torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.benchmark = old
    return out


def run_ours(args, cfgd, cfg_name):
    rank, world, local = _dist()
    torch.set_grad_enabled(False)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    import mivos_b200
    from mivos_b200 import _lib, ops, sharding, synth

    Hh, Ww, K, top_k, T, inter = cfgd["H"], cfgd["W"], cfgd["K"], cfgd["top_k"], args.frames or cfgd["frames"], cfgd["inter"]
    inter = tuple(i if i < T else T - 1 for i in inter)
    frames = propagated_frames(T, inter)
    nh, nw = (Hh + 15) // 16 * 16, (Ww + 15) // 16 * 16
    sd = synth.make_prop_state_dict()
    fsd = synth.make_fusion_state_dict() if len(inter) > 1 else None
    mask2 = synth.second_interaction_mask(K, Hh, Ww) if len(inter) > 1 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    class Lane:
        """One clip slot of this GPU: own network object (own packed weights, workspaces and captured
        graphs), own CUDA stream, own clips.  Lanes run concurrently from Python threads; their kernels
        interleave on the device and fill the SMs the latency-bound per-frame chain leaves idle."""

        def __init__(self, i, C, L, act):
            self.L = L
            self.net = mivos_b200.PropagationNetwork(top_k=top_k, act_dtype=act)
            self.net.load_state_dict(sd)
            self.net = self.net.to(dev)
            self.fuse = None
            if fsd is not None:
                self.fuse = mivos_b200.FusionNet()
                self.fuse.load_state_dict(fsd)
                self.fuse = self.fuse.to(dev)
            self.stream = torch.cuda.Stream(device=dev)
            mine = sharding.clips_of_rank(world * C * L, rank, world)  # clip c -> rank c % world
            self.clips = mine[i * L:(i + 1) * L]
            data = [synth.synthetic_clip(T, Hh, Ww, K, seed=1234 + c) for c in self.clips]
            self.images_l, self.masks_l = [d[0] for d in data], [d[1] for d in data]
            self.checksums = [0] * L
            self.results = []
            self.last = []  # per interaction, the masks of every clip from the latest step
            self.step_wall = []

        def run(self, cores, nsteps):
            """`nsteps` steps over this lane's L sessions, reused from step to step: InferenceCore.reset()
            returns a session to its freshly-constructed state (query cache dropped, certain memories
            forgotten), so every step recomputes everything; what is NOT repeated is the construction —
            clip upload / pinning and buffer allocation — which the metric excludes (SURVEY.md 8d)."""
            torch.cuda.set_device(dev)
            with torch.cuda.stream(self.stream):
                for _ in range(nsteps):
                    # interact() returns the host u8 masks of the clip: the D2H read of the step's
                    # result is inside the timed region, the checksum over them is not
                    t0 = time.perf_counter()
                    for c in cores:
                        c.reset()
                    res, outs = None, []
                    for j, idx in enumerate(inter):
                        ms = self.masks_l if j == 0 else [mask2] * self.L
                        if self.L == 1:
                            res = [cores[0].interact(ms[0], idx)]
                        else:
                            res = mivos_b200.LockstepSession(cores).interact(ms, idx)
                        outs.append(res)
                    self.results.append(res)
                    self.last = outs
                    self.step_wall.append(time.perf_counter() - t0)  # interact() ends with a stream sync

        def take_checksum(self):
            for per_clip in self.results:
                for j, m in enumerate(per_clip):
                    self.checksums[j] += int(m.sum(dtype="int64"))
            self.results = []

    def timed_region(lanes, C, L, mem_profile, nsteps, warm):
        cores = [[mivos_b200.InferenceCore(ln.net, ln.fuse, ln.images_l[j], K, mem_profile=mem_profile, mem_freq=MEM_FREQ,
                                           device=dev) for j in range(L)] for ln in lanes]
        for ln, cs in zip(lanes, cores):  # warm-up lane by lane (graph capture is single-threaded)
            ln.run(cs, warm)
            ln.results = []
            ln.step_wall = []
        barrier()
        l0 = _lib.load().mivos_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        main = torch.cuda.current_stream(dev)
        t0 = time.perf_counter()
        e0.record(main)
        for ln in lanes:
            ln.stream.wait_event(e0)
        threads = [threading.Thread(target=ln.run, args=(cs, nsteps)) for ln, cs in zip(lanes, cores)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        for ln in lanes:
            main.wait_stream(ln.stream)
        e1.record(main)
        barrier()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        launches = _lib.load().mivos_launch_count() - l0
        for ln in lanes:
            ln.take_checksum()
        step_ms = [[round(1e3 * x, 2) for x in ln.step_wall] for ln in lanes]
        per_clip = sharding.gather_clip_results([(c, ln.checksums[j]) for ln in lanes for j, c in enumerate(ln.clips)],
                                                world * C * L)
        del cores
        return {"ms": sharding.max_over_ranks(ms, dev), "launches": launches, "checksum": sum(per_clip), "wall": wall, "step_ms": step_ms}

    def measure(act, C, L, nsteps, warm, sample_clocks=False, keep_outputs=False):
        """value (mem_profile 0) and e2e (mem_profile 1) of one (element type, lanes, lock-step) setting.
        keep_outputs: also return the masks of the last `value` step, {(clip, interaction): u8 [T, H, W]}."""
        lanes = [Lane(i, C, L, act) for i in range(C)]
        sampler = ClockSampler(local) if sample_clocks else None
        if sampler:
            sampler.start()
        r0 = timed_region(lanes, C, L, 0, nsteps, warm)
        clocks = sampler.stop() if sampler else None
        outputs = {(c, j): per_clip[i] for ln in lanes for j, per_clip in enumerate(ln.last)
                   for i, c in enumerate(ln.clips)} if keep_outputs else None
        r1 = timed_region(lanes, C, L, 1, nsteps, max(1, warm // 3))
        n = world * C * L * frames * nsteps
        out = {"value": n / (r0["ms"] / 1e3), "e2e": n / (r1["ms"] / 1e3), "ms_per_step": r0["ms"] / nsteps,
               "e2e_ms_per_step": r1["ms"] / nsteps, "steps": nsteps, "lanes": C, "lockstep": L, "r0": r0, "r1": r1, "clocks": clocks,
               "outputs": outputs}
        return out, lanes

    C = max(1, args.clips_per_gpu if args.clips_per_gpu is not None else cfgd["lanes"])
    L = max(1, args.lockstep if args.lockstep is not None else cfgd["lockstep"])
    head, lanes = measure(ACT_DTYPE, C, L, args.steps, args.warmup, sample_clocks=True, keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, head.pop("outputs"), rank)
    h2d = world * C * L * (T * 3 * nh * nw * 4 + len(inter) * (K + 1) * Hh * Ww * 4)  # whole job, like `value`
    d2h = world * C * L * len(inter) * T * Hh * Ww

    # ---------------- roofline of the dominant kernel (conv implicit GEMM) + the memory read,
    # measured live with CUDA events around each launch on the launching stream (rank 0)
    roof, roof_mr, cpu, extra = None, None, None, {}
    peaks, peak_src = _peaks()
    fp16 = ACT_DTYPE == torch.float16
    ln0 = lanes[0]
    if rank == 0 and not args.skip_roofline:
        m2 = None if mask2 is None else [mask2]
        try:  # (a) one clip, eager — the pass every earlier profile of this repo refers to
            rec, prof_ms = _bracketed_pass(mivos_b200, ops, ln0.net, ln0.images_l[:1], ln0.masks_l[:1], dev, ln0.fuse, inter, m2)
            roof, roof_mr = _roofline_dicts(rec, prof_ms, peaks, peak_src, fp16, "one clip, eager")
        except Exception as e:  # never lose the timed numbers to a failure of the explanatory pass
            extra["roofline_error"] = f"{type(e).__name__}: {e}"
        if L > 1 and roof is not None:
            try:  # (b) the unit of the timed workload: one lane = L clips in lock-step (C*K maps per conv launch)
                rec, prof_ms = _bracketed_pass(mivos_b200, ops, ln0.net, ln0.images_l, ln0.masks_l, dev, ln0.fuse, inter,
                                               None if mask2 is None else [mask2] * L)
                r2, mr2 = _roofline_dicts(rec, prof_ms, peaks, peak_src, fp16, f"one lane: {L} clips in lock-step, eager")
                extra.update({"roofline_single_clip": roof, "roofline_memory_read_single_clip": roof_mr})
                roof, roof_mr = r2, mr2
            except Exception as e:
                extra["roofline_lockstep_error"] = f"{type(e).__name__}: {e}"
    del lanes, ln0
    gc.collect(); torch.cuda.empty_cache()

    # ---------------- the same metric through ONE InferenceCore.interact, and on the fp32-comparable path
    xs = max(1, min(args.steps, args.extra_steps))
    single = tf32 = None
    if not args.skip_extras:
        if C * L > 1:
            s, ls = measure(ACT_DTYPE, 1, 1, xs, 2)
            single = {"value": s["value"], "e2e": s["e2e"], "unit": "frames/s", "steps": xs, "ms_per_step": s["ms_per_step"],
                      "path": "1 lane x 1 clip: InferenceCore.interact as the unchanged reference callers issue it"}
            del ls
            gc.collect(); torch.cuda.empty_cache()
        other = torch.float32 if fp16 else torch.float16
        t, lt = measure(other, C, L, xs, 2)
        tf32 = {"dtype": "tf32" if fp16 else "fp16", "value": t["value"], "e2e": t["e2e"], "unit": "frames/s", "steps": xs,
                "ms_per_step": t["ms_per_step"], "lanes": C, "lockstep": L}
        if rank == 0 and not args.skip_roofline:
            try:
                l0_ = lt[0]
                rec, prof_ms = _bracketed_pass(mivos_b200, ops, l0_.net, l0_.images_l, l0_.masks_l, dev, l0_.fuse, inter,
                                               None if mask2 is None else [mask2] * L)
                r3, mr3 = _roofline_dicts(rec, prof_ms, peaks, peak_src, not fp16,
                                          f"one lane: {L} clip(s){' in lock-step' if L > 1 else ''}, eager")
                tf32["roofline"], tf32["roofline_memory_read"] = r3, mr3
            except Exception as e:
                tf32["roofline_error"] = f"{type(e).__name__}: {e}"
        del lt
        gc.collect(); torch.cuda.empty_cache()

    eager = None
    if rank == 0 and not args.skip_cuda_eager:
        try:
            eager = _cuda_eager(cfgd, dev)
        except Exception as e:
            eager = {"error": f"{type(e).__name__}: {e}"}
        gc.collect(); torch.cuda.empty_cache()

    # ---------------- CPU baseline: the oracle port on this box's host cores, bounded sample of `config`
    if rank == 0 and world == 1 and not args.skip_cpu_baseline:
        sample = CpuSample(cfgd, args.ref_frames)
        sample.run()  # warm the thread pool / allocator
        dt, _ = sample.run()
        cpu = {"value": sample.frames / dt, "unit": "frames/s", "cores": sample.cores, "kind": "port",
               "sample": sample.describe(dt), "torch": torch.__version__}

    if rank == 0:
        act_name = "fp16" if fp16 else "tf32"
        line = {
            "metric": cfgd["metric"], "value": head["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": act_name, "data": "synthetic", "config": _workload_config(cfgd, cfg_name),
            "execution": {"frames_per_step": frames * C * L * world, "clips_per_step": world * C * L, "clips_per_gpu": C * L, "lanes": C,
                          "lockstep": L, "parallelism": f"clip-sharded: {world} GPU(s) x {C} concurrent lane(s) per GPU (one CUDA stream + "
                          f"one thread per lane)" + (f" x {L} clips advanced in lock-step as one batch per lane" if L > 1 else "")},
            "e2e": {"value": head["e2e"], "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": head["e2e_ms_per_step"], "path": "InferenceCore(mem_profile=1).interact(): pinned host clip, per-frame H2D, masks D2H"},
            "single_session": single, ("tf32" if fp16 else "fp16"): tf32,
            "value_single_session": None if single is None else single["value"],
            "e2e_single_session": None if single is None else single["e2e"],
            ("value_tf32" if fp16 else "value_fp16"): None if tf32 is None else tf32["value"],
            ("e2e_tf32" if fp16 else "e2e_fp16"): None if tf32 is None else tf32["e2e"],
            "roofline_tf32": None if (tf32 is None or not fp16) else tf32.get("roofline"),
            "reference_cuda_eager": eager,
            "gpu_launches": head["r0"]["launches"], "launch_mode": "cuda-graph replay per frame" if os.environ.get("MIVOS_GRAPH", "1") != "0" else "eager",
            "clocks": head["clocks"], "roofline": roof, "roofline_memory_read": roof_mr, **extra,
            "cpu_baseline": cpu, "mask_checksum": [head["r0"]["checksum"], head["r1"]["checksum"]], "wall_s": [head["r0"]["wall"], head["r1"]["wall"]],
            "interact_wall_ms": {"resident": head["r0"]["step_ms"], "e2e": head["r1"]["step_ms"]},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS), help="BASELINE.json configuration (default cfg2: the metric's)")
    ap.add_argument("--frames", type=int, default=None, help="override the clip length of the configuration")
    ap.add_argument("--ref-frames", type=int, default=None, help="frames of the bounded CPU sample (default per configuration)")
    ap.add_argument("--extra-steps", type=int, default=4, help="timed steps of the single-session / other-dtype measurements")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="no single-session / other-dtype measurements")
    ap.add_argument("--skip-cuda-eager", action="store_true", help="no PyTorch-eager CUDA comparator")
    ap.add_argument("--skip-roofline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the masks the last timed step returned as DIR/<name>.npy (float32; a fixed sample if large)")
    ap.add_argument("--act", default=os.environ.get("MIVOS_ACT_DTYPE", DEFAULT_ACT), choices=["tf32", "fp16"],
                    help="convolution operand / activation type of the headline measurement (fp16 = the reference GUI's autocast "
                         "precision; the other type is measured beside it)")
    ap.add_argument("--clips-per-gpu", type=int, default=(int(os.environ["MIVOS_CLIPS_PER_GPU"]) if "MIVOS_CLIPS_PER_GPU" in os.environ else None),
                    help="concurrent lanes per GPU (own network object, CUDA stream and Python thread each); default per configuration")
    ap.add_argument("--lockstep", type=int, default=(int(os.environ["MIVOS_LOCKSTEP"]) if "MIVOS_LOCKSTEP" in os.environ else None),
                    help="clips each lane advances in lock-step as ONE batch through the conv layers (mivos_b200.LockstepSession); "
                         "1 = off; default per configuration (cfg2: 3 lanes x 4 clips)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global ACT_DTYPE
    ACT_DTYPE = torch.float16 if args.act == "fp16" else torch.float32
    cfgd = dict(CONFIGS[args.config])
    if args.impl == "reference":
        run_reference(args, cfgd, args.config)
    else:
        run_ours(args, cfgd, args.config)


if __name__ == "__main__":
    main()
