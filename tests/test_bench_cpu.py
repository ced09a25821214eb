"""CPU: bench.py's roofline helpers (the event-bracketed eager pass over one clip and over one lock-step
lane, and the dictionaries built from it) run over the emulated operators, so that the measurement code
itself — which switches graph replay off and back on around the pass — cannot break the bench line."""
import os
import sys

import torch

import abi_emulator

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_bracketed_pass_and_roofline_dicts(monkeypatch, prop_sd):
    import bench
    from oracle import weights as Wt
    mv = abi_emulator.install_host_runtime(monkeypatch)
    from mivos_b200 import ops
    net = mv.PropagationNetwork(top_k=20, act_dtype=torch.float32)
    net.load_state_dict(prop_sd, strict=True)
    clips = [Wt.synthetic_clip(7, 64, 96, bench.K_OBJ, seed=70 + i) for i in range(2)]
    images, masks = [c[0] for c in clips], [c[1] for c in clips]
    peaks = {"hbm_gbs": 6500.0, "bf16_tflops": 1600.0, "bf16_tflops_sustained": 1400.0}
    monkeypatch.setenv("MIVOS_GRAPH", "1")  # what a bench run has; the pass must switch it off and restore it
    orig_conv, orig_mr = ops.conv_gemm, ops.memory_read

    rec, ms = bench._bracketed_pass(mv, ops, net, images[:1], masks[:1], "cpu")
    assert len(rec["memread"]) == 6 and len(rec["conv"]) > 100 and ms == 1.0
    roof, roof_mr = bench._roofline_dicts(rec, ms, peaks, "test", True, "one clip, eager")
    assert roof["bound"] == "tensor" and roof["peak"] == 1400.0 and 0 < roof["frac"] and roof["launches"] == len(rec["conv"])
    assert roof_mr["peak"] == 700.0 and roof_mr["launches"] == 6 and roof_mr["measured_on"] == "one clip, eager"
    assert os.environ["MIVOS_GRAPH"] == "1" and ops.conv_gemm is orig_conv and ops.memory_read is orig_mr

    # lock-step lane: a cached step object in graph mode must run eagerly for the pass and be restored
    from mivos_b200.lockstep import _LockStep
    cores = [mv.InferenceCore(net, None, im, bench.K_OBJ, mem_freq=bench.MEM_FREQ, device="cpu") for im in images]
    monkeypatch.setenv("MIVOS_GRAPH", "0")
    mv.LockstepSession(cores).interact(masks, 0)  # creates and caches the step (eager here: no CUDA graphs on the CPU)
    monkeypatch.setenv("MIVOS_GRAPH", "1")
    steps = list(net.engine().__dict__["_lock_steps"].values())
    assert len(steps) == 1 and isinstance(steps[0], _LockStep)
    steps[0].use_graph = True
    rec2, _ = bench._bracketed_pass(mv, ops, net, images, masks, "cpu")
    assert steps[0].use_graph is True and os.environ["MIVOS_GRAPH"] == "1"
    assert len(net.engine().__dict__["_lock_steps"]) == 1  # the pass reused the cached step
    assert len(rec2["memread"]) == 6  # ONE read per lock-step frame serves both clips (query sets, q_div)
    # C*K maps per launch: fewer conv launches than two single-clip passes, same algorithmic flops
    assert len(rec2["conv"]) < 2 * len(rec["conv"])
    fl1, fl2 = sum(f for _, _, f in rec["conv"]), sum(f for _, _, f in rec2["conv"])
    assert abs(fl2 - 2 * fl1) <= 1e-6 * fl2
    # live slot counts (read through dyn_slots), not the bank capacity, enter the memory-read flops
    assert abs(sum(f for _, _, f, _ in rec2["memread"]) - 2 * sum(f for _, _, f, _ in rec["memread"])) < 1.0


def test_cpu_sample_is_the_configured_workload(monkeypatch):
    """The bounded CPU sample both arms time (bench.CpuSample): same shapes / top-k as `config`, bank pre-filled
    so that every frame of the sample sees the mean bank of the full clip; frame count from the pass plan."""
    import bench
    nthreads = torch.get_num_threads()
    monkeypatch.setenv("MIVOS_CPU_THREADS", str(nthreads))  # no sweep, and the process-wide thread count stays what it was
    cfgd = dict(bench.CONFIGS["cfg2"], H=64, W=96, ref_frames=7, ref_bank=4)
    s = bench.CpuSample(cfgd)
    assert s.frames == 6 and s.pre_k.shape == (1, 128, 3, 4, 6) and s.pre_v.shape == (1, 512, 3, 4, 6)
    dt, masks = s.run()
    assert masks.shape == (7, 64, 96) and dt > 0
    # the oracle saw 4 certain frames (3 pre-filled + the interacted one): first frame reads 4 bank frames
    core = s.O.OracleInferenceCore(s.psd, None, s.images, 1, mem_freq=bench.MEM_FREQ, top_k=20)
    core.certain_mem_k, core.certain_mem_v = s.pre_k, s.pre_v
    core.interact(s.mask, 0)
    assert core.bank_trace[0] == (1, 4) and core.bank_trace[-1] == (6, 5)
    # cfg4: two interactions, every frame of the second pass is fused
    cfgd4 = dict(bench.CONFIGS["cfg4"], H=64, W=96, ref_frames=5, ref_bank=2, top_k=20)  # 24 slots per bank frame
    s4 = bench.CpuSample(cfgd4)
    assert s4.frames == 4 + 3
    dt4, m4 = s4.run()
    assert m4.shape == (5, 64, 96)


def test_dump_outputs_whole_and_sampled(tmp_path, monkeypatch):
    """--dump-outputs: float32 masks per (clip, interaction), whole when they fit DUMP_BYTES, otherwise the
    same seeded sample of positions in every array, identical from run to run."""
    import bench
    import numpy as np
    rng = np.random.default_rng(1)
    outs = {(c, j): rng.integers(0, 3, (5, 8, 12), dtype=np.uint8) for c in range(3) for j in range(2)}
    bench.dump_outputs(str(tmp_path / "whole"), outs)
    assert not (tmp_path / "whole" / "masks_sample_index.npy").exists()
    for (c, j), m in outs.items():
        a = np.load(tmp_path / "whole" / f"masks_clip{c:03d}_inter{j}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, m)
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * (4 * len(outs) + 8))  # room for 100 elements per array
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), outs)
    idx = np.load(tmp_path / "a" / "masks_sample_index.npy")
    assert idx.dtype == np.float64 and idx.shape == (100,) and len(set(idx.tolist())) == 100
    assert np.array_equal(idx, np.load(tmp_path / "b" / "masks_sample_index.npy"))
    for (c, j), m in outs.items():
        a = np.load(tmp_path / "a" / f"masks_clip{c:03d}_inter{j}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, m.reshape(-1)[idx.astype(np.int64)])
    assert sum(f.stat().st_size - 128 for f in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES  # (npy headers: 128 B)


def test_propagated_frames_and_workload_config():
    import bench
    assert bench.propagated_frames(101, (0,)) == 100
    assert bench.propagated_frames(61, (0, 60)) == 60 + 59
    assert bench.propagated_frames(9, (4,)) == 8
    a = bench._workload_config(bench.CONFIGS["cfg2"], "cfg2")
    assert a["clip_frames"] == 101 and a["top_k"] == 20 and a["objects"] == 1
    # identical in both arms by construction: only the configuration enters
    assert a == bench._workload_config(dict(bench.CONFIGS["cfg2"]), "cfg2")
