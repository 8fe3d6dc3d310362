#!/usr/bin/env python
"""bench.py -- learn_from_batch steps/sec, DQN + prioritized replay, batch 512 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...     # the reference's CPU path (oracle port), rank 0 only
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N    # one process per GPU, NCCL gradient all-reduce
    python bench.py ... --dump-outputs DIR      # also write what the last timed step computed to DIR/*.npy (rank 0)

Workload = BASELINE config 2 ("Atari Pong DQN, 1M-transition PrioritizedExperienceReplay, 84x84x4 uint8, batch 512"):
per GPU one HBM-resident replay shard with a 2^20-leaf fp64 sum/min/max tree and 2^20 ring slots (59.2 GB), synthetic
transitions (uniform random uint8 frames, actions U{0..5}, rewards in {-1,0,1}, done every 1000th), priorities
|N(0,1)|, DQN network conv(32,8,4)-conv(64,4,2)-conv(64,3,1)-fc512-fc6 with random (glorot) weights, Huber loss,
Adam(2.5e-4, 0.9, 0.99, 1e-4), gamma 0.99, hard target copy every 2500 train steps.

One "step" = Agent.train(): uniforms (host MT19937, 4 KB H2D) -> fused PER sample + gather -> target/online forward ->
TD targets -> Huber head -> backward -> global norm -> [all-reduce] -> Adam -> priority update (libm-exact route:
4 KB of TD errors to the host, 8 KB of priorities back, overlapped with the backward pass).
  value : steps/s with the replay resident in HBM and no per-step result read-back (device-timed, max over ranks)
  e2e   : steps/s through the public plugin API with host buffers: per step 4 new host transitions are store()d
          (num_consecutive_playing_steps = 4, dqn_agent.py:37) and the loss is read back (fetch=True)
Inputs (59 GB ring per GPU) are far larger than the 126 MB L2, so consecutive iterations cannot hit in L2.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OBS = (84, 84, 4)
ROW = 84 * 84 * 4
N_ACTIONS = 6
BATCH = 512
ENV_STEPS_PER_TRAIN = 4
# algorithmic bytes of ONE fused sample+gather launch (SURVEY.md section 8d / BASELINE.md contract figure, staged copy
# written): read B*(2*28224+8+8+1) of transition columns + B*21*8 of tree, write the same columns + B*(8+8) idx/weight
GATHER_BYTES = BATCH * (2 * ROW + 8 + 8 + 1) * 2 + BATCH * 21 * 8 + BATCH * 16
# what the fused sample + gather + space-to-depth kernel moves: the uint8 frames are read once (28.9 MB), the bf16
# operand planes of the first convolution are written (2 bytes per pixel value: 57.8 MB), plus tree / small columns
GATHER_S2D_MOVED = BATCH * 2 * ROW * (1 + 2) + BATCH * (8 + 8 + 1) * 2 + BATCH * 21 * 8 + BATCH * 16
# frame-deduplicated replay: s and s' of a transition share 3 of their 8 frames -- 5 distinct 7,056-byte frames are read
# per sample (18.1 MB per batch; the 3 repeats hit L2), plus two int32[4] slot rows; the planes are written as before
GATHER_DEDUP_MOVED = BATCH * (5 * (ROW // 4) + 2 * 16) + BATCH * 2 * ROW * 2 + BATCH * (8 + 8 + 1) * 2 + BATCH * 21 * 8 + \
    BATCH * 16
# multiply-accumulates of one learn step per sample: target fwd + online fwd (9.346 M each) + backward
# (weight grads 9.346 M + data grads 6.069 M: conv2, conv3, fc1, out); the online forward is computed once
MACS_PER_SAMPLE = 2 * 9346048 + 9346048 + (9346048 - 3276800)


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, busy, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            try:
                busy.append(float(f[9]) >= 50.0)
            except (ValueError, IndexError):
                busy.append(True)
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        load = [c for c, b in zip(sm, busy) if b] or sm        # samples taken while the GPU was busy with the step
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_under_load": len(load)}


# =====================================================================================================================
def synth_chunk(rng, n):
    return (rng.randint(0, 6, n).astype(np.int64), rng.randint(-1, 2, n).astype(np.float64))


def fill_frame_stream(mem, size, device, gen, rng, episode=1000):
    """Synthetic Atari-like frame stream for the frame-deduplicated replay: episodes of `episode` transitions, every
    transition adds ONE new frame (the first of an episode two), states are the sliding 4-frame windows with the
    episode's first frame replicated at its start (observation_stacking_filter.py:89-101).  Appended in chunks of 16
    episodes: the distinct frames once + int32 [n, 4] indices into them (DeviceTransitionRing._append_frames)."""
    import torch
    done_total = 0
    while done_total < size:
        n_ep = min(16, (size - done_total + episode - 1) // episode)
        lens = [min(episode, size - done_total - e * episode) for e in range(n_ep)]
        lens = [l for l in lens if l > 0]
        n = int(sum(lens))
        nf = n + len(lens)
        frames = torch.randint(0, 256, (nf, 84 * 84), dtype=torch.uint8, device=device, generator=gen)
        si, s2i, done = np.zeros((n, 4), np.int32), np.zeros((n, 4), np.int32), np.zeros(n, np.uint8)
        t = f0 = 0
        for L in lens:
            j = np.arange(L)
            for c in range(4):
                si[t:t + L, c] = f0 + np.maximum(j - 3 + c, 0)
                s2i[t:t + L, c] = f0 + np.maximum(j - 2 + c, 0)
            done[t + L - 1] = 1 if L == episode else 0
            t += L
            f0 += L + 1
        a, r = synth_chunk(rng, n)
        mem.store_columns({"frames": frames, "state:observation": torch.from_numpy(si),
                           "next_state:observation": torch.from_numpy(s2i), "action": a, "reward": r,
                           "game_over": done})
        done_total += n


def build_device_agent(capacity, seed, device, config="dqn", frame_dedup=False):
    import torch
    from coach_b200.agents.dqn_agent import DDQNAgent, DDQNAgentParameters, DQNAgent, DQNAgentParameters
    from coach_b200.base_parameters import MiddlewareScheme
    from coach_b200.base_parameters import TrainingSteps
    from coach_b200.memories.memory import MemoryGranularity
    from coach_b200.memories.prioritized_experience_replay import PrioritizedExperienceReplayParameters
    from coach_b200.schedules import LinearSchedule
    dueling = config == "dueling"
    ap = DDQNAgentParameters() if dueling else DQNAgentParameters()
    ap.memory = PrioritizedExperienceReplayParameters()
    ap.memory.max_size = (MemoryGranularity.Transitions, capacity)
    ap.memory.frame_dedup = bool(frame_dedup)
    ap.memory.beta = LinearSchedule(0.4, 1, 12500000)
    ap.algorithm.num_steps_between_copying_online_weights_to_target = TrainingSteps(2500 if not dueling else 10000)
    ap.algorithm.num_consecutive_playing_steps.num_steps = ENV_STEPS_PER_TRAIN
    net = ap.network_wrappers["main"]
    net.batch_size = BATCH
    net.replace_mse_with_huber_loss = True
    if dueling:
        # BASELINE config 5 = presets/Atari_Dueling_DDQN_with_PER_OpenAI.py:14-19: DDQN, dueling head directly on the
        # conv map (MiddlewareScheme.Empty), lr 1e-4, global-norm clip 10, target copy every 40000 env steps
        net.learning_rate = 0.0001
        net.middleware_parameters.scheme = MiddlewareScheme.Empty
        net.heads_parameters = ["DuelingQHead"]
        net.clip_gradients = 10
    agent = (DDQNAgent if dueling else DQNAgent)(ap, observation_shape=OBS, num_actions=N_ACTIONS, device=device,
                                                 seed=seed)
    mem = agent.memory
    size = mem.power_of_2_size
    gen = torch.Generator(device=device).manual_seed(seed)
    rng = np.random.RandomState(seed)
    chunk = 1 << 14
    if frame_dedup:
        fill_frame_stream(mem, size, device, gen, rng)
    for lo in range(0, size if not frame_dedup else 0, chunk):
        n = min(chunk, size - lo)
        s = torch.randint(0, 256, (n, ROW), dtype=torch.uint8, device=device, generator=gen)
        s2 = torch.randint(0, 256, (n, ROW), dtype=torch.uint8, device=device, generator=gen)
        a, r = synth_chunk(rng, n)
        done = ((np.arange(lo, lo + n) % 1000) == 999).astype(np.uint8)
        mem.store_columns({"state:observation": s.view(n, *OBS), "next_state:observation": s2.view(n, *OBS),
                           "action": a, "reward": r, "game_over": done})
    # non-degenerate tree: |N(0,1)| errors on every leaf (device route for the bulk initialisation)
    err = torch.randn(size, dtype=torch.float64, device=device, generator=gen).abs()
    idx = torch.arange(size, dtype=torch.int64, device=device)
    mode = mem.priority_mode
    mem.priority_mode = "device"
    mem.update_priorities(idx, err)
    mem.priority_mode = mode
    torch.cuda.synchronize()
    return agent


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(agent, out_dir):
    """Writes what the last learn step computed, as a caller of Agent.train() / learn_from_batch sees it, to
    out_dir/<name>.npy: the loss and the squared global gradient norm the step returns, its sampled batch (leaf
    indices, importance weights), TD targets and errors, the priorities written back to the sampled leaves of the sum
    tree, and the online network's parameters after the optimizer step.  float32 / float64 only (the leaf indices are
    exact in float64).  The inputs depend only on the command-line arguments, so two builds can be compared file by
    file."""
    import torch
    torch.cuda.synchronize()
    net, mem, bb = agent.networks["main"], agent.memory, agent.batch_buffers
    idx = bb["idx"]
    outs = {"loss": agent.loss_dev, "grad_sumsq": net.sumsq, "idx": idx.to(torch.float64),
            "is_weights": bb["weight"], "td_targets": agent.targets, "td_errors": agent.td_err,
            "priorities": mem.sum_tree[mem.power_of_2_size - 1 + idx], "online_params": net.store.theta}
    outs = {k: v.detach().cpu().numpy() for k, v in outs.items()}
    for k, v in outs.items():
        assert v.dtype in (np.float32, np.float64), (k, v.dtype)
    total = sum(v.nbytes for v in outs.values())
    assert total <= DUMP_LIMIT_BYTES, "outputs of one step: %d bytes" % total
    os.makedirs(out_dir, exist_ok=True)
    for k, v in outs.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def host_transitions(rng, n, stacked_by_filter=False):
    """n new host-side transitions (what Agent.observe would hand to memory.store).  stacked_by_filter: the states are
    the LazyStacks an ObservationStackingFilter(4) hands out along one episode (one new 84x84 frame per transition,
    the other three shared with its neighbours), as in the reference's Atari presets."""
    from coach_b200.core_types import Transition
    out = []
    if stacked_by_filter:
        from coach_b200.filters.filter import ObservationStackingFilter
        flt = ObservationStackingFilter(4)
        s = flt.filter(rng.randint(0, 256, OBS[:2]).astype(np.uint8))
        for _ in range(n):
            s2 = flt.filter(rng.randint(0, 256, OBS[:2]).astype(np.uint8))
            out.append(Transition(state={"observation": s}, action=int(rng.randint(0, N_ACTIONS)),
                                  reward=float(rng.randint(-1, 2)), next_state={"observation": s2}, game_over=False))
            s = s2
        return out
    for _ in range(n):
        out.append(Transition(state={"observation": rng.randint(0, 256, OBS).astype(np.uint8)},
                              action=int(rng.randint(0, N_ACTIONS)), reward=float(rng.randint(-1, 2)),
                              next_state={"observation": rng.randint(0, 256, OBS).astype(np.uint8)},
                              game_over=False))
    return out


def run_device(args):
    import torch
    from coach_b200 import _lib, parallel
    rank, world = parallel.init_from_env()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    lib = _lib.load()
    lib.cb200_tune(b"gemm_tc", 0 if args.no_tc else 1)
    if args.no_tc:
        os.environ["CB200_GEMM_TILED"] = "0"      # no pre-split planes / tiled tcgen05 GEMMs either
    random.seed(1000 + rank)
    np.random.seed(1000 + rank)
    agent = build_device_agent(args.capacity, 100 + rank, device, args.config, frame_dedup=args.frame_dedup)
    mem = agent.memory
    if not args.no_l2_persist:
        lib.cb200_l2_persist(mem.sum_tree.data_ptr(), (1 << 17) * 8, _lib.current_stream())
    K, W = args.steps, max(args.warmup, 3)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def one_step(fetch):
        agent.total_steps_counter += ENV_STEPS_PER_TRAIN
        return agent.train(fetch=fetch)

    # ---- device-resident leg (value) ------------------------------------------------------------------------------
    # clocks / throttle reasons: nvidia-smi samples every 20 ms from BEFORE the warm-up; the timed region of a short run
    # (20 steps = 15 ms) is shorter than one sampling period, so the same step keeps running after it (untimed) until
    # the sampler has seen the GPU under this load for >= 0.6 s
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(W):
        one_step(False)
    barrier()
    launches0 = lib.cb200_launch_count()
    graph_launches0 = agent.graph_kernel_launches     # kernels run through CUDA-graph replays of the learn step
    # per-kernel-group device timing inside the timed region: events around the fused sample+gather launch
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True),
           torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    orig_sample = agent.sample_batch
    step_i = [0]

    def timed_sample():
        a, b, _ = ev[step_i[0]]
        mem.kernel_events = (a, b)        # recorded immediately around the fused sample+gather launch
        return orig_sample()

    agent.sample_batch = timed_sample
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    barrier()
    t0.record()
    for i in range(K):
        step_i[0] = i
        one_step(False)
        ev[i][2].record()
    if hasattr(agent, "_join_optimizer"):
        agent._join_optimizer()            # the last step's optimizer part (own stream) belongs to the timed region
    t1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(agent, args.dump_outputs)        # before any untimed step below changes the agent's state
    agent.sample_batch = orig_sample
    mem.kernel_events = None
    ms_total = t0.elapsed_time(t1)
    launches = lib.cb200_launch_count() - launches0 + agent.graph_kernel_launches - graph_launches0
    t_load = time.perf_counter()
    while time.perf_counter() - t_load < 0.6:         # same step, same load, untimed: lets the 20 ms sampler see it
        for _ in range(50):
            one_step(False)
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed region + 0.6 s of the same steps (nvidia-smi -lms 20)"
    gather_us = float(np.mean([a.elapsed_time(b) for a, b, _ in ev])) * 1e3
    learn_us = float(np.mean([b.elapsed_time(c) for _, b, c in ev])) * 1e3
    ms_total = parallel.max_over_ranks(ms_total, device)

    # ---- per-launch timing of the dominant kernel family (the tiled tcgen05 GEMMs): one traced step lists the
    # launches, then every distinct prepared call is timed with CUDA events on the launching stream over 10
    # back-to-back launches (the step itself has host-side bubbles between some launches, which per-launch events
    # inside the step would count as kernel time).  Operands are in the L2 state the step leaves them in.
    from coach_b200.architectures.tiled import TGemmOp
    gemm_ops = {}
    if not args.no_tc:
        TGemmOp.trace = []
        graph_mode, agent.use_graph = agent.use_graph, False     # the trace needs the eager launch path
        one_step(False)                                # every rank: the step contains the gradient all-reduce
        agent.use_graph = graph_mode
        torch.cuda.synchronize()
        trace, TGemmOp.trace = TGemmOp.trace, None
        if rank != 0:
            trace = []
        for op, _, _ in trace:
            rec = gemm_ops.setdefault(id(op), {"op": op, "tag": op.tag, "macs": op.macs, "nprod": op.nprod, "n": 0})
            rec["n"] += 1
        for rec in gemm_ops.values():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for _ in range(2):
                rec["op"].run()
            a.record()
            for _ in range(10):
                rec["op"].run()
            b.record()
            torch.cuda.synchronize()
            rec["us"] = a.elapsed_time(b) * 1e2          # ms / 10 launches -> us
    barrier()

    # ---- end-to-end leg through the public API with host buffers ---------------------------------------------------
    rng = np.random.RandomState(7 + rank)
    Ke = max(5, K // 2)
    dedup = bool(mem.ring.stack_cols)
    # frame-deduplicated replay: the states are LazyStacks of one continuing episode (a fresh frame per transition)
    pool = host_transitions(rng, ENV_STEPS_PER_TRAIN * (Ke + 3) if dedup else 64, stacked_by_filter=dedup)
    if dedup:
        pool_iter = iter(pool)
        pool_at = lambda i: [next(pool_iter) for _ in range(ENV_STEPS_PER_TRAIN)]                  # noqa: E731
    else:
        pool_at = lambda i: pool[(4 * i) % 60:(4 * i) % 60 + ENV_STEPS_PER_TRAIN]                  # noqa: E731
    for i in range(3):
        for t in pool_at(i):
            mem.store(t)
        one_step(True)
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(Ke):
        for t in pool_at(i):
            mem.store(t)                              # host transition -> pinned staging -> H2D -> ring + tree
        loss = one_step(True)                         # reads the loss back (D2H) every step
    e1.record()
    barrier()
    e2e_ms = parallel.max_over_ranks(e0.elapsed_time(e1), device)
    # per stored transition: both stacked states (verbatim ring) or ONE new 84x84 frame + two int32[4] slot rows
    per_t = (ROW // 4 + 2 * 16 + 8 + 8 + 1) if dedup else (2 * ROW + 8 + 8 + 1)
    h2d = ENV_STEPS_PER_TRAIN * per_t + BATCH * 8 + 2 * BATCH * 8
    d2h = BATCH * 8 + 4 + 4

    if rank != 0:
        return
    pk, pk_kind = peaks()
    steps_per_s = world * K / (ms_total * 1e-3)
    gather_gbs = GATHER_BYTES / gather_us / 1e3
    moved = GATHER_BYTES if agent.s2d is None else (GATHER_DEDUP_MOVED if mem.ring.stack_cols else GATHER_S2D_MOVED)
    gemm_tflops = 2.0 * MACS_PER_SAMPLE * BATCH / (learn_us * 1e-6) / 1e12
    # dominant kernel family: every launch of gemm_tc_tiled_kernel in one step.  "achieved" counts the bf16
    # tensor-core FLOPs actually ISSUED (6 products per fp32 multiply-accumulate, 3 for the exact uint8 operand): that
    # is what the tensor pipe executes; the useful fp32-equivalent rate is reported next to it.
    ops = []
    for rec in gemm_ops.values():
        us = rec["us"]
        ops.append({"op": rec["tag"], "us": round(us, 1), "launches_per_step": rec["n"],
                    "issued_tflops": round(2.0 * rec["macs"] * rec["nprod"] / us / 1e6, 1),
                    "fp32_equiv_tflops": round(2.0 * rec["macs"] / us / 1e6, 1)})
    tl_us = sum(o["us"] * o["launches_per_step"] for o in ops)
    tl_issued = sum(2.0 * r["macs"] * r["nprod"] * r["n"] for r in gemm_ops.values())
    tl_useful = sum(2.0 * r["macs"] * r["n"] for r in gemm_ops.values())
    tiled_tflops = tl_issued / tl_us / 1e6 if tl_us else 0.0
    line = {
        "metric": "learn_from_batch steps/sec (DQN PER batch 512)", "value": round(steps_per_s, 2),
        "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": round(ms_total / K, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "Atari-shaped DQN + PrioritizedExperienceReplay: %d-slot ring (%.1f GB HBM) and "
                               "2^%d-leaf fp64 trees per GPU, 84x84x4 uint8, batch 512 per GPU, Huber, Adam"
                               % (mem.ring.capacity, mem.ring.hbm_bytes() / 1e9,
                                  int(np.log2(mem.power_of_2_size))),
                   "parallelism": "dp%d (one replay shard per GPU, flat fp32 gradient all-reduce over NCCL)" % world,
                   "l2": "inputs (ring) >> L2, no flush needed", "priority_mode": mem.priority_mode,
                   "frame_dedup": bool(mem.ring.stack_cols),
                   "cuda_graph": bool(agent.use_graph),
                   "l2_persist_tree_top": not args.no_l2_persist},
        "clocks": clocks,
        "e2e": {"value": round(world * Ke / (e2e_ms * 1e-3), 2), "unit": "steps/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": Ke,
                "what": "per step: 4 host Transitions store()d + train(fetch=True) reading the loss back"},
        "gpu_launches": int(launches),
        "roofline": {"kernel": "gemm_tc_tiled_kernel (multi-tap tcgen05 GEMM on TMA-fed bf16 planes; all %d launches of a "
                               "step, conv / dense forward, data and weight gradients)" % sum(
                                   o["launches_per_step"] for o in ops),
                     "bound": "tensor", "achieved": round(tiled_tflops, 1), "peak": pk["bf16_tflops_sustained"],
                     "unit": "TFLOP/s", "frac": round(tiled_tflops / pk["bf16_tflops_sustained"], 4),
                     "frac_algorithmic": round(tl_useful / tl_us / 1e6 / pk["bf16_tflops_sustained"], 4) if tl_us else 0.0,
                     "peak_kind": pk_kind + " (sustained dense bf16, kernel timed inside the step)",
                     "us_per_step": round(tl_us, 1), "share_of_step": round(tl_us / (ms_total / K * 1e3), 3),
                     "share_of_step_note": "sum of the launches' stand-alone durations / step time; inside the step "
                                           "the target forward, the weight gradients and the optimizer run on side "
                                           "streams beside the main chain, so the launches overlap.  Serialised "
                                           "(profiles/launches_r2k_one_step.txt, ncu, one launch at a time, cold "
                                           "caches): the same launches incl. their split-reduce passes are 545 of "
                                           "680 us = 0.80 of the step",
                     "frac_over_whole_step": round(tl_issued / (ms_total / K * 1e-3) / 1e12
                                                   / pk["bf16_tflops_sustained"], 4),
                     "issued_flops_per_step": tl_issued, "algorithmic_flops_per_step": tl_useful, "fp32_equivalent_tflops": round(tl_useful / tl_us / 1e6, 1)
                     if tl_us else 0.0,
                     "what": "achieved = bf16 tensor-core FLOPs issued (3xBF16 split: 6 products per fp32 MAC, 3 for "
                             "the exact uint8 operand) / CUDA-event time of the launches (each prepared call timed over "
                             "10 back-to-back launches incl. its split-reduce pass, weighted by launches per step)",
                     "traffic": TRAFFIC_NCU.get("gemm_tc_tiled"),
                     "traffic_note": "dram bytes summed over the launches of one step, from the committed ncu --set full "
                                     "capture under profiles/ (cold caches), not this run", "ops": ops},
        "roofline_gather": {"kernel": ("sample_gather_s2d_kernel (fused sum-tree descent + IS weights + TMA bulk-copy gather + "
                                       "uint8 -> bf16 space-to-depth operand plane of conv1: replaces the staged uint8 "
                                       "copy and the two conversion passes over it)") if agent.s2d is not None else
                            "per_sample_gather_kernel (fused sum-tree descent + IS weights + TMA bulk-copy gather)",
                     "bound": "hbm", "achieved": round(gather_gbs, 1), "peak": pk["hbm_gbs"], "unit": "GB/s",
                     "frac": round(gather_gbs / pk["hbm_gbs"], 4), "peak_kind": pk_kind + " (burst copy)",
                     "us_per_launch": round(gather_us, 2), "algorithmic_bytes": GATHER_BYTES,
                     "algorithmic_bytes_note": "the 57.9 MB contract figure of SURVEY 8d (columns read + staged copy "
                                               "written)" + ("; this kernel reads 28.9 MB of frames and writes 57.8 MB "
                                               "of bf16 planes: bytes_moved" if agent.s2d is not None else "") +
                                              ("; frame-deduplicated replay: 18.1 MB of distinct frames read"
                                               if mem.ring.stack_cols else ""),
                     "bytes_moved": moved,
                     "frac_bytes_moved": round(moved / gather_us / 1e3 / pk["hbm_gbs"], 4),
                     "traffic": TRAFFIC_NCU.get("sample_gather_s2d" if agent.s2d is not None else "per_sample_gather"),
                     "traffic_note": "dram bytes from the committed ncu --set full capture under profiles/, not this run",
                     "frac_of_8TBps": round(gather_gbs / 8000.0, 4)},
        "roofline_learn": {"kernels": ("fp32 FFMA gather-GEMMs" if args.no_tc else
                                       "tcgen05 gather-GEMMs (3xBF16 split, 6 MMAs per product, fp32 TMEM accumulators)")
                           + " (conv/dense fwd+bwd) + element-wise",
                           "bound": "tensor", "achieved": round(gemm_tflops, 2), "peak": pk["bf16_tflops_sustained"],
                           "unit": "TFLOP/s", "frac": round(gemm_tflops / pk["bf16_tflops_sustained"], 5),
                           "us_per_step": round(learn_us, 1),
                           "note": "achieved = fp32-equivalent FLOPs of the step / time; the 3xBF16 split issues 6x "
                                   "as many tensor-core MACs" if not args.no_tc else
                                   "fp32 CUDA-core path; nominal fp32 FFMA peak ~72 TFLOP/s"},
        "share_of_step": {"sample_gather": round(gather_us / (gather_us + learn_us), 4),
                          "learn": round(learn_us / (gather_us + learn_us), 4)},
    }
    if world == 1:          # the CPU baseline is reported by the single-GPU run only
        line["cpu_baseline"] = cpu_reference(steps=args.cpu_steps, warmup=1, quiet=True)
    print(json.dumps(line))
    sys.stdout.flush()


# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture (profiles/)
# (gemm_tc_tiled: sum over the 15 launches of one step, profiles/ncu_tiled_gemm_r1p_summary.txt -- cold caches under ncu)
# dram__bytes_read.sum + dram__bytes_write.sum per launch (per step for the GEMM family: 16 launches), cold caches:
# profiles/ncu_step_r2f_summary.txt (sample_gather_s2d: 30.4 MB read + 4.9 MB written -- the bf16 planes stay in L2),
# profiles/ncu_tiled_r2f_summary.txt, profiles/ncu_per_sample_gather_r1b_summary.txt
TRAFFIC_NCU = {"per_sample_gather": 30270000, "sample_gather_s2d": 35286016, "gemm_tc_tiled": 473743616}


# =====================================================================================================================
def cpu_reference(steps, warmup, quiet=False):
    """The reference's CPU path for the same step, as the oracle port: per-sample Python loops for the PER (that is how
    the reference runs: one interpreter thread), numpy AoS->SoA Batch gather, torch-CPU fp32 network on all host
    cores.  Bounded sample of the workload: full 2^20-leaf trees, but only 2^13 distinct transitions of frame data
    (leaf -> transition modulo 2^13) so that the host-RAM footprint stays at 0.5 GB."""
    import torch
    from oracle import memory as om
    from oracle import nets as on
    cores = os.cpu_count() or 1
    rng = np.random.RandomState(0)
    size, distinct = 1 << 20, 1 << 13

    class T(object):
        __slots__ = ("state", "next_state", "action", "reward", "game_over", "info")

    data = []
    for i in range(distinct):
        t = T()
        t.state = {"observation": rng.randint(0, 256, OBS).astype(np.uint8)}
        t.next_state = {"observation": rng.randint(0, 256, OBS).astype(np.uint8)}
        t.action = int(rng.randint(0, N_ACTIONS))
        t.reward = float(rng.randint(-1, 2))
        t.game_over = False
        t.info = {}
        data.append(t)
    mem = om.OraclePrioritizedExperienceReplay(size, alpha=0.6, beta=om.OracleLinearSchedule(0.4, 1, 12500000),
                                               backend="c")
    mem.store_many([None] * size)
    mem.update_priorities(np.arange(size), np.abs(rng.randn(size)))
    for tr in (mem.sum_tree, mem.min_tree, mem.max_tree):
        tr.backend = "python"
    mem.backend = "python"
    net = on.QNetOracle(OBS, N_ACTIONS, False, torch.float32)
    from collections import OrderedDict
    g = torch.Generator().manual_seed(0)
    shapes = [(8, 8, 4, 32), (32,), (4, 4, 32, 64), (64,), (3, 3, 64, 64), (64,), (3136, 512), (512,),
              (512, N_ACTIONS), (N_ACTIONS,)]
    online = OrderedDict(("p%d" % i, torch.randn(s, generator=g) * 0.05) for i, s in enumerate(shapes))
    target = OrderedDict((k, v.clone()) for k, v in online.items())
    opt = on.AdamTF(list(online.values()), 2.5e-4, 0.9, 0.99, 1e-4)
    random.seed(0)
    # "all the host threads it can use": pick the thread count at which the network step is fastest on this host
    xs = rng.randint(0, 256, (BATCH,) + OBS).astype(np.uint8)
    probe = dict(states=xs, next_states=xs, actions=rng.randint(0, N_ACTIONS, BATCH), rewards=np.zeros(BATCH),
                 game_overs=np.zeros(BATCH, bool), weights=None)
    best = None
    for nthreads in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16)}, reverse=True):
        torch.set_num_threads(nthreads)
        popt = on.AdamTF(list(online.values()), 2.5e-4, 0.9, 0.99, 1e-4)
        on.dqn_learn_step(net, online, target, popt, probe, 0.99, True)
        t = time.perf_counter()
        on.dqn_learn_step(net, online, target, popt, probe, 0.99, True)
        dt = time.perf_counter() - t
        if best is None or dt < best[0]:
            best = (dt, nthreads)
    cores_used = best[1]
    torch.set_num_threads(cores_used)

    def step():
        nonlocal online
        idx, w = mem.sample_indices(BATCH)                                   # PER.sample
        batch = [data[i % distinct] for i in idx]
        s, s2, a, r, d = om.batch_columns(batch)                             # Batch AoS -> SoA
        out = on.dqn_learn_step(net, online, target, opt, dict(states=s, next_states=s2, actions=a, rewards=r,
                                                               game_overs=d, weights=w), 0.99, True)
        mem.update_priorities(list(idx), list(out["td_errors"]))             # PER.update_priorities
        online = out["new_params"]

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return {"value": round(steps / dt, 3), "unit": "steps/s", "cores": cores_used, "host_cores": cores,
            "kind": "port",
            "sample": "%d steps of the same B=512 step: full 2^20-leaf trees, 2^13 distinct Atari-shaped transitions; "
                      "PER/Batch in one Python thread (as the reference runs), torch-CPU fp32 network on %d threads "
                      "(fastest of the tried thread counts on this host)" % (steps, cores_used)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    K, W = args.steps, args.warmup
    W = max(3, min(W, 10))              # same warm-up as the device arm (bounded: a CPU step is ~0.2 s)
    base = cpu_reference(steps=K, warmup=W)
    line = {"impl": "reference", "metric": "learn_from_batch steps/sec (DQN PER batch 512)", "value": base["value"],
            "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(1e3 / base["value"], 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "Atari-shaped DQN + PrioritizedExperienceReplay, 2^20-leaf trees, batch 512 "
                                   "(CPU, oracle port of the reference path; one process)"},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def _finish():
    """Orderly end of a multi-rank run: CUDA graphs that captured NCCL kernels are destroyed BEFORE the communicator
    (the other order can block in the communicator's teardown), and a teardown that still does not return within 20 s
    ends the process instead of holding the launcher."""
    import gc
    import threading
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return
    gc.collect()
    torch.cuda.synchronize()
    sys.stdout.flush()
    t = threading.Thread(target=dist.destroy_process_group, daemon=True)
    t.start()
    t.join(20.0)
    if t.is_alive():
        sys.stderr.write("bench: process-group teardown did not return in 20 s, exiting\n")
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--capacity", type=int, default=1000000, help="replay capacity in transitions (rounded up to 2^k)")
    ap.add_argument("--cpu-steps", type=int, default=6, help="steps of the cpu_baseline leg")
    ap.add_argument("--no-l2-persist", action="store_true")
    ap.add_argument("--frame-dedup", type=int, default=0, choices=[0, 1],
                    help="1: frame-deduplicated replay -- every 84x84 frame stored once (9.3 GB instead of 59.2 GB for "
                         "2^20 transitions, 41 KB instead of 238 KB over PCIe per step), stacks assembled by the "
                         "gather (measured 3 %% slower per step: profiles/README.md); 0 (default): stacked states "
                         "verbatim")
    ap.add_argument("--no-tc", action="store_true", help="fp32 FFMA GEMMs instead of the tcgen05 3xBF16 path")
    ap.add_argument("--config", default="dqn", choices=["dqn", "dueling", "cartpole", "ppo", "sac", "td3"],
                    help="dqn: BASELINE config 2 (Atari DQN + PER, the headline metric, default); dueling: config 5 "
                         "(dueling DDQN + PER, no middleware, clip-norm 10); cartpole / ppo / sac / td3: configs 1, 3, 4 "
                         "(bench_configs.py)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (loss, sampled batch, TD errors, priorities, network "
                         "parameters) to DIR/<name>.npy; dqn / dueling configurations of this repo's CUDA path")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config not in ("dqn", "dueling")):
        ap.error("--dump-outputs covers the dqn and dueling configurations of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    elif args.config in ("cartpole", "ppo", "sac", "td3"):
        import bench_configs
        bench_configs.run(args, ClockSampler)
        _finish()
    else:
        run_device(args)
        _finish()


if __name__ == "__main__":
    main()
