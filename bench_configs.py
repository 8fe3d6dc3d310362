"""bench.py --config {cartpole,ppo,sac,td3}: the other BASELINE.json configurations, same JSON contract as the default
(config 2) line -- device-timed `value`, `e2e` through the public API with host buffers, kernel launches per step,
`cpu_baseline` (the oracle port of the reference path timed on the host cores, bounded sample).

  cartpole  config 1: CartPole_DQN, 10,000-transition uniform ExperienceReplay, batch 32, net 4-256-512-2, MSE
  ppo       config 3: Hopper-shaped ClippedPPO, 64 envs x 2048 steps rollout (17-dim obs, 6-dim actions), GAE 0.95,
                      10 epochs x minibatch 64 over the WHOLE rollout (the reference's [:2048] truncation, SURVEY Q8,
                      is switched off: truncate_dataset_to_playing_steps = False); a "step" = one training phase
  sac, td3  config 4: HalfCheetah-shaped (17 / 6), 1M-transition replay shard per GPU, batch 256; under torchrun every
                      rank owns a shard and the gradients are all-reduced over NCCL (parallel.allreduce_gradients)

These steps are launch / latency bound (0.4 MFLOP per sample): the line reports us per step and kernels per step next
to steps/s, as SURVEY section 8(d) asks.
"""
import json
import os
import random
import sys
import time

import numpy as np


def _clock_and_sync(torch, parallel, world):
    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
    return barrier


def _timed(torch, parallel, device, world, K, W, step, barrier, lib, sampler_cls, local, rank):
    sampler = sampler_cls(local)
    if rank == 0:
        sampler.start()
    for _ in range(W):
        step()
    barrier()
    l0 = lib.cb200_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(K):
        step()
    t1.record()
    barrier()
    ms = parallel.max_over_ranks(t0.elapsed_time(t1), device)
    launches = lib.cb200_launch_count() - l0
    t_load = time.perf_counter()
    while time.perf_counter() - t_load < 0.6:
        step()
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "warm-up + timed region + 0.6 s of the same steps (nvidia-smi -lms 20)"
    return ms, launches, clocks


def _line(metric, value, unit, world, K, W, ms, workload, clocks, launches, e2e, extra, cpu):
    line = {"metric": metric, "value": round(value, 3), "unit": unit, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(ms / K, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "parallelism": "dp%d (one replay / rollout shard per GPU, flat fp32 "
                                                            "gradient all-reduce over NCCL)" % world,
                       "l2": "latency-bound step: working set (parameters + one minibatch) is L2 resident by design; "
                             "the replay rows are drawn at random from a buffer >> L2 where the config has one"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches)}
    line.update(extra)
    if cpu is not None:
        line["cpu_baseline"] = cpu
    return line


# =====================================================================================================================
def run(args, sampler_cls):
    import torch
    from coach_b200 import _lib, parallel
    rank, world = parallel.init_from_env()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    lib = _lib.load()
    random.seed(1000 + rank)
    np.random.seed(1000 + rank)
    K, W = args.steps, max(args.warmup, 3)
    barrier = _clock_and_sync(torch, parallel, world)
    fn = {"cartpole": _cartpole, "ppo": _ppo, "sac": _sac, "td3": _td3}[args.config]
    line = fn(args, torch, parallel, lib, device, rank, world, local, K, W, barrier, sampler_cls)
    if rank == 0:
        print(json.dumps(line))
        sys.stdout.flush()


# ---- config 1 -----------------------------------------------------------------------------------------------------------
def _cartpole(args, torch, parallel, lib, device, rank, world, local, K, W, barrier, sampler_cls):
    from coach_b200.agents.dqn_agent import DQNAgent
    from coach_b200.core_types import Transition
    from coach_b200.memories.memory import MemoryGranularity
    from coach_b200.presets import CartPole_DQN as preset
    import copy
    ap = copy.deepcopy(preset.agent_params)
    ap.memory.max_size = (MemoryGranularity.Transitions, 10000)          # BASELINE.json config 1
    agent = DQNAgent(ap, observation_shape=(4,), num_actions=2, device=device, seed=100 + rank)
    rng = np.random.RandomState(100 + rank)
    n = 10000
    agent.memory.store_columns({"state:observation": rng.uniform(-1, 1, (n, 4)).astype(np.float32),
                                "next_state:observation": rng.uniform(-1, 1, (n, 4)).astype(np.float32),
                                "action": rng.randint(0, 2, n).astype(np.int64),
                                "reward": np.ones(n), "game_over": (rng.rand(n) < 0.02).astype(np.uint8)})

    def step(fetch=False):
        agent.total_steps_counter += 1
        return agent.train(fetch=fetch)
    ms, launches, clocks = _timed(torch, parallel, device, world, K, W, step, barrier, lib, sampler_cls, local, rank)
    # end to end: one host transition stored per step (num_consecutive_playing_steps = 1), loss read back
    pool = [Transition(state={"observation": rng.uniform(-1, 1, 4).astype(np.float32)}, action=int(rng.randint(0, 2)),
                       reward=1.0, next_state={"observation": rng.uniform(-1, 1, 4).astype(np.float32)},
                       game_over=False) for _ in range(64)]
    Ke = max(10, K)
    for i in range(5):
        agent.memory.store(pool[i])
        step(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(Ke):
        agent.memory.store(pool[i % 64])
        step(True)
    e1.record()
    barrier()
    e_ms = parallel.max_over_ranks(e0.elapsed_time(e1), device)
    cpu = _cpu_cartpole() if (rank == 0 and world == 1) else None
    e2e = {"value": round(world * Ke / (e_ms * 1e-3), 2), "unit": "steps/s", "h2d_bytes_per_step": 2 * 16 + 17 + 32 * 8,
           "d2h_bytes_per_step": 8, "steps": Ke,
           "what": "per step: 1 host Transition store()d + train(fetch=True) reading the loss back"}
    return _line("learn_from_batch steps/sec (CartPole DQN, uniform replay 10k, batch 32)", world * K / (ms * 1e-3),
                 "steps/s", world, K, W, ms, "CartPole-shaped DQN: 4-dim fp32 observations, 2 actions, 10,000-slot uniform "
                 "ExperienceReplay, batch 32, MSE head, Adam, net 4-256-512-2 (CUDA-core gather-GEMMs: batch < 128)",
                 clocks, launches, e2e, {"us_per_step": round(ms / K * 1e3, 2),
                                         "kernels_per_step": round(launches / K, 1)}, cpu)


def _cpu_cartpole(steps=200):
    import torch
    from collections import OrderedDict
    from oracle import memory as om
    from oracle import nets as on
    rng = np.random.RandomState(0)

    class T(object):
        __slots__ = ("state", "next_state", "action", "reward", "game_over", "info")
    mem = om.OracleExperienceReplay(10000, True)
    for i in range(10000):
        t = T()
        t.state = {"observation": rng.uniform(-1, 1, 4).astype(np.float32)}
        t.next_state = {"observation": rng.uniform(-1, 1, 4).astype(np.float32)}
        t.action, t.reward, t.game_over, t.info = int(rng.randint(0, 2)), 1.0, False, {}
        mem.store(t)
    net = on.QNetOracle((4,), 2, False, torch.float32)
    g = torch.Generator().manual_seed(0)
    shapes = [(4, 256), (256,), (256, 512), (512,), (512, 2), (2,)]
    online = OrderedDict(("p%d" % i, torch.randn(s, generator=g) * 0.05) for i, s in enumerate(shapes))
    target = OrderedDict((k, v.clone()) for k, v in online.items())
    opt = on.AdamTF(list(online.values()), 2.5e-4, 0.9, 0.99, 1e-4)
    torch.set_num_threads(1)                 # B = 32: one thread is the fastest setting for this size

    def step():
        nonlocal online
        batch = mem.sample(32)
        s, s2, a, r, d = om.batch_columns(batch)
        out = on.dqn_learn_step(net, online, target, opt, dict(states=s, next_states=s2, actions=a, rewards=r,
                                                               game_overs=d, weights=None), 0.99, False)
        online = out["new_params"]
    for _ in range(10):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return {"value": round(steps / dt, 2), "unit": "steps/s", "cores": 1, "host_cores": os.cpu_count(), "kind": "port",
            "sample": "%d steps of the same B=32 step: uniform replay of 10,000 Python transitions, numpy Batch gather, "
                      "torch-CPU fp32 network on 1 thread" % steps}


# ---- config 3 -----------------------------------------------------------------------------------------------------------
def _ppo(args, torch, parallel, lib, device, rank, world, local, K, W, barrier, sampler_cls):
    from coach_b200.agents.clipped_ppo_agent import ClippedPPOAgent
    from coach_b200.memories.memory import MemoryGranularity
    from coach_b200.presets import Mujoco_ClippedPPO as preset
    import copy
    ENVS, T, D, A = 64, 2048, preset.observation_dim, preset.action_dim
    n = ENVS * T
    ap = copy.deepcopy(preset.agent_params)
    ap.memory.max_size = (MemoryGranularity.Transitions, n)
    ap.algorithm.truncate_dataset_to_playing_steps = False
    agent = ClippedPPOAgent(ap, observation_dim=D, action_dim=A, device=device, seed=100 + rank)
    rng = np.random.RandomState(100 + rank)
    cols = {"state:observation": rng.randn(n, D).astype(np.float32), "next_state:observation":
            rng.randn(n, D).astype(np.float32), "action": rng.randn(n, A).astype(np.float32), "reward": rng.randn(n)}
    done = (rng.rand(n) < 1.0 / 500).astype(np.uint8)
    done[T - 1::T] = 1                                                     # forced at the end of every env's rollout
    cols["game_over"] = done
    W = min(W, 2)                              # a phase is 20,480 minibatch steps: seconds, not milliseconds
    phase_ms = []

    def step():
        agent.memory.store_columns(cols)                                   # the rollout of this phase (H2D inside e2e)
        agent.total_steps_counter += T
        agent.train()
    ms, launches, clocks = _timed(torch, parallel, device, world, K, W, step, barrier, lib, sampler_cls, local, rank)
    mb_steps = (n // agent.B) * ap.algorithm.optimization_epochs
    cpu = _cpu_ppo(D, A) if (rank == 0 and world == 1) else None
    h2d = sum(v.nbytes for v in cols.values())
    e2e = {"value": round(world * K / (ms * 1e-3), 4), "unit": "phases/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": 8, "steps": K,
           "what": "the timed step already is end to end: the 131,072-transition host rollout is store_columns()d (H2D) "
                   "inside the timed region, then Agent.train() runs filter + fill_advantages + 10 epochs"}
    return _line("ClippedPPO training phases/sec (64 envs x 2048 steps, GAE 0.95, 10 epochs x minibatch 64)",
                 world * K / (ms * 1e-3), "phases/s", world, K, W, ms,
                 "Hopper-shaped ClippedPPO: 17-dim fp32 observations, 6-dim actions, 64 x 2048 rollout per GPU, observation "
                 "normalisation (running stats), GAE scan, 10 epochs x 2048 minibatches of 64 (CUDA-graph replay of the "
                 "minibatch step)", clocks, launches, e2e,
                 {"minibatch_steps_per_phase": mb_steps, "us_per_minibatch_step": round(ms / K * 1e3 / mb_steps, 2),
                  "minibatch_steps_per_s": round(world * K * mb_steps / (ms * 1e-3), 1)}, cpu)


def _cpu_ppo(D, A, steps=300):
    import torch
    from oracle import actor_critic as oac
    from oracle import rl_math as orm
    rng = np.random.RandomState(0)
    n = 64 * 2048
    r, v = rng.randn(n), rng.randn(n).astype(np.float32)
    done = (rng.rand(n) < 1.0 / 500)
    done[2047::2048] = True
    t0 = time.perf_counter()
    orm.ppo_fill_advantages(r, v, done, 0.99, 0.95)
    gae_s = time.perf_counter() - t0
    shapes = [(D, 64), (64,), (64, 64), (64,), (64, 1), (1,), (), (D, 64), (64,), (64, 64), (64,), (64, A), (A,), (A,), ()]
    named = {"p%d" % i: (rng.randn(*s) * 0.1).astype(np.float32) if len(s) else np.float32(1.0) for i, s in
             enumerate(shapes)}
    torch.set_num_threads(1)
    try:
        opt = oac.make_adam(named, 3e-4, 0.9, 0.999, 1e-5)
        mb = dict(states=rng.randn(64, D).astype(np.float32), actions=rng.randn(64, A).astype(np.float32),
                  advantages=rng.randn(64).astype(np.float32), value_targets=rng.randn(64).astype(np.float32))
        cur = named
        for _ in range(5):
            oac.ppo_minibatch_step(cur, named, opt, mb, 0.2, 0.0)
        t0 = time.perf_counter()
        for _ in range(steps):
            oac.ppo_minibatch_step(cur, named, opt, mb, 0.2, 0.0)
        per = (time.perf_counter() - t0) / steps
    except Exception as exc:                 # the oracle's parameter naming is its own: report the GAE part at least
        return {"value": None, "unit": "phases/s", "cores": 1, "kind": "port", "sample": "oracle step failed: %r" % exc}
    phase = gae_s + per * 20480
    return {"value": round(1.0 / phase, 5), "unit": "phases/s", "cores": 1, "host_cores": os.cpu_count(), "kind": "port",
            "sample": "GAE / fill_advantages of the full 131,072-transition rollout (%.2f s) + %d timed minibatch steps of "
                      "the torch-CPU fp32 oracle (%.0f us each) extrapolated to the 20,480 of a phase" %
                      (gae_s, steps, per * 1e6)}


# ---- config 4 -----------------------------------------------------------------------------------------------------------
def _fill_continuous(agent, rng, n, D, A, episodic):
    chunk = 1 << 16
    for lo in range(0, n, chunk):
        m = min(chunk, n - lo)
        cols = {"state:observation": rng.randn(m, D).astype(np.float32),
                "next_state:observation": rng.randn(m, D).astype(np.float32),
                "action": rng.uniform(-1, 1, (m, A)).astype(np.float32), "reward": rng.randn(m)}
        done = np.zeros(m, np.uint8)
        done[999::1000] = 1
        cols["game_over"] = done
        agent.memory.store_columns(cols)


def _offpolicy(kind, args, torch, parallel, lib, device, rank, world, local, K, W, barrier, sampler_cls):
    import copy
    from coach_b200.core_types import Transition
    from coach_b200.memories.memory import MemoryGranularity
    D, A, B, N = 17, 6, 256, 1 << 20
    if kind == "sac":
        from coach_b200.agents.soft_actor_critic_agent import SoftActorCriticAgent as cls
        from coach_b200.presets import Mujoco_SAC as preset
    else:
        from coach_b200.agents.ddpg_agent import TD3Agent as cls
        from coach_b200.presets import Mujoco_TD3 as preset
    ap = copy.deepcopy(preset.agent_params)
    ap.memory.max_size = (MemoryGranularity.Transitions, N)
    for nw in ap.network_wrappers.values():
        nw.batch_size = B
    kw = dict(observation_dim=D, action_dim=A, device=device, seed=100 + rank)
    agent = cls(ap, **kw)
    rng = np.random.RandomState(100 + rank)
    _fill_continuous(agent, rng, N, D, A, kind != "sac")
    torch.cuda.synchronize()

    def step(fetch=False):
        agent.total_steps_counter += 1
        return agent.train(fetch=fetch)
    ms, launches, clocks = _timed(torch, parallel, device, world, K, W, step, barrier, lib, sampler_cls, local, rank)
    pool = [Transition(state={"observation": rng.randn(D).astype(np.float32)},
                       action=rng.uniform(-1, 1, A).astype(np.float32), reward=float(rng.randn()),
                       next_state={"observation": rng.randn(D).astype(np.float32)}, game_over=False)
            for _ in range(64)]
    Ke = max(10, K)
    for i in range(5):
        agent.memory.store(pool[i])
        step(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(Ke):
        agent.memory.store(pool[i % 64])                                  # one environment step per train step
        step(True)
    e1.record()
    barrier()
    e_ms = parallel.max_over_ranks(e0.elapsed_time(e1), device)
    cpu = _cpu_offpolicy(kind, D, A, B) if (rank == 0 and world == 1) else None
    e2e = {"value": round(world * Ke / (e_ms * 1e-3), 2), "unit": "steps/s",
           "h2d_bytes_per_step": 2 * D * 4 + A * 4 + 9 + B * 8, "d2h_bytes_per_step": 8, "steps": Ke,
           "what": "per step: 1 host Transition store()d + train(fetch=True) reading the critic loss back"}
    name = {"sac": "SoftActorCritic", "td3": "TD3"}[kind]
    return _line("learn_from_batch steps/sec (%s, 1M replay, batch 256)" % name, world * K / (ms * 1e-3), "steps/s",
                 world, K, W, ms, "HalfCheetah-shaped %s: 17-dim fp32 observations, 6-dim actions, 2^20-transition replay "
                 "shard per GPU, batch 256 per GPU, Adam; %s" % (name, "policy / twin-Q / V networks (289,039 parameters)"
                                                             if kind == "sac" else
                                                             "actor + twin critic (389,708 parameters), delayed actor "
                                                             "update every 2nd step"),
                 clocks, launches, e2e, {"us_per_step": round(ms / K * 1e3, 2),
                                         "kernels_per_step": round(launches / K, 1)}, cpu)


def _sac(*a):
    return _offpolicy("sac", *a)


def _td3(*a):
    return _offpolicy("td3", *a)


def _cpu_offpolicy(kind, D, A, B, steps=100):
    import torch
    from collections import OrderedDict
    from oracle import actor_critic as oac
    rng = np.random.RandomState(0)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    batch = dict(states=rng.randn(B, D).astype(np.float32), next_states=rng.randn(B, D).astype(np.float32),
                 actions=rng.uniform(-1, 1, (B, A)).astype(np.float32), rewards=rng.randn(B),
                 game_overs=np.zeros(B, bool))

    def params(shapes):
        return OrderedDict(("p%d" % i, (rng.randn(*s) * 0.05).astype(np.float32) if len(s) else np.float32(1.0))
                           for i, s in enumerate(shapes))
    try:
        if kind == "td3":
            actor = params([(D, 400), (400,), (400, 300), (300,), (300, A), (A,), ()])
            critic = params([(A + D, 400), (400,), (400, 300), (300,), (A + D, 400), (400,), (400, 300), (300,),
                             (300, 1), (1,), (300, 1), (1,), ()])
            oa, oc = oac.make_adam(actor, 1e-3, 0.9, 0.999, 1e-8), oac.make_adam(critic, 1e-3, 0.9, 0.999, 1e-8)
            noise = rng.normal(0, 0.2, (B, A))

            def step():
                oac.ddpg_td3_step(actor, actor, critic, critic, oa, oc, batch, twin=True, noise=noise)
        else:
            from oracle import sac as osac
            pol = params([(D, 256), (256,), (256, 256), (256,), (256, 2 * A), (2 * A,), ()])
            q = params([(D, 256), (256,), (A, 256), (256,), (256, 256), (256,), (256, 1), (1,)] * 2 + [()])
            v = params([(D, 256), (256,), (256, 256), (256,), (256, 1), (1,), ()])
            o = [oac.make_adam(x, 3e-4, 0.9, 0.99, 1e-4) for x in (pol, q, v)]
            noise = [rng.standard_normal((B, A)).astype(np.float32) for _ in range(3)]

            def step():
                osac.sac_step(pol, q, v, v, o[0], o[1], o[2], batch, noise)
        for _ in range(3):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = time.perf_counter() - t0
    except Exception as exc:
        return {"value": None, "unit": "steps/s", "cores": 1, "kind": "port", "sample": "oracle step failed: %r" % exc}
    return {"value": round(steps / dt, 2), "unit": "steps/s", "cores": torch.get_num_threads(),
            "host_cores": os.cpu_count(), "kind": "port",
            "sample": "%d learn steps of the torch-CPU fp32 oracle on one fixed minibatch of 256 (network arithmetic "
                      "only: the reference's replay sampling / Batch gather would add to it)" % steps}
