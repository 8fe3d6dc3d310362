"""Generates the fixtures of tests/test_boundary.py and tests/test_acting.py by running the UNMODIFIED reference
(imported through oracle/ref_loader.py):

* tests/golden/boundary.json -- the reference's plug points as plain data: constructor arguments and method
  signatures of its replay memories, the memory calls of its priority-update gate, the path strings its loader
  resolves, the defaults of its agent / network / memory parameters, and what its checkpoint-state reader and writer
  make of a set of state-file contents.
* tests/golden/e_greedy.npz -- actions of one reference EGreedy per environment (numpy's global generator, agent
  order) on a fixed stream of Q values, in the train and the test phase.

    python -m oracle.make_golden_boundary

TEST INFRASTRUCTURE ONLY.
"""
import inspect
import json
import os
import sys
import tempfile
from types import SimpleNamespace

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

MEMORIES = {
    "ExperienceReplay": "rl_coach.memories.non_episodic.experience_replay",
    "PrioritizedExperienceReplay": "rl_coach.memories.non_episodic.prioritized_experience_replay",
    "EpisodicExperienceReplay": "rl_coach.memories.episodic.episodic_experience_replay",
}
# every public memory method the replay -> learn path of the reference agents calls
USED_METHODS = ["store", "sample", "num_transitions", "length", "clean", "freeze", "assert_not_frozen", "get_transition",
                "get", "remove_transition", "update_priorities", "store_episode", "num_complete_episodes",
                "num_transitions_in_complete_episodes", "verify_last_episode_is_closed", "mean_reward", "save",
                "load_pickled", "get_shuffled_training_data_generator"]
# state-file contents put to the reference's checkpoint reader
STATE_FILE_CONTENTS = ["7_Step-123456.ckpt", "12_Step-99.ckpt", "not a checkpoint"]
E_GREEDY = dict(envs=5, actions=6, steps=40, seed=11, start=1.0, end=0.1, decay_steps=25, evaluation_epsilon=0.05)


def _ref():
    from oracle import ref_loader
    ref_loader.load()


def _args(fn):
    return [a for a in inspect.getfullargspec(fn).args if a not in ("self", "lock")]


def _value(v):
    """a reference parameter value as the fields tests/test_boundary.py compares"""
    out = {"type": type(v).__name__}
    if hasattr(v, "num_steps"):
        out["num_steps"] = v.num_steps
    if hasattr(v, "current_value"):
        out["current_value"] = float(v.current_value)
    if hasattr(v, "name") and isinstance(getattr(v, "name"), str):
        out["name"] = v.name
    if isinstance(v, tuple):
        out["tuple"] = list(v)
    elif isinstance(v, (int, float, str, bool, type(None))):
        out["value"] = v
    return out


def memories():
    import importlib
    out = {}
    for cls_name, path in MEMORIES.items():
        cls = getattr(importlib.import_module(path), cls_name)
        out[cls_name] = {"module": path, "ctor_args": _args(cls),
                         "methods": {name: _args(fn) for name, fn in inspect.getmembers(cls, inspect.isfunction)
                                     if name in USED_METHODS}}
    return out


def priority_gate():
    """the memory calls of ValueOptimizationAgent.update_transition_priorities_and_get_weights on a PER memory"""
    from rl_coach.agents.value_optimization_agent import ValueOptimizationAgent
    from rl_coach.memories.non_episodic.prioritized_experience_replay import PrioritizedExperienceReplay
    calls = []
    fake = SimpleNamespace(memory=PrioritizedExperienceReplay.__new__(PrioritizedExperienceReplay),
                           call_memory=lambda f, a: calls.append([f, len(a)]))
    batch = SimpleNamespace(info=lambda k: k)
    w = ValueOptimizationAgent.update_transition_priorities_and_get_weights(fake, [0.1, 0.2, 0.3], batch)
    return {"calls": calls, "weights_from_info": w}


def loader_paths():
    from rl_coach.memories.non_episodic.experience_replay import ExperienceReplayParameters
    from rl_coach.memories.non_episodic.prioritized_experience_replay import PrioritizedExperienceReplayParameters
    from rl_coach.memories.episodic.episodic_experience_replay import EpisodicExperienceReplayParameters
    from rl_coach.utils import short_dynamic_import
    out = {}
    for p in (ExperienceReplayParameters(), PrioritizedExperienceReplayParameters(),
              EpisodicExperienceReplayParameters()):
        out[type(p).__name__] = {"path": p.path, "resolves_to": short_dynamic_import(p.path).__name__,
                                 "passed": sorted(k for k in vars(p) if k in _args(short_dynamic_import(p.path)))}
    return out


def parameter_defaults():
    from rl_coach.agents.dqn_agent import DQNAgentParameters as RDQN
    from rl_coach.agents.ddqn_agent import DDQNAgentParameters as RDDQN
    from rl_coach.agents.clipped_ppo_agent import ClippedPPOAgentParameters as RPPO
    from rl_coach.agents.ddpg_agent import DDPGAgentParameters as RDDPG
    from rl_coach.agents.td3_agent import TD3AgentParameters as RTD3
    from rl_coach.agents.soft_actor_critic_agent import SoftActorCriticAgentParameters as RSAC
    from rl_coach.agents.categorical_dqn_agent import CategoricalDQNAgentParameters as RC51
    out = {}
    for ref in (RDQN(), RDDQN(), RPPO(), RDDPG(), RTD3(), RSAC(), RC51()):
        out[type(ref).__name__] = {
            "algorithm": {k: _value(v) for k, v in vars(ref.algorithm).items()},
            "network_wrappers": {net: {k: _value(v) for k, v in vars(ref.network_wrappers[net]).items()}
                                 for net in ref.network_wrappers},
            "memory": type(ref.memory).__name__}
    return out


def checkpoint_state():
    from rl_coach.checkpoint import (CheckpointFilenameParser, CheckpointStateFile, CheckpointStateReader,
                                     SingleCheckpoint)

    def ckpt(c):
        return None if c is None else [c.num, c.name]

    out = {"state_file": CheckpointStateFile.checkpoint_state_filename, "parse": [], "written": []}
    for content in STATE_FILE_CONTENTS:
        with tempfile.TemporaryDirectory() as d:
            with open(os.path.join(d, CheckpointStateFile.checkpoint_state_filename), "w") as f:
                f.write(content)
            latest = CheckpointStateReader(d, checkpoint_state_optional=False).get_latest()
            out["parse"].append({"content": content, "filename_parser": ckpt(CheckpointFilenameParser().parse(content)),
                                 "state_file_read": ckpt(CheckpointStateFile(d).read()), "latest": ckpt(latest)})
    for num, name in ((7, "7_Step-123456.ckpt"), (12, "12_Step-99.ckpt")):
        with tempfile.TemporaryDirectory() as d:
            CheckpointStateFile(d).write(SingleCheckpoint(num, name))
            files = sorted(os.listdir(d))
            with open(os.path.join(d, CheckpointStateFile.checkpoint_state_filename)) as f:
                out["written"].append({"num": num, "name": name, "files": files, "content": f.read()})
    return out


def e_greedy():
    from rl_coach.core_types import RunPhase
    from rl_coach.exploration_policies.e_greedy import EGreedy
    from rl_coach.schedules import LinearSchedule
    from rl_coach.spaces import DiscreteActionSpace
    g = E_GREEDY
    E, A, T = g["envs"], g["actions"], g["steps"]
    rng = np.random.RandomState(0)
    q = rng.randn(T, E, A).astype(np.float32)
    q[3, 1, 2] = q[3, 1, 4] = q[3, 1].max() + 1.0            # exact ties: random tie-break consumes the stream
    q[7, 0] = 0.5
    out = dict(q=q, **{k: np.array(v) for k, v in g.items()})
    for tag, phase in (("train", RunPhase.TRAIN), ("test", RunPhase.TEST)):
        np.random.seed(g["seed"])
        refs = [EGreedy(DiscreteActionSpace(A), LinearSchedule(g["start"], g["end"], g["decay_steps"]),
                        g["evaluation_epsilon"]) for _ in range(E)]
        for p in refs:
            p.change_phase(phase)
        actions = np.zeros((T, E), dtype=np.int64)
        for t in range(T):
            for e in range(E):
                actions[t, e], _ = refs[e].get_action(q[t, e])
        out["actions_" + tag] = actions
        out["epsilon_" + tag] = np.float64(refs[0].epsilon_schedule.current_value)
    return out


def main():
    _ref()
    os.makedirs(OUT, exist_ok=True)
    data = {"memories": memories(), "priority_gate": priority_gate(), "loader_paths": loader_paths(),
            "parameter_defaults": parameter_defaults(), "checkpoint_state": checkpoint_state()}
    with open(os.path.join(OUT, "boundary.json"), "w") as f:
        json.dump(data, f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(os.path.join(OUT, "e_greedy.npz"), **e_greedy())
    print("boundary.json, e_greedy.npz ok")


if __name__ == "__main__":
    main()
