"""The plug points of INTEGRATION.md checked against the UNMODIFIED reference.  What the reference's code says about
them -- constructor arguments and method signatures of its memories, the memory calls of its priority-update gate, the
path strings its loader resolves, its parameter defaults, its checkpoint-state reader and writer -- is stored in
tests/golden/boundary.json (oracle/make_golden_boundary.py).  CPU only: nothing here launches a kernel -- the device
classes are resolved and type-checked, not run."""
import importlib
import inspect
import json
import os

import pytest


@pytest.fixture
def ref(golden_dir):
    with open(os.path.join(golden_dir, "boundary.json")) as f:
        return json.load(f)


def _args(fn):
    return [a for a in inspect.getfullargspec(fn).args if a not in ("self", "lock")]


def test_bound_per_passes_the_reference_isinstance_gate_and_loader(ref):
    """INTEGRATION.md 'isinstance gates': a class derived from the device PER and the reference PER (device class first
    in the MRO) satisfies ``isinstance(self.memory, PrioritizedExperienceReplay)``
    (agents/value_optimization_agent.py:77) and is resolved by the reference's own
    dynamic_import_and_instantiate_module_from_params (utils.py:389-404) from a Parameters.path string."""
    from coach_b200.memories import prioritized_experience_replay as dev
    from coach_b200.utils import short_dynamic_import
    rper = ref["memories"]["PrioritizedExperienceReplay"]
    # MRO: every public method the reference agents call is defined by the device class (or its own bases), so it
    # comes first in a class derived from (device PER, reference PER)
    for name in ("store", "sample", "update_priorities", "num_transitions", "clean", "freeze", "get_transition"):
        assert name in rper["methods"], name
        owner = next(c for c in dev.PrioritizedExperienceReplay.__mro__ if name in c.__dict__)
        assert owner.__module__.startswith("coach_b200"), (name, owner)
    # the gate of value_optimization_agent.py:77 on a PER memory: one call_memory('update_priorities', (idx, errors))
    # and the batch's 'weight' info as the importance weights
    gate = ref["priority_gate"]
    assert gate["calls"] == [["update_priorities", 2]] and gate["weights_from_info"] == "weight"
    assert len(_args(dev.PrioritizedExperienceReplay.update_priorities)) >= 2
    # the reference loader resolves 'module.path:Class' strings and passes the constructor arguments
    params = dev.PrioritizedExperienceReplayParameters()
    rpath = ref["loader_paths"]["PrioritizedExperienceReplayParameters"]
    assert rpath["path"].count(":") == 1 and params.path.count(":") == 1 and "/" not in params.path
    cls = short_dynamic_import(params.path)
    assert cls is dev.PrioritizedExperienceReplay and cls.__name__ == rpath["resolves_to"]
    ctor = set(inspect.getfullargspec(cls).args)
    assert set(rper["ctor_args"]) <= ctor, "device PER must accept every constructor argument of the reference PER"
    passed = {k for k in params.__dict__ if k in ctor}
    assert set(rpath["passed"]) <= passed
    assert {"max_size", "alpha", "beta", "epsilon", "allow_duplicates_in_batch_sampling"} <= passed


@pytest.mark.parametrize("dev_path,ref_path,cls_name", [
    ("coach_b200.memories.experience_replay", "rl_coach.memories.non_episodic.experience_replay", "ExperienceReplay"),
    ("coach_b200.memories.prioritized_experience_replay", "rl_coach.memories.non_episodic.prioritized_experience_replay",
     "PrioritizedExperienceReplay"),
    ("coach_b200.memories.episodic_experience_replay", "rl_coach.memories.episodic.episodic_experience_replay",
     "EpisodicExperienceReplay"),
])
def test_memory_method_surface_covers_the_reference(dev_path, ref_path, cls_name, ref):
    """every public method of the reference memory that the replay -> learn path calls exists on the device class with
    the same leading arguments"""
    dcls = getattr(importlib.import_module(dev_path), cls_name)
    assert ref["memories"][cls_name]["module"] == ref_path
    methods = ref["memories"][cls_name]["methods"]
    assert methods
    for name, ra in sorted(methods.items()):
        assert hasattr(dcls, name), "%s.%s missing" % (cls_name, name)
        da = _args(getattr(dcls, name))
        assert da[:len(ra)] == ra or name in ("sample",), (cls_name, name, ra, da)


def test_parameter_defaults_match_the_reference(ref):
    """the Parameters classes carry the reference's defaults for every field they define (agents' algorithm / network
    parameters, memory parameters)"""
    from coach_b200.agents.categorical_dqn_agent import CategoricalDQNAgentParameters
    from coach_b200.agents.dqn_agent import DQNAgentParameters, DDQNAgentParameters
    from coach_b200.agents.clipped_ppo_agent import ClippedPPOAgentParameters
    from coach_b200.agents.ddpg_agent import DDPGAgentParameters, TD3AgentParameters
    from coach_b200.agents.soft_actor_critic_agent import SoftActorCriticAgentParameters

    def same(a, b):
        """a: our value; b: the reference's, as stored by oracle/make_golden_boundary.py"""
        if hasattr(a, "num_steps"):
            return type(a).__name__ == b["type"] and a.num_steps == b.get("num_steps")
        if hasattr(a, "current_value"):
            return float(a.current_value) == b.get("current_value")
        if "name" in b and isinstance(a, str):             # enums of the reference are plain strings here
            return a == b["name"]
        if isinstance(a, tuple):
            return "tuple" in b and list(a) == b["tuple"]
        if isinstance(a, (int, float, str, bool, type(None))):
            return "value" in b and a == b["value"]
        return True                                   # structured values (filters, lists of layer objects): not compared

    own_only = {"hidden_units", "truncate_dataset_to_playing_steps", "middleware_parameters", "heads_parameters"}
    defaults = ref["parameter_defaults"]
    mines = (DQNAgentParameters(), DDQNAgentParameters(), ClippedPPOAgentParameters(), DDPGAgentParameters(),
             TD3AgentParameters(), SoftActorCriticAgentParameters(), CategoricalDQNAgentParameters())
    assert sorted(type(m).__name__ for m in mines) == sorted(defaults)
    for mine in mines:
        rd = defaults[type(mine).__name__]
        for k, v in vars(mine.algorithm).items():
            if k in own_only or k not in rd["algorithm"]:
                continue
            assert same(v, rd["algorithm"][k]), (type(mine).__name__, "algorithm", k, v, rd["algorithm"][k])
        for net in mine.network_wrappers:
            for k, v in vars(mine.network_wrappers[net]).items():
                if k in own_only or k not in rd["network_wrappers"][net]:
                    continue
                rv = rd["network_wrappers"][net][k]
                assert same(v, rv), (type(mine).__name__, net, k, v, rv)
        assert type(mine.memory).__name__ == rd["memory"], type(mine).__name__


def test_presets_define_the_five_baseline_configurations():
    """coach_b200/presets/*: agent parameters whose path strings resolve to the device classes"""
    from coach_b200.utils import short_dynamic_import
    for name in ("CartPole_DQN", "Atari_DQN_with_PER", "Atari_Dueling_DDQN_with_PER_OpenAI", "Mujoco_ClippedPPO",
                 "Mujoco_SAC", "Mujoco_TD3", "Atari_C51"):
        mod = importlib.import_module("coach_b200.presets." + name)
        ap = mod.agent_params
        assert short_dynamic_import(ap.path).__module__.startswith("coach_b200.agents")
        assert short_dynamic_import(ap.memory.path).__module__.startswith("coach_b200.memories")
    from coach_b200.presets import Atari_Dueling_DDQN_with_PER_OpenAI as p5
    from coach_b200.architectures.q_network import QNetworkDef
    from coach_b200.base_parameters import MiddlewareScheme
    net = p5.agent_params.network_wrappers["main"]
    qn = QNetworkDef("cpu", p5.observation_shape, p5.num_actions, dueling="DuelingQHead" in net.heads_parameters,
                     middleware_units=MiddlewareScheme.units[net.middleware_parameters.scheme])
    assert qn.store.num_params() - 1 == 3293863          # SURVEY section 8d, config 5 (+1: the rescaler scalar)


def test_checkpoint_names_and_state_file_interoperate_with_the_reference(tmp_path, ref):
    """coach_b200/checkpoint.py follows the reference's on-disk conventions (checkpoint.py:115-155, :247-273,
    graph_manager.py:630): the reference's CheckpointStateFile / CheckpointFilenameParser read what we write -- number
    and name -- and we read what the reference writes; a half-written or foreign state file is ignored by both."""
    from coach_b200 import checkpoint as ck
    rck = ref["checkpoint_state"]
    parse = {p["content"]: p for p in rck["parse"]}
    d = str(tmp_path)
    name = ck.checkpoint_name(7, 123456)
    assert name == "7_Step-123456.ckpt"                                   # '{}_Step-{}.ckpt' of graph_manager.py:630
    assert parse[name]["filename_parser"] == [7, name]
    assert rck["state_file"] == ck.STATE_FILE
    ck._write_state_file(d, name)
    assert os.listdir(d) == [ck.STATE_FILE]
    with open(os.path.join(d, ck.STATE_FILE)) as f:
        content = f.read()
    # the reference reads this state file as checkpoint 7 (CheckpointStateFile and CheckpointStateReader alike), and
    # writes the same bytes for that checkpoint
    assert parse[content]["state_file_read"] == [7, name] and parse[content]["latest"] == [7, name]
    assert [w["content"] for w in rck["written"] if w["num"] == 7] == [content]
    # the other direction
    for w in rck["written"]:
        with open(os.path.join(d, ck.STATE_FILE), "w") as f:
            f.write(w["content"])
        assert ck.read_state_file(d) == w["name"]
        assert w["files"] == [ck.STATE_FILE]
    assert ck.read_state_file(d) == "12_Step-99.ckpt" == ck.checkpoint_name(12, 99)
    # garbage in the state file: no checkpoint for either reader
    with open(str(tmp_path / ck.STATE_FILE), "w") as f:
        f.write("not a checkpoint")
    assert ck.read_state_file(d) is None
    assert parse["not a checkpoint"]["state_file_read"] is None
