"""The batched epsilon-greedy of the device acting path against the UNMODIFIED reference policy objects (one EGreedy per
environment, all drawing from numpy's global generator in agent order).  CPU only.  The reference's actions are stored
in tests/golden/e_greedy.npz (oracle/make_golden_boundary.py)."""
import os

import numpy as np
import pytest


@pytest.mark.parametrize("test_phase", [False, True])
def test_batched_e_greedy_selects_the_reference_actions(test_phase, golden_dir):
    from coach_b200.exploration_policies.e_greedy import BatchedEGreedy, RunPhase
    from coach_b200.schedules import LinearSchedule
    fx = np.load(os.path.join(golden_dir, "e_greedy.npz"))
    q = fx["q"]
    T, E, A = q.shape
    tag = "test" if test_phase else "train"
    want = fx["actions_" + tag]
    np.random.seed(int(fx["seed"]))
    mine = BatchedEGreedy(A, E, LinearSchedule(float(fx["start"]), float(fx["end"]), int(fx["decay_steps"])),
                          float(fx["evaluation_epsilon"]))
    mine.change_phase(RunPhase.TEST if test_phase else RunPhase.TRAIN)
    got = np.zeros((T, E), dtype=np.int64)
    for t in range(T):
        got[t], probs = mine.get_actions(q[t])
        assert np.allclose(probs.sum(1), 1.0)
    np.testing.assert_array_equal(got, want)
    assert float(mine.epsilon_schedules[0].current_value) == float(fx["epsilon_" + tag])
