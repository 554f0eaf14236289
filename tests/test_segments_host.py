"""Host-side rules of a trajectory run in epoch segments (eskf_run_epochs): the epoch range check and the first step of
every trajectory's segment, which the kernels count as the running sum of n_prop with every epoch clamped to what is left of
the stream (epoch_steps3)."""
import numpy as np
import pytest

from dvi_ekf_b200.engine import check_run_geometry, segment_steps


def _epoch_steps_loop(n_prop, T):
    """the kernels' count, one epoch at a time: k(e) for e = 0 .. E, every epoch clamped to [0, T - k]"""
    k, out = 0, [0]
    for n in n_prop:
        k += int(min(max(n, 0), T - k))
        out.append(k)
    return np.array(out)


@pytest.mark.parametrize("seed", range(6))
def test_segment_steps_against_the_clamped_loop(seed):
    rng = np.random.default_rng(seed)
    n_traj, E, T = 5, 40, 120
    npr = rng.integers(-3, 9, (n_traj, E)).astype(np.int32)
    npr[1] = 0  # a trajectory that never moves
    npr[2, :10] = 20  # one that exhausts the stream early (device-resident streams are not validated)
    ks = np.array([_epoch_steps_loop(r, T) for r in npr])
    for e0 in range(E + 1):
        for e1 in (e0, min(E, e0 + 1), min(E, e0 + 7), E):
            k0, k1 = segment_steps(npr, T, e0, e1)
            assert np.array_equal(k0, ks[:, e0]) and np.array_equal(k1, ks[:, e1])
    k0, k1 = segment_steps(npr[0], T, 3, 9)  # one trajectory, [E]
    assert k0.shape == (1,) and k1[0] == ks[0, 9]


def test_stacked_trajectories_start_at_their_own_steps():
    npr = np.array([[10, 10, 10], [3, 0, 1], [0, 0, 5]], np.int32)
    k0, k1 = segment_steps(npr, 30, 1, 3)
    assert k0.tolist() == [10, 3, 0] and k1.tolist() == [30, 4, 5]


@pytest.mark.parametrize("epochs", [(-1, 2), (3, 2), (0, 8), (8, 8)])
def test_bad_epoch_ranges_are_refused(epochs):
    with pytest.raises(ValueError, match="epoch range"):
        check_run_geometry(52, 4, 13, 0, 70, 7, epochs=epochs)


@pytest.mark.parametrize("epochs", [(0, 0), (0, 7), (3, 3), (2, 5), (7, 7), None])
def test_good_epoch_ranges_pass(epochs):
    check_run_geometry(52, 4, 13, 0, 70, 7, np.full((4, 7), 10, np.int32), epochs=epochs)
