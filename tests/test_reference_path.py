"""mission.reference_path against a direct restatement: segment boundaries, zero-length segments,
holding at the end, one polyline or one per drone."""
import numpy as np
import pytest

from dart_planner_b200.mission import reference_path


def direct(w, speed, dt, T):
    """Sample by sample: walk the segments until the arc length falls inside one."""
    P, V = np.zeros((T, 3)), np.zeros((T, 3))
    seg = [np.sqrt(((w[i + 1] - w[i]) ** 2).sum()) for i in range(len(w) - 1)]
    L = float(np.sum(seg)) if seg else 0.0
    for j in range(T):
        s = (speed * j) * dt
        if s >= L:
            P[j] = w[-1]
            continue
        acc = 0.0
        for i, li in enumerate(seg):
            if acc <= s < acc + li:
                P[j] = w[i] + ((s - acc) / li) * (w[i + 1] - w[i])
                V[j] = (speed / li) * (w[i + 1] - w[i])
                break
            acc += li
    return P, V


def test_boundaries_zero_segments_and_the_end():
    # legs of 1 m and 2 m with a zero-length segment between; 0.25 m per sample hits every boundary
    w = np.array([[0.0, 0.0, 1.0], [1.0, 0.0, 1.0], [1.0, 0.0, 1.0], [1.0, 2.0, 1.0]])
    P, V = reference_path(w, 1.0, 0.25, 16)
    assert P.shape == V.shape == (1, 16, 3)
    assert (P[0, 4] == [1.0, 0.0, 1.0]).all() and (V[0, 4] == [0.0, 1.0, 0.0]).all()   # the next leg's velocity
    assert (V[0, :4] == [1.0, 0.0, 0.0]).all()
    assert (P[0, 12:] == w[-1]).all() and (V[0, 12:] == 0).all() and not np.signbit(V[0, 12:]).any()  # +0
    Pd, Vd = direct(w, 1.0, 0.25, 16)
    assert P[0].tobytes() == Pd.tobytes() and V[0].tobytes() == Vd.tobytes()


@pytest.mark.parametrize("seed", range(4))
def test_matches_the_restatement(seed):
    rng = np.random.default_rng(seed)
    B, W, T = 16, 6, 80
    w = rng.uniform(-5, 5, (B, W, 3))
    w[:, 3] = w[:, 2]                                     # a zero-length segment in every polyline
    w[0, 1:] = w[0, 0]                                    # a polyline of length 0: held from the start
    speed, dt = rng.uniform(0.5, 3), rng.choice([0.05, 0.1])
    P, V = reference_path(w, speed, dt, T)
    for b in range(B):
        Pd, Vd = direct(w[b], speed, dt, T)
        assert P[b].tobytes() == Pd.tobytes() and V[b].tobytes() == Vd.tobytes(), b
    assert (P[0] == w[0, 0]).all() and (V[0] == 0).all()
    # one polyline for every drone = (1, T, 3)
    P1, V1 = reference_path(w[3], speed, dt, T)
    assert P1.tobytes() == P[3:4].tobytes() and V1.tobytes() == V[3:4].tobytes()


def test_refusals():
    with pytest.raises(ValueError):
        reference_path(np.zeros((3, 2)), 1.0, 0.1, 4)
    with pytest.raises(ValueError):
        reference_path(np.zeros((3, 3)), 0.0, 0.1, 4)
    with pytest.raises(ValueError):
        reference_path(np.zeros((3, 3)), 1.0, 0.1, 0)
