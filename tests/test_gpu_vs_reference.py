"""The CUDA path against the unmodified reference (RatInABox v1.15.3) -- no oracle restatement in between.  BASELINE.json
configs[0]: 1 agent, default box, 100 Gaussian PlaceCells, dt = 10 ms.  Teacher-forced like the oracle's mode A: the
reference's geometry jitter is zeroed and its `scale == dt` normals are taped, every step starts from the reference's state.
The reference's 300 steps are stored in tests/golden/config1.npz (oracle/gen_golden.py config1).  GPU only."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

STATE = ("pos", "velocity", "rotational_velocity", "measured_velocity", "head_direction", "distance_travelled")


@pytest.mark.parametrize("walls", [[], [[[0.3, 0.0], [0.3, 0.5]], [[0.7, 1.0], [0.7, 0.5]]]])
def test_config1_against_the_live_reference(golden, walls):
    import ratinabox_b200 as rb
    g = golden("config1.npz")
    name = "box2" if walls else "open"
    assert np.array_equal(g[f"{name}_walls"], np.array(walls, dtype=float).reshape(-1, 2, 2))
    centres, xi, ref_rates = g[f"{name}_centres"], g[f"{name}_xi"], g[f"{name}_rates"]
    ref_state = {k: g[f"{name}_{k}"] for k in STATE}
    steps, N = len(xi), len(centres)
    assert steps == 300 and N == 100
    geom = "line_of_sight" if walls else "euclidean"
    np.random.seed(5)
    E = rb.Environment()
    for w in walls:
        E.add_wall(w)
    Ag = rb.Agent(E, {"dt": 0.01})
    PCs = rb.PlaceCells(Ag, {"n": N, "place_cell_centres": centres, "widths": 0.2, "wall_geometry": geom})
    worst_p = worst_r = 0.0
    for s in range(steps):
        for k in STATE:                                        # teacher forcing: start from the reference's state
            setattr(Ag, k, np.array(ref_state[k][s], dtype=float))
        Ag.update(_xi=xi[s])                                   # the reference's two OU draws of this step
        PCs.update()
        worst_p = max(worst_p, float(np.abs(np.asarray(Ag.pos) - ref_state["pos"][s + 1]).max()))
        worst_r = max(worst_r, float(np.abs(np.asarray(PCs.firingrate) - ref_rates[s]).max()))
    assert worst_p <= 1e-6, worst_p                            # north_star: positions <= 1e-6 m
    assert worst_r <= 1e-5, worst_r                            # rates <= 1e-5 of the rate scale (max_fr = 1)
