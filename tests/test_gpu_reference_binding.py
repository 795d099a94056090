"""INTEGRATION.md section 2 as a test: subclasses of the REFERENCE's own Agent / PlaceCells (examples/reference_binding.py)
whose update() / get_state() call the C ABI, run next to the unmodified classes on the same taped normals.  GPU only;
skipped when the reference is not importable (oracle/_ref not staged)."""
import contextlib
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import ref_driver  # noqa: E402


@contextlib.contextmanager
def taped_normals(tape, used):
    """np.random.normal as the reference calls it: jitter scales -> zeros, `scale == dt` draws -> popped from `tape`
    (standard normals; the reference scales them itself) and logged in `used`."""
    orig = np.random.normal

    def patched(loc=0.0, scale=1.0, size=None):
        if scale in (1e-9, 1e-6):
            return np.zeros(size)
        n = int(np.prod(size)) if size not in (None, ()) else 1
        vals = np.array([tape.pop(0) for _ in range(n)], dtype=float)
        used.extend(vals.tolist())
        out = loc + scale * vals
        return out.reshape(size) if size not in (None, ()) else float(out[0])

    np.random.normal = patched
    try:
        yield
    finally:
        np.random.normal = orig


@pytest.mark.skipif(not ref_driver.available(), reason="oracle/_ref not staged (python oracle/make_ref.py)")
def test_reference_classes_step_on_the_gpu_through_the_c_abi():
    import ref_shim
    ref_shim.import_reference()
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    import reference_binding as B
    from ratinabox.Environment import Environment
    from ratinabox.Agent import Agent
    from ratinabox.Neurons import PlaceCells
    walls = [[[0.3, 0.0], [0.3, 0.5]], [[0.7, 1.0], [0.7, 0.5]]]
    rs = np.random.RandomState(11)
    centres = rs.uniform(0.05, 0.95, (60, 2))
    pcs_params = {"n": 60, "place_cell_centres": centres, "widths": 0.2, "wall_geometry": "line_of_sight"}

    def make(agent_cls, cells_cls):
        import io, contextlib
        np.random.seed(2)
        Env = Environment()
        for w in walls:
            Env.add_wall(np.array(w))
        Ag = agent_cls(Env, {"dt": 0.01})
        Ag.pos, Ag.velocity = np.array([0.42, 0.31]), np.array([0.06, -0.04])
        Ag.measured_velocity = Ag.velocity.copy()
        with contextlib.redirect_stdout(io.StringIO()):
            return Ag, cells_cls(Ag, dict(pcs_params))

    RA, RP = make(Agent, PlaceCells)                      # the unmodified reference
    GA, GP = make(B.CudaAgent, B.CudaPlaceCells)          # its classes with the two methods bound to libriab_b200
    assert isinstance(GA, Agent) and isinstance(GP, PlaceCells)
    for s in range(200):
        tape, used = rs.normal(size=2 + 60).tolist(), []
        with taped_normals(tape, used):
            RA.update(); RP.update()
        with taped_normals([0.0] * 60, []):               # Neurons.update's (x 0) noise draw of the subclass
            GA.update(xi=np.array(used[:2])); GP.update()
        assert np.abs(GA.pos - RA.pos).max() <= 1e-9, s   # free-running: no teacher forcing
        assert np.abs(np.asarray(GP.firingrate) - np.asarray(RP.firingrate)).max() <= 1e-5
    assert len(GA.history["pos"]) == len(RA.history["pos"]) == 200
    assert np.abs(np.array(GA.history["pos"]) - np.array(RA.history["pos"])).max() <= 1e-9
    assert GP.get_state(evaluate_at="all").shape == RP.get_state(evaluate_at="all").shape
