"""TEST / BASELINE INFRASTRUCTURE -- drives the UNMODIFIED reference (ratinabox v1.15.3) the way its users do:
one Agent per Python object, `Ag.update(); Ns.update()` in a Python loop (tests/test_advanced.py:17-23 of the reference).
Used by bench.py's CPU legs (`--impl reference`, `cpu_baseline`) and oracle/gen_golden.py config1; never by the product."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import ref_shim  # noqa: E402


def available():
    return ref_shim.reference_root() is not None


def build(walls, populations, pos=None, vel=None, dt=0.01, seed=0, env_params=None):
    """populations: list of (kind, params dict, attrs dict) with kind in place / grid / bvc; attrs are assigned after
    construction (the reference's documented way of setting vector-cell tunings, Neurons.py:1612).
    Returns (ratinabox module, Environment, Agent, [Neurons])."""
    rb = ref_shim.import_reference()
    if rb is None:
        raise RuntimeError("reference not available: run oracle/make_ref.py in the build container")
    import warnings
    np.random.seed(seed)
    rb.verbose = False
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from ratinabox.Environment import Environment
        from ratinabox.Agent import Agent
        from ratinabox.Neurons import PlaceCells, GridCells, BoundaryVectorCells
        Env = Environment(dict(env_params or {}))
        for w in walls:
            Env.add_wall(np.array(w, dtype=float))
        Ag = Agent(Env, {"dt": dt})
        if pos is not None:
            Ag.pos = np.array(pos, dtype=float)
        if vel is not None:
            Ag.velocity = np.array(vel, dtype=float)
            Ag.measured_velocity = np.array(vel, dtype=float)
        cls = {"place": PlaceCells, "grid": GridCells, "bvc": BoundaryVectorCells}
        pops = []
        import io
        import contextlib
        for kind, params, attrs in populations:
            with contextlib.redirect_stdout(io.StringIO()):           # the reference prints its soft fall-backs
                ns = cls[kind](Ag, dict(params))
            for k, v in (attrs or {}).items():
                setattr(ns, k, v)
            pops.append(ns)
    return rb, Env, Ag, pops


def step(Ag, pops, n):
    for _ in range(n):
        Ag.update()
        for ns in pops:
            ns.update()
