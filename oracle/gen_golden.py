"""TEST INFRASTRUCTURE -- generate tests/golden/*.npz from the LIVE, unmodified
reference (/root/reference, imported through oracle/ref_shim.py).

Run in the build container only:   python oracle/gen_golden.py
The fixtures travel to the GPU box; /root/reference does not.

Fixtures
  native_c1.npz      config 1 (default box, 100 Gaussian PlaceCells, dt=10 ms), global
                     NumPy RNG, jitter on: RNG state after construction + full history.
  native_walls.npz   2x1 box with two internal walls, fast agent (bounces), line_of_sight
                     PlaceCells + GridCells + BVCs, global RNG, jitter on.
  modeA_motion.npz   teacher-forced single steps, zero jitter, injected normals
                     (SURVEY.md section 8c mode A): inputs, outputs, collision masks.
  modeA_rates.npz    get_state(evaluate_at=None, pos=P) for every cell type/variant,
                     zero jitter.
  host_mirror.npz    Environment / utils set-up helpers under fixed np.random seeds.
  config1.npz        config 1 teacher-forced for 300 steps, open box and box + 2 walls.
"""
import contextlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_shim  # noqa: E402

GOLD = os.path.join(os.path.dirname(HERE), "tests", "golden")

BOX_WALLS = [[[0.3, 0.0], [0.3, 0.5]], [[0.7, 1.0], [0.7, 0.5]]]          # SURVEY.md section 8(d), configs 2/5


def maze_walls(n=8, length=0.6):
    """SURVEY.md section 8(d) config 4: walls at x=k/9 alternately from floor / ceiling."""
    out = []
    for k in range(1, n + 1):
        x = k / (n + 1)
        out.append([[x, 0.0], [x, length]] if k % 2 else [[x, 1.0], [x, 1.0 - length]])
    return out


@contextlib.contextmanager
def mode_a(tape, used=None):
    """Zero the geometry jitter and feed ``scale == dt`` normals from ``tape``
    (a list that is popped from the front); the standard normals drawn are appended to ``used``."""
    orig = np.random.normal

    def patched(loc=0.0, scale=1.0, size=None):
        if scale in (1e-9, 1e-6):
            return np.zeros(size)
        n = int(np.prod(size)) if size not in (None, ()) else 1
        vals = np.array([tape.pop(0) if tape else 0.0 for _ in range(n)], dtype=float)
        if used is not None:
            used.extend(vals.tolist())
        out = loc + scale * vals
        return out.reshape(size) if size not in (None, ()) else float(out[0])

    np.random.normal = patched
    try:
        yield
    finally:
        np.random.normal = orig


def main():
    riab = ref_shim.import_reference()
    assert riab is not None, "reference not present"
    from ratinabox.Environment import Environment
    from ratinabox.Agent import Agent
    from ratinabox.Neurons import PlaceCells, GridCells, BoundaryVectorCells, FieldOfViewBVCs
    os.makedirs(GOLD, exist_ok=True)

    # ------------------------------------------------------------ native_c1
    np.random.seed(0)
    Env = Environment()
    Ag = Agent(Env, {"dt": 0.01})
    PCs = PlaceCells(Ag, {"n": 100})
    init = dict(pos0=Ag.pos.copy(), vel0=Ag.velocity.copy(), centres=PCs.place_cell_centres.copy(),
                widths=PCs.place_cell_widths.copy())
    st = np.random.get_state()
    for _ in range(600):
        Ag.update()
        PCs.update()
    np.savez_compressed(
        os.path.join(GOLD, "native_c1.npz"), rng_keys=st[1], rng_pos=st[2], rng_has_gauss=st[3],
        rng_cached=st[4], **init, pos=np.array(Ag.history["pos"]), vel=np.array(Ag.history["vel"]),
        rot_vel=np.array(Ag.history["rot_vel"]), head_direction=np.array(Ag.history["head_direction"]),
        distance_travelled=np.array(Ag.history["distance_travelled"]), t=np.array(Ag.history["t"]),
        firingrate=np.array(PCs.history["firingrate"]), spikes=np.packbits(np.array(PCs.history["spikes"])),
        wall_geometry=np.array(PCs.wall_geometry))

    # --------------------------------------------------------- native_walls
    np.random.seed(1)
    Env = Environment({"aspect": 2, "scale": 1})
    Env.add_wall([[1, 0], [1, 0.35]])
    Env.add_wall([[1, 0.65], [1, 1]])
    Ag = Agent(Env, {"dt": 0.05, "speed_mean": 0.4})
    Ag.pos = np.array([0.5, 0.5])
    PCs = PlaceCells(Ag, {"n": 20, "description": "gaussian_threshold", "widths": 0.40,
                          "wall_geometry": "line_of_sight", "max_fr": 10, "min_fr": 0.1})
    PCs.place_cell_centres[-1] = np.array([1.1, 0.5])
    GCs = GridCells(Ag, {"n": 12})
    BVCs = BoundaryVectorCells(Ag, {"n": 10})
    init = dict(pos0=Ag.pos.copy(), vel0=Ag.velocity.copy(), walls=Env.walls.copy(),
                centres=PCs.place_cell_centres.copy(), widths=PCs.place_cell_widths.copy(),
                gridscales=GCs.gridscales.copy(), phase_offsets=GCs.phase_offsets.copy(), gc_w=GCs.w.copy(),
                bvc_mu_d=BVCs.tuning_distances.copy(), bvc_mu_t=BVCs.tuning_angles.copy(),
                bvc_sg_d=BVCs.sigma_distances.copy(), bvc_sg_t=BVCs.sigma_angles.copy(),
                bvc_norm=BVCs.cell_fr_norm.copy(), bvc_test_angles=BVCs.test_angles.copy(),
                bvc_test_dirs=BVCs.test_directions.copy())
    st = np.random.get_state()
    ncoll = 0
    orig_check = Env.check_wall_collisions

    def counting_check(step):
        nonlocal ncoll
        r = orig_check(step)
        ncoll += int(True in r[1])
        return r

    Env.check_wall_collisions = counting_check
    for _ in range(1500):
        Ag.update()
        PCs.update()
        GCs.update()
        BVCs.update()
    print("native_walls: wall bounces =", ncoll)
    np.savez_compressed(
        os.path.join(GOLD, "native_walls.npz"), rng_keys=st[1], rng_pos=st[2], rng_has_gauss=st[3],
        rng_cached=st[4], **init, n_bounces=ncoll, pos=np.array(Ag.history["pos"]),
        vel=np.array(Ag.history["vel"]), rot_vel=np.array(Ag.history["rot_vel"]),
        head_direction=np.array(Ag.history["head_direction"]),
        distance_travelled=np.array(Ag.history["distance_travelled"]),
        pc_fr=np.array(PCs.history["firingrate"]), gc_fr=np.array(GCs.history["firingrate"]),
        bvc_fr=np.array(BVCs.history["firingrate"]))

    # --------------------------------------------------------- modeA_motion
    rs = np.random.RandomState(1234)
    for name, walls in (("box2", BOX_WALLS), ("maze8", maze_walls())):
        Env = Environment()
        for w in walls:
            Env.add_wall(w)
        Ag = Agent(Env, {"dt": 0.01})
        A = 768
        pos0 = rs.uniform(0.002, 0.998, size=(A, 2))
        # a third of the agents hug a wall so that repulsion / bounces are exercised
        near = rs.choice(A, A // 3, replace=False)
        wl = Env.walls[rs.randint(0, len(Env.walls), size=len(near))]
        lam = rs.uniform(0, 1, size=(len(near), 1))
        pos0[near] = np.clip(wl[:, 0] + lam * (wl[:, 1] - wl[:, 0]) + rs.normal(scale=2e-3, size=(len(near), 2)),
                             0.0005, 0.9995)
        speed = rs.rayleigh(0.08, size=A) * rs.choice([1.0, 1.0, 6.0], size=A)
        ang = rs.uniform(0, 2 * np.pi, size=A)
        vel0 = speed[:, None] * np.stack((np.cos(ang), np.sin(ang)), axis=1)
        rot0 = rs.normal(scale=2.0, size=A)
        mv0 = vel0 + rs.normal(scale=0.01, size=(A, 2))
        hd0 = mv0 / np.linalg.norm(mv0, axis=1, keepdims=True)
        dist0 = rs.uniform(0, 5, size=A)
        xi = rs.normal(size=(A, 2))
        drift = rs.normal(scale=0.1, size=(A, 2))
        use_drift = rs.uniform(size=A) < 0.25
        out = {k: [] for k in ("pos", "vel", "rot", "mv", "mrot", "hd", "dist", "dclose", "n_iter", "first_hit")}
        masks = np.zeros((A, 4, len(Env.walls)), dtype=bool)     # up to 4 loop iterations recorded
        recorded = []
        orig_check = Env.check_wall_collisions

        def rec_check(step, _o=orig_check):
            r = _o(step)
            recorded.append(np.array(r[1]).copy())
            return r

        Env.check_wall_collisions = rec_check
        for a in range(A):
            Ag.pos, Ag.velocity = pos0[a].copy(), vel0[a].copy()
            Ag.rotational_velocity = float(rot0[a])
            Ag.measured_velocity = mv0[a].copy()
            Ag.head_direction = hd0[a].copy()
            Ag.distance_travelled = float(dist0[a])
            Ag.t = 0.0
            recorded.clear()
            tape = list(xi[a])
            with mode_a(tape):
                if use_drift[a]:
                    Ag.update(drift_velocity=drift[a].copy(), drift_to_random_strength_ratio=2.0)
                else:
                    Ag.update()
            out["pos"].append(Ag.pos.copy()); out["vel"].append(Ag.velocity.copy())
            out["rot"].append(Ag.rotational_velocity); out["mv"].append(Ag.measured_velocity.copy())
            out["mrot"].append(Ag.measured_rotational_velocity); out["hd"].append(Ag.head_direction.copy())
            out["dist"].append(Ag.distance_travelled); out["dclose"].append(Ag.distance_to_closest_wall)
            out["n_iter"].append(len(recorded))
            fh = [int(np.argwhere(m)[0][0]) for m in recorded if m.any()]
            out["first_hit"].append((fh + [-1, -1, -1, -1])[:4])
            for i, m in enumerate(recorded[:4]):
                masks[a, i] = m
        print(f"modeA_motion[{name}]: agents with a bounce = {int((np.array(out['n_iter']) > 1).sum())} / {A}")
        np.savez_compressed(
            os.path.join(GOLD, f"modeA_motion_{name}.npz"), walls=Env.walls, dt=0.01, pos0=pos0, vel0=vel0,
            rot0=rot0, mv0=mv0, hd0=hd0, dist0=dist0, xi=xi, drift=drift, use_drift=use_drift,
            drift_ratio=2.0, masks=np.packbits(masks), masks_shape=np.array(masks.shape),
            **{"out_" + k: np.array(v) for k, v in out.items()})

    # ---------------------------------------------------------- modeA_rates
    rs = np.random.RandomState(4321)
    P = rs.uniform(0.001, 0.999, size=(384, 2))[:160]       # the first 160 of 384 draws keep the fixture under 1 MB
    res = {"P": P}
    with mode_a([]):
        Env = Environment()
        for w in BOX_WALLS:
            Env.add_wall(w)
        Ag = Agent(Env, {"dt": 0.01})
        np.random.seed(7)
        for desc in ("gaussian", "gaussian_threshold", "diff_of_gaussians", "top_hat", "one_hot"):
            for geom in ("euclidean", "line_of_sight"):
                pc = PlaceCells(Ag, {"n": 96, "description": desc, "wall_geometry": geom, "widths": 0.2,
                                     "min_fr": 0.05, "max_fr": 3.0})
                res[f"pc_{desc}_{geom}"] = pc.get_state(evaluate_at=None, pos=P)
                res[f"pc_{desc}_{geom}_centres"] = pc.place_cell_centres.copy()
        # geodesic needs exactly one internal wall
        Env1 = Environment()
        Env1.add_wall([[0.5, 0.0], [0.5, 0.6]])
        Ag1 = Agent(Env1, {"dt": 0.01})
        pc = PlaceCells(Ag1, {"n": 64, "wall_geometry": "geodesic", "widths": 0.15})
        res["pc_gaussian_geodesic"] = pc.get_state(evaluate_at=None, pos=P)
        res["pc_gaussian_geodesic_centres"] = pc.place_cell_centres.copy()
        res["geodesic_walls"] = Env1.walls.copy()
        for desc in ("rectified_cosines", "shifted_cosines"):
            gs = np.random.uniform(0.2, 1.0, size=80)
            th = np.random.uniform(0, np.pi / 3, size=80)
            ph = np.random.uniform(0, 2 * np.pi, size=(80, 2))
            gc = GridCells(Ag, {"gridscale": gs, "orientation": th, "phase_offset": ph, "description": desc,
                                "min_fr": 0.1, "max_fr": 2.0})
            res[f"gc_{desc}"] = gc.get_state(evaluate_at=None, pos=P)
            res[f"gc_{desc}_gridscales"], res[f"gc_{desc}_orient"], res[f"gc_{desc}_phase"] = gs, th, ph
            res[f"gc_{desc}_w"] = gc.w.copy()
        for name, walls in (("box2", BOX_WALLS), ("maze8", maze_walls())):
            E = Environment()
            for w in walls:
                E.add_wall(w)
            AgE = Agent(E, {"dt": 0.01})
            bvc = BoundaryVectorCells(AgE, {"n": 48, "min_fr": 0.0, "max_fr": 5.0})
            res[f"bvc_{name}"] = bvc.get_state(evaluate_at=None, pos=P)
            res[f"bvc_{name}_walls"] = E.walls.copy()
            for k in ("tuning_distances", "tuning_angles", "sigma_distances", "sigma_angles", "cell_fr_norm",
                      "test_angles", "test_directions"):
                res[f"bvc_{name}_{k}"] = np.array(getattr(bvc, k)).copy()
    res["box2_walls"] = Env.walls.copy()
    np.savez_compressed(os.path.join(GOLD, "modeA_rates.npz"), **res)

    # ------------------------------------------------- modeA_fov (egocentric BVCs)
    rs = np.random.RandomState(777)
    Pe = rs.uniform(0.001, 0.999, size=(160, 2))
    ang = rs.uniform(0, 2 * np.pi, size=160)
    HD = np.stack((np.cos(ang), np.sin(ang)), axis=1) * rs.uniform(0.5, 1.5, size=(160, 1))
    fov = {"P": Pe, "HD": HD}
    with mode_a([]):
        for name, walls in (("box2", BOX_WALLS), ("maze8", maze_walls())):
            E = Environment()
            for w in walls:
                E.add_wall(w)
            AgE = Agent(E, {"dt": 0.01})
            f = FieldOfViewBVCs(AgE, {"min_fr": 0.0, "max_fr": 2.0})
            out = np.zeros((f.n, len(Pe)))
            for j in range(len(Pe)):
                out[:, j] = f.get_state(evaluate_at=None, pos=Pe[j], head_direction=HD[j])[:, 0]
            fov[f"fov_{name}"] = out
            fov[f"fov_{name}_walls"] = E.walls.copy()
            for k in ("tuning_distances", "tuning_angles", "sigma_distances", "sigma_angles", "cell_fr_norm"):
                fov[f"fov_{name}_{k}"] = np.array(getattr(f, k)).copy()
            # the Agent's own head direction (evaluate_at="agent")
            AgE.pos, AgE.head_direction = Pe[0].copy(), HD[0] / np.linalg.norm(HD[0])
            fov[f"fov_{name}_agent"] = f.get_state()[:, 0]
    np.savez_compressed(os.path.join(GOLD, "modeA_fov.npz"), **fov)

    # ------------------------------------------------- periodic boundary conditions
    per = {}
    for name, walls in (("open", []), ("wall", [[[0.5, 0.2], [0.5, 0.8]]])):
        np.random.seed(11)
        Env = Environment({"boundary_conditions": "periodic"})
        for w in walls:
            Env.add_wall(w)
        Ag = Agent(Env, {"dt": 0.05, "speed_mean": 0.5})
        PCs = PlaceCells(Ag, {"n": 30, "widths": 0.15})
        GCs = GridCells(Ag, {"n": 9})
        per[f"{name}_walls"] = Env.walls.copy()
        per[f"{name}_pos0"], per[f"{name}_vel0"] = Ag.pos.copy(), Ag.velocity.copy()
        per[f"{name}_centres"], per[f"{name}_widths"] = PCs.place_cell_centres.copy(), PCs.place_cell_widths.copy()
        per[f"{name}_geom"] = np.array(PCs.wall_geometry)
        per[f"{name}_gridscales"], per[f"{name}_phase"], per[f"{name}_w"] = GCs.gridscales.copy(), GCs.phase_offsets.copy(), GCs.w.copy()
        st = np.random.get_state()
        per[f"{name}_rng_keys"], per[f"{name}_rng_pos"], per[f"{name}_rng_has_gauss"], per[f"{name}_rng_cached"] = st[1], st[2], st[3], st[4]
        for _ in range(800):
            Ag.update(); PCs.update(); GCs.update()
        pos = np.array(Ag.history["pos"])
        wraps = int((np.abs(np.diff(pos, axis=0)) > 0.5).any(axis=1).sum())
        print(f"periodic[{name}]: boundary crossings = {wraps}")
        per[f"{name}_pos"], per[f"{name}_vel"] = pos, np.array(Ag.history["vel"])
        per[f"{name}_rot_vel"], per[f"{name}_dist"] = np.array(Ag.history["rot_vel"]), np.array(Ag.history["distance_travelled"])
        per[f"{name}_pc_fr"], per[f"{name}_gc_fr"] = np.array(PCs.history["firingrate"]), np.array(GCs.history["firingrate"])
        # mode A single steps near / across the boundary + rates at positions
        rs = np.random.RandomState(99)
        A = 256
        pos0 = rs.uniform(0.0, 1.0, size=(A, 2))
        edge = rs.choice(A, A // 2, replace=False)
        pos0[edge, rs.randint(0, 2, size=len(edge))] = rs.choice([0.002, 0.998], size=len(edge)) + rs.normal(scale=1e-3, size=len(edge))
        pos0 = np.clip(pos0, 1e-4, 1 - 1e-4)
        ang = rs.uniform(0, 2 * np.pi, size=A)
        vel0 = rs.rayleigh(0.5, size=A)[:, None] * np.stack((np.cos(ang), np.sin(ang)), axis=1)
        xi = rs.normal(size=(A, 2))
        outp, outmv, outd = [], [], []
        for a in range(A):
            Ag.pos, Ag.velocity = pos0[a].copy(), vel0[a].copy()
            Ag.rotational_velocity, Ag.measured_velocity = 0.0, vel0[a].copy()
            Ag.head_direction, Ag.distance_travelled = vel0[a] / np.linalg.norm(vel0[a]), 0.0
            with mode_a(list(xi[a])):
                Ag.update()
            outp.append(Ag.pos.copy()); outmv.append(Ag.measured_velocity.copy()); outd.append(Ag.distance_travelled)
        per[f"{name}_A_pos0"], per[f"{name}_A_vel0"], per[f"{name}_A_xi"] = pos0, vel0, xi
        per[f"{name}_A_pos"], per[f"{name}_A_mv"], per[f"{name}_A_dist"] = np.array(outp), np.array(outmv), np.array(outd)
        print(f"periodic[{name}] mode A: wrapped = {int((np.abs(np.array(outp) - pos0) > 0.5).any(axis=1).sum())} / {A}")
        with mode_a([]):
            per[f"{name}_A_pc"] = PCs.get_state(evaluate_at=None, pos=pos0)
    np.savez_compressed(os.path.join(GOLD, "periodic.npz"), **per)
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)) // 1024, "KiB")


LROOM = [[0, 0], [1, 0], [1, 0.5], [0.5, 0.5], [0.5, 1], [0, 1]]          # an L-shaped room (6 boundary walls)
HOLE = [[0.4, 0.4], [0.6, 0.4], [0.6, 0.6], [0.4, 0.6]]


def gen_polygon():
    """Polygon boundary / holes (Environment.py:112-160, :807-817): the walls are the polygon's and the holes' edges,
    PlaceCells keep the hard-coded `walls[4:]` (Environment.py:715-717).  shapely is absent here: the in-environment
    test comes from oracle/ref_shim.py's stub, everything else is the unmodified reference."""
    riab = ref_shim.import_reference()
    assert riab is not None, "reference not present"
    from ratinabox.Environment import Environment
    from ratinabox.Agent import Agent
    from ratinabox.Neurons import PlaceCells, BoundaryVectorCells
    out = {}
    cases = (("lroom", {"boundary": LROOM, "walls": [[[0.25, 0.0], [0.25, 0.3]]]}),
             ("holed", {"holes": [HOLE], "walls": [[[0.8, 0.0], [0.8, 0.35]]]}))
    for name, params in cases:
        np.random.seed(23)
        Env = Environment(dict(params))
        Ag = Agent(Env, {"dt": 0.02, "speed_mean": 0.25})
        PCs = PlaceCells(Ag, {"n": 24, "widths": 0.15})
        BVCs = BoundaryVectorCells(Ag, {"n": 6})
        out[f"{name}_walls"] = Env.walls.copy()
        out[f"{name}_extent"] = np.array(Env.extent, dtype=float)
        out[f"{name}_pos0"], out[f"{name}_vel0"] = Ag.pos.copy(), Ag.velocity.copy()
        out[f"{name}_centres"], out[f"{name}_widths"] = PCs.place_cell_centres.copy(), PCs.place_cell_widths.copy()
        out[f"{name}_geom"] = np.array(PCs.wall_geometry)
        out[f"{name}_bvc"] = np.stack((BVCs.tuning_distances, BVCs.tuning_angles, BVCs.sigma_distances, BVCs.sigma_angles))
        st = np.random.get_state()
        out[f"{name}_rng_keys"], out[f"{name}_rng_pos"], out[f"{name}_rng_has_gauss"], out[f"{name}_rng_cached"] = st[1], st[2], st[3], st[4]
        for _ in range(1000):
            Ag.update(); PCs.update(); BVCs.update()
        out[f"{name}_pos"], out[f"{name}_vel"] = np.array(Ag.history["pos"]), np.array(Ag.history["vel"])
        out[f"{name}_pc_fr"], out[f"{name}_bvc_fr"] = np.array(PCs.history["firingrate"]), np.array(BVCs.history["firingrate"])
        inside = all(Env.check_if_position_is_in_environment(p) for p in out[f"{name}_pos"])
        print(f"polygon[{name}]: {len(Env.walls)} walls, geometry {PCs.wall_geometry}, trajectory inside: {inside}")
        # mode A single steps from positions inside the environment, half of them hugging a wall at speed
        rs = np.random.RandomState(5)
        A = 384
        np.random.seed(77)
        pos0 = Env.sample_positions(n=A, method="random")
        wl = Env.walls
        for a in range(A // 2):
            w = wl[rs.randint(len(wl))]
            q = w[0] + rs.uniform(0.05, 0.95) * (w[1] - w[0])
            nrm = np.array([-(w[1] - w[0])[1], (w[1] - w[0])[0]]); nrm /= np.linalg.norm(nrm)
            for sgn in (1.0, -1.0):
                cand = q + sgn * rs.uniform(0.002, 0.02) * nrm
                if Env.check_if_position_is_in_environment(cand):
                    pos0[a] = cand
                    break
        ang = rs.uniform(0, 2 * np.pi, size=A)
        vel0 = rs.rayleigh(0.4, size=A)[:, None] * np.stack((np.cos(ang), np.sin(ang)), axis=1)
        xi = rs.normal(size=(A, 2))
        outp, outv, outmv = [], [], []
        for a in range(A):
            Ag.pos, Ag.velocity = pos0[a].copy(), vel0[a].copy()
            Ag.rotational_velocity, Ag.measured_velocity = 0.0, vel0[a].copy()
            Ag.head_direction, Ag.distance_travelled = vel0[a] / np.linalg.norm(vel0[a]), 0.0
            with mode_a(list(xi[a])):
                Ag.update()
            outp.append(Ag.pos.copy()); outv.append(Ag.velocity.copy()); outmv.append(Ag.measured_velocity.copy())
        out[f"{name}_A_pos0"], out[f"{name}_A_vel0"], out[f"{name}_A_xi"] = pos0, vel0, xi
        out[f"{name}_A_pos"], out[f"{name}_A_vel"], out[f"{name}_A_mv"] = np.array(outp), np.array(outv), np.array(outmv)
        bounced = int((np.abs(np.linalg.norm(np.array(outv), axis=1) - 0.5 * 0.25) < 1e-12).sum())
        print(f"polygon[{name}] mode A: {bounced} / {A} steps bounced")
        with mode_a([]):
            out[f"{name}_A_pc"] = PCs.get_state(evaluate_at=None, pos=pos0)
            out[f"{name}_A_bvc"] = BVCs.get_state(evaluate_at=None, pos=pos0)
        np.random.seed(3)
        out[f"{name}_samples_uj"] = Env.sample_positions(n=50, method="uniform_jitter")
    np.savez_compressed(os.path.join(GOLD, "polygon.npz"), **out)
    print("polygon.npz", os.path.getsize(os.path.join(GOLD, "polygon.npz")) // 1024, "KiB")


OVC_WALLS = [[[0.3, 0.0], [0.3, 0.5]], [[0.7, 1.0], [0.7, 0.5]]]
OVC_OBJECTS = [([0.15, 0.2], 0), ([0.5, 0.8], "same"), ([0.85, 0.3], "new"), ([0.5, 0.25], "new"), ([0.9, 0.9], 1)]


def gen_ovc():
    """ObjectVectorCells / FieldOfViewOVCs (Neurons.py:1892-2160): five objects of three types in the two-wall box."""
    riab = ref_shim.import_reference()
    assert riab is not None, "reference not present"
    from ratinabox.Environment import Environment
    from ratinabox.Agent import Agent
    from ratinabox.Neurons import ObjectVectorCells, FieldOfViewOVCs
    out = {}
    np.random.seed(31)
    Env = Environment()
    for w in OVC_WALLS:
        Env.add_wall(w)
    for o, t in OVC_OBJECTS:
        Env.add_object(o, type=t)
    out["objects"], out["object_types"] = Env.objects["objects"].copy(), Env.objects["object_types"].copy()
    Ag = Agent(Env, {"dt": 0.02})
    pops = {"allo": ObjectVectorCells(Ag, {"n": 12}),
            "eucl": ObjectVectorCells(Ag, {"n": 6, "walls_occlude": False, "object_tuning_type": 1}),
            "fov": FieldOfViewOVCs(Ag, {"object_tuning_type": 0, "spatial_resolution": 0.05})}
    for k, P in pops.items():
        out[f"{k}_tuning"] = np.stack((P.tuning_distances, P.tuning_angles, P.sigma_distances, P.sigma_angles))
        out[f"{k}_types"] = np.array(P.tuning_types)
        out[f"{k}_geom"] = np.array(P.wall_geometry)
        print(f"ovc[{k}]: n = {P.n}, frame {P.reference_frame}, geometry {P.wall_geometry}")
    out["pos0"], out["vel0"] = Ag.pos.copy(), Ag.velocity.copy()
    st = np.random.get_state()
    out["rng_keys"], out["rng_pos"], out["rng_has_gauss"], out["rng_cached"] = st[1], st[2], st[3], st[4]
    for _ in range(400):
        Ag.update()
        for P in pops.values():
            P.update()
    out["pos"], out["head"] = np.array(Ag.history["pos"]), np.array(Ag.history["head_direction"])
    for k, P in pops.items():
        out[f"{k}_fr"] = np.array(P.history["firingrate"])
    rs = np.random.RandomState(17)
    A = 384
    pos = rs.uniform(0.02, 0.98, size=(A, 2))
    ang = rs.uniform(0, 2 * np.pi, size=A)
    hd = np.stack((np.cos(ang), np.sin(ang)), axis=1)
    out["A_pos"], out["A_hd"] = pos, hd
    with mode_a([]):
        out["A_allo"] = pops["allo"].get_state(evaluate_at=None, pos=pos)
        out["A_eucl"] = pops["eucl"].get_state(evaluate_at=None, pos=pos)
        out["A_fov"] = np.stack([pops["fov"].get_state(evaluate_at=None, pos=pos[a], head_direction=hd[a])[:, 0] for a in range(A)], axis=1)
    print("ovc: max rates", out["A_allo"].max(), out["A_eucl"].max(), out["A_fov"].max())
    np.savez_compressed(os.path.join(GOLD, "ovc.npz"), **out)
    print("ovc.npz", os.path.getsize(os.path.join(GOLD, "ovc.npz")) // 1024, "KiB")


# Agent parameter / keyword variants of Agent.update (Agent.py:268-521): (constructor params, update kwargs)
PARAM_VARIANTS = {
    "speed_std0": ({"speed_std": 0.0}, {}),                                   # Agent.py:310-311: s' = speed_mean
    "thigmotaxis0": ({"thigmotaxis": 0.0}, {}),                               # spring only
    "thigmotaxis1": ({"thigmotaxis": 1.0}, {}),                               # conveyor belt only
    "no_repel": ({"wall_repel_strength": 0.0}, {}),                           # Agent.py:359-360: skipped
    "strong_repel": ({"wall_repel_strength": 2.5, "wall_repel_distance": 0.2}, {}),
    "fast_head": ({"head_direction_smoothing_timescale": 0.005}, {}),         # tau_h <= dt: head = measured direction
    "timescales": ({"speed_coherence_time": 0.1, "rotational_velocity_coherence_time": 0.3,
                    "rotational_velocity_std": 3.0, "speed_mean": 0.2}, {}),
    "kwargs": ({}, {"speed_mean": 0.3, "speed_coherence_time": 0.2, "rotational_velocity_std": 1.0,
                    "rotational_velocity_coherence_time": 0.05, "rotational_velocity_drift": 0.7,
                    "thigmotaxis": 0.8, "wall_repel_distance": 0.15, "wall_repel_strength": 1.5,
                    "head_direction_smoothing_timescale": 0.4}),             # the kwarg quirks of :280-285, :302-311, :483-489
    "kw_std0": ({"speed_std": 0.0}, {"speed_mean": 0.3}),                     # attribute speed_std, kwarg speed_mean
    "dt_arg": ({}, {"dt": 0.05}),                                             # dt persists (:193-194)
    "drift_weak": ({}, {"drift_ratio": 0.5}),
    "drift_strong": ({"speed_mean": 0.15}, {"drift_ratio": 5.0}),
}


def gen_params():
    """Single teacher-forced steps (zero jitter, injected normals) of the unmodified reference for every parameter /
    keyword variant in PARAM_VARIANTS, 160 agents each in the two-wall box, half of them next to a wall."""
    riab = ref_shim.import_reference()
    assert riab is not None, "reference not present"
    from ratinabox.Environment import Environment
    from ratinabox.Agent import Agent
    out = {}
    rs = np.random.RandomState(77)
    A = 160
    Env0 = Environment()
    for w in BOX_WALLS:
        Env0.add_wall(w)
    pos0 = rs.uniform(0.002, 0.998, size=(A, 2))
    near = rs.choice(A, A // 2, replace=False)
    wl = Env0.walls[rs.randint(0, len(Env0.walls), size=len(near))]
    lam = rs.uniform(0, 1, size=(len(near), 1))
    pos0[near] = np.clip(wl[:, 0] + lam * (wl[:, 1] - wl[:, 0]) + rs.normal(scale=4e-3, size=(len(near), 2)), 0.0005, 0.9995)
    speed = rs.rayleigh(0.1, size=A) * rs.choice([1.0, 1.0, 5.0], size=A)
    ang = rs.uniform(0, 2 * np.pi, size=A)
    vel0 = speed[:, None] * np.stack((np.cos(ang), np.sin(ang)), axis=1)
    rot0 = rs.normal(scale=2.0, size=A)
    mv0 = vel0 + rs.normal(scale=0.01, size=(A, 2))
    hd0 = mv0 / np.linalg.norm(mv0, axis=1, keepdims=True)
    xi = rs.normal(size=(A, 2))
    drift = rs.normal(scale=0.15, size=(A, 2))
    out.update(pos0=pos0, vel0=vel0, rot0=rot0, mv0=mv0, hd0=hd0, xi=xi, drift=drift, walls=Env0.walls)
    for name, (params, kw) in PARAM_VARIANTS.items():
        Env = Environment()
        for w in BOX_WALLS:
            Env.add_wall(w)
        Ag = Agent(Env, dict({"dt": 0.01}, **params))
        kw = dict(kw)
        ratio = kw.pop("drift_ratio", None)
        res = {k: [] for k in ("pos", "vel", "rot", "mv", "mrot", "hd", "dist", "dclose")}
        for a in range(A):
            Ag.pos, Ag.velocity = pos0[a].copy(), vel0[a].copy()
            Ag.rotational_velocity, Ag.measured_velocity = float(rot0[a]), mv0[a].copy()
            Ag.head_direction, Ag.distance_travelled, Ag.t, Ag.dt = hd0[a].copy(), 0.0, 0.0, 0.01
            with mode_a(list(xi[a])):
                if ratio is not None:
                    Ag.update(drift_velocity=drift[a].copy(), drift_to_random_strength_ratio=ratio, **kw)
                else:
                    Ag.update(**kw)
            res["pos"].append(Ag.pos.copy()); res["vel"].append(Ag.velocity.copy()); res["rot"].append(Ag.rotational_velocity)
            res["mv"].append(Ag.measured_velocity.copy()); res["mrot"].append(Ag.measured_rotational_velocity)
            res["hd"].append(Ag.head_direction.copy()); res["dist"].append(Ag.distance_travelled)
            res["dclose"].append(Ag.distance_to_closest_wall)
        for k, v in res.items():
            out[f"{name}_{k}"] = np.array(v)
        print(f"params[{name}]: dt after = {Ag.dt}, max speed out = {np.linalg.norm(np.array(res['vel']), axis=1).max():.3f}")
    np.savez_compressed(os.path.join(GOLD, "modeA_params.npz"), **out)
    print("modeA_params.npz", os.path.getsize(os.path.join(GOLD, "modeA_params.npz")) // 1024, "KiB")


def gen_histogram():
    """utils.bin_data_for_histogramming (utils.py:544-589) on random 2D data: plain, weighted and bin-count-normalised."""
    riab = ref_shim.import_reference()
    assert riab is not None, "reference not present"
    from ratinabox import utils
    rs = np.random.RandomState(8)
    data = rs.uniform(-0.02, 1.52, size=(4000, 2)) * np.array([1.0, 0.66])        # some samples fall outside the extent
    data[:5] = [[0.0, 0.0], [1.5, 1.0], [1.5, 0.3], [0.7, 1.0], [0.75, 0.5]]      # on edges / the right-most edges
    w = rs.uniform(0, 3, size=4000)
    extent, dx = [0.0, 1.5, 0.0, 1.0], 0.05
    out = {"data": data, "weights": w, "extent": np.array(extent), "dx": dx}
    out["plain"] = utils.bin_data_for_histogramming(data, extent, dx)
    out["weighted"] = utils.bin_data_for_histogramming(data, extent, dx, weights=w)
    hm, zb = utils.bin_data_for_histogramming(data, extent, dx, weights=w, norm_by_bincount=True, return_zero_bins=True)
    out["normed"], out["zero_bins"] = hm, zb
    np.savez_compressed(os.path.join(GOLD, "histogram.npz"), **out)
    print("histogram.npz", out["plain"].shape, int(out["plain"].sum()), "of", len(data), "samples inside")


def gen_api_defaults():
    """default_params of the reference's classes on the path -> tests/golden/api_defaults.json (the host mirror must
    accept the same keys with the same defaults)."""
    import json
    riab = ref_shim.import_reference()
    assert riab is not None, "reference not present"
    from ratinabox.Environment import Environment
    from ratinabox.Agent import Agent
    import importlib
    RN = importlib.import_module("ratinabox.Neurons")      # (the package attribute `Neurons` is the class)

    def clean(d):
        out = {}
        for k, v in d.items():
            if isinstance(v, np.ndarray):
                v = v.tolist()
            elif isinstance(v, tuple):
                v = list(v)
            try:
                json.dumps(v)
            except TypeError:
                v = repr(v)
            out[k] = v
        return out

    ref = {"Environment": clean(Environment.default_params), "Agent": clean(Agent.default_params)}
    for name in ("Neurons", "PlaceCells", "GridCells", "VectorCells", "BoundaryVectorCells", "FieldOfViewBVCs",
                 "ObjectVectorCells", "FieldOfViewOVCs"):
        ref[name] = clean(getattr(RN, name).default_params)
    with open(os.path.join(GOLD, "api_defaults.json"), "w") as f:
        json.dump(ref, f, indent=1, sort_keys=True)
    print("api_defaults.json", {k: len(v) for k, v in ref.items()})


def gen_host_utils():
    """Host-side helpers the mirror re-implements: Environment.sample_positions (box), utils.distribution_sampler and the
    three vector-cell assemblies, each under a fixed np.random seed -> tests/golden/host_utils.npz."""
    riab = ref_shim.import_reference()
    assert riab is not None, "reference not present"
    from ratinabox.Environment import Environment
    from ratinabox import utils
    out = {}
    Env = Environment({"aspect": 2, "scale": 0.8})
    for method in ("random", "uniform", "uniform_jitter"):
        for n in (7, 40, 100):
            np.random.seed(5)
            out[f"sample_{method}_{n}"] = Env.sample_positions(n=n, method=method)
    for k, (name, prm) in enumerate((("uniform", (0.1, 0.4)), ("rayleigh", (0.2,)), ("normal", (1.0, 0.3)), ("logarithmic", (0.05, 1.0)),
                                     ("delta", (0.7,)), ("modules", (0.3, 0.5, 0.8)), ("truncnorm", (0.0, 1.0, 0.5, 0.2)))):
        np.random.seed(9)
        out[f"dist_{name}"] = np.asarray(utils.distribution_sampler(name, prm, (23,)))
    np.random.seed(4)
    out["assembly_random"] = np.stack(utils.create_random_assembly(n=17))
    np.random.seed(4)
    out["assembly_random_lists"] = np.stack(utils.create_random_assembly(tuning_distance=[0.1, 0.2, 0.3], sigma_angle=[10.0, 20.0, 30.0]))
    out["assembly_uniform"] = np.stack(utils.create_uniform_radial_assembly(distance_range=[0.02, 0.3], angle_range=[0, 60], spatial_resolution=0.04))
    out["assembly_diverging"] = np.stack(utils.create_diverging_radial_assembly(distance_range=[0.02, 0.4], angle_range=[0, 75], spatial_resolution=0.02, beta=5))
    np.savez_compressed(os.path.join(GOLD, "host_utils.npz"), **out)
    print("host_utils.npz", {k: v.shape for k, v in out.items() if k.startswith("assembly")})


def gen_host_mirror():
    """The 2 x 1 box with a doorway (Environment walls, extent, discretisation, sample_positions under np.random.seed(5))
    and the set-up helpers (distribution_sampler, create_random_assembly, rotate) that the host mirror must reproduce bit
    for bit -> tests/golden/host_mirror.npz."""
    riab = ref_shim.import_reference()
    assert riab is not None, "reference not present"
    from ratinabox.Environment import Environment
    from ratinabox import utils
    R = Environment({"aspect": 2, "scale": 1})
    R.add_wall([[1, 0], [1, 0.35]])
    R.add_wall([[1, 0.65], [1, 1]])
    out = {"walls": R.walls, "extent": np.asarray(R.extent, dtype=float), "flattened_discrete_coords": R.flattened_discrete_coords}
    for method, n in (("uniform_jitter", 100), ("uniform", 30), ("random", 7), ("uniform_jitter", 1024)):
        np.random.seed(5)
        out[f"sample_{method}_{n}"] = R.sample_positions(n=n, method=method)
    for name, prm, shape in (("uniform", (0.2, 1.0), (9,)), ("modules", (0.3, 0.5, 0.8), (10,)), ("rayleigh", (0.3,), (5,)),
                             ("normal", (0, 1), (4, 2)), ("logarithmic", (0.1, 1.0), (6,)), ("delta", (0.4,), (3,))):
        np.random.seed(3)
        out[f"dist_{name}"] = np.asarray(utils.distribution_sampler(name, prm, shape))
    np.random.seed(4)
    out["assembly_n12"] = np.stack(utils.create_random_assembly(n=12))
    out["rotate"] = utils.rotate(np.array([1, 0]), 0.3)
    np.savez_compressed(os.path.join(GOLD, "host_mirror.npz"), **out)
    print("host_mirror.npz", {k: v.shape for k, v in out.items()})


def gen_config1():
    """BASELINE.json configs[0] (1 agent, default box, 100 Gaussian PlaceCells, dt = 10 ms) in the open box and with the
    two internal walls, 300 steps of the reference teacher-forced like mode A: geometry jitter zeroed, the `scale == dt`
    normals fed from RandomState(7).  Per step the Agent's state before it, the two Ornstein-Uhlenbeck normals it drew and
    the firing rates after it -> tests/golden/config1.npz."""
    import ref_driver
    steps, N = 300, 100
    state = ("pos", "velocity", "rotational_velocity", "measured_velocity", "head_direction", "distance_travelled")
    out = {}
    for name, walls in (("open", []), ("box2", BOX_WALLS)):
        rs = np.random.RandomState(7)
        centres = rs.uniform(0.05, 0.95, (N, 2))
        geom = "line_of_sight" if walls else "euclidean"
        _, _, RA, (RP,) = ref_driver.build(walls, [("place", {"n": N, "place_cell_centres": centres, "widths": 0.2,
                                                              "wall_geometry": geom}, None)],
                                           pos=[0.5, 0.52], vel=[0.05, 0.06], dt=0.01, seed=3)
        rec = {k: [np.array(getattr(RA, k), dtype=float)] for k in state}
        xi, fr = [], []
        for s in range(steps):
            tape, used = rs.normal(size=2 + N).tolist(), []
            with mode_a(tape, used):
                RA.update()
                RP.update()
            assert len(used) <= 2 + N                       # every draw came from the tape
            xi.append(used[:2])
            fr.append(np.array(RP.firingrate, dtype=float))
            for k in state:
                rec[k].append(np.array(getattr(RA, k), dtype=float))
        out[f"{name}_walls"] = np.array(walls, dtype=float).reshape(-1, 2, 2)
        out[f"{name}_centres"], out[f"{name}_xi"], out[f"{name}_rates"] = centres, np.array(xi), np.array(fr)
        for k in state:
            out[f"{name}_{k}"] = np.array(rec[k])
    np.savez_compressed(os.path.join(GOLD, "config1.npz"), **out)
    print("config1.npz", os.path.getsize(os.path.join(GOLD, "config1.npz")) // 1024, "KiB")


if __name__ == "__main__":
    if sys.argv[1:] == ["api"]:
        gen_api_defaults()
    elif sys.argv[1:] == ["host"]:
        gen_host_utils()
    elif sys.argv[1:] == ["histogram"]:
        gen_histogram()
    elif sys.argv[1:] == ["params"]:
        gen_params()
    elif sys.argv[1:] == ["polygon"]:
        gen_polygon()
    elif sys.argv[1:] == ["ovc"]:
        gen_ovc()
    elif sys.argv[1:] == ["mirror"]:
        gen_host_mirror()
    elif sys.argv[1:] == ["config1"]:
        gen_config1()
    else:
        main()
        gen_polygon()
        gen_ovc()
        gen_params()
        gen_histogram()
        gen_api_defaults()
        gen_host_utils()
        gen_host_mirror()
        gen_config1()
