"""CPU-only checks: the C-ABI library loads and exports every symbol include/riab_b200.h
declares; the host-side packers agree with NumPy; the host mirror of Environment agrees
with the oracle and with the reference's stored outputs (tests/golden); sharding helpers work
under a world_size-2 gloo group.  No CUDA calls."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

import riab_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from ratinabox_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "riab_b200.h")).read()
    declared = set(re.findall(r"\b(riab_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in riab_b200.h but not exported"
        assert name in _lib.SYMBOLS, f"{name} has no ctypes prototype"
    assert lib.riab_abi_version() == 2
    assert lib.riab_launch_count() == 0


def test_struct_sizes_match_header():
    """ctypes mirrors must have the C layout (spot check through the packers that fill them)."""
    from ratinabox_b200 import _lib
    assert C.sizeof(_lib.MotionParams) == 14 * 8
    assert C.sizeof(_lib.Agents) == 10 * 8
    assert C.sizeof(_lib.Env) == 8 + 4 + 4 + 32 + 4 + 4 + 8 + 4 + 4   # + boundary_mode, n_hole_walls, scale, hole_wall0, reserved
    assert C.sizeof(_lib.StepIO) == 9 * 8


def test_place_pack_matches_numpy():
    from ratinabox_b200 import _lib
    lib = _lib.load()
    rs = np.random.RandomState(0)
    n = 37
    centres = rs.uniform(0, 1, (n, 2))
    widths = rs.uniform(0.1, 0.3, n)
    env = O.OracleEnvironment(walls=[[[0.3, 0.0], [0.3, 0.5]], [[0.7, 1.0], [0.7, 0.5]]])
    walls = np.ascontiguousarray(env.walls)
    ext = np.ascontiguousarray(env.extent)
    meta = _lib.PlaceCells()
    nfl = lib.riab_place_pack_floats(n, 2)
    out = np.zeros(nfl, dtype=np.float32)
    f = lambda a: a.ctypes.data_as(_lib.c_double_p)
    rc = lib.riab_place_pack(f(centres), f(widths), n, f(walls), 6, 4, f(ext), 1, C.byref(meta),
                             out.ctypes.data_as(_lib.c_float_p))
    assert rc == 0
    npad = meta.n_pad
    assert npad % 128 == 0 and npad >= n and meta.n_inner_walls == 2
    assert np.allclose(out[:n], centres[:, 0] - 0.5, atol=1e-7)
    assert np.allclose(out[npad:npad + n], centres[:, 1] - 0.5, atol=1e-7)
    assert np.allclose(out[2 * npad:2 * npad + n], np.log2(np.e) / (2 * widths ** 2), rtol=1e-6)
    # wall 0 = x=0.3 from y=0 to 0.5: f = signed distance to the line, t = parameter along it
    fc, tc = out[4 * npad:4 * npad + n], out[5 * npad:5 * npad + n]
    assert np.allclose(np.abs(fc), np.abs(centres[:, 0] - 0.3), atol=1e-6)
    assert np.allclose(tc, centres[:, 1] / 0.5, atol=1e-6)
    assert meta.eps[0] > 0 and meta.eps[1] > 0
    # bad arguments are refused with a message, not a crash
    assert lib.riab_place_pack(None, f(widths), n, f(walls), 6, 4, f(ext), 1, C.byref(meta),
                               out.ctypes.data_as(_lib.c_float_p)) < 0
    assert b"riab_place_pack" in lib.riab_last_error()


def test_grid_and_bvc_pack():
    from ratinabox_b200 import _lib
    lib = _lib.load()
    rs = np.random.RandomState(1)
    n = 10
    gs, th, ph = rs.uniform(0.2, 1, n), rs.uniform(0, 1, n), rs.uniform(0, 2 * np.pi, (n, 2))
    w = O.grid_cells_w(th)
    ext = np.array([0.0, 1.0, 0.0, 1.0])
    meta = _lib.GridCells()
    out = np.zeros(lib.riab_grid_pack_floats(n), dtype=np.float32)
    f = lambda a: np.ascontiguousarray(a).ctypes.data_as(_lib.c_double_p)
    assert lib.riab_grid_pack(f(gs), f(ph), f(w), n, f(ext), C.byref(meta), out.ctypes.data_as(_lib.c_float_p)) == 0
    npad = meta.n_pad
    # reconstruct phi at a test position and compare with the oracle's phases
    p = np.array([0.37, 0.81])
    origin = gs[:, None] * ph / (2 * np.pi)
    for k in range(3):
        kx, ky, ph0 = out[(3 * k) * npad:(3 * k) * npad + n], out[(3 * k + 1) * npad:(3 * k + 1) * npad + n], out[(3 * k + 2) * npad:(3 * k + 2) * npad + n]
        phi = ph0 - ((p[0] - 0.5) * kx + (p[1] - 0.5) * ky)
        ref = (2 * np.pi / gs) * ((origin - p) @ np.eye(2) * w[:, k, :]).sum(axis=1)
        assert np.abs(np.cos(phi) - np.cos(ref)).max() < 2e-5
    T = 180
    dirs, angs = O.bvc_test_angles(2)
    mu_d, mu_t, sg_d, sg_t = rs.uniform(0.05, 0.3, n), rs.uniform(0, 6.28, n), rs.uniform(0.08, 0.1, n), rs.uniform(0.17, 0.5, n)
    bmeta = _lib.BvcCells()
    bout = np.zeros(lib.riab_bvc_pack_floats(n, T), dtype=np.float32)
    assert lib.riab_bvc_pack(f(mu_d), f(mu_t), f(sg_d), f(sg_t), n, f(angs), T, C.byref(bmeta),
                             bout.ctypes.data_as(_lib.c_float_p)) == 0
    np_ = bmeta.n_pad
    assert np_ == 64
    assert np.allclose(bout[2 * np_:2 * np_ + n], 1 / O.bvc_cell_fr_norm(angs, sg_t), rtol=1e-6)
    # von Mises table in SLOT order (cells sorted by preferred angle), perm[slot] = cell, one angular window per 32 slots
    tail = bout[6 * np_ + np_ * T + 2 * T:].view(np.int32)
    perm, win = tail[:np_], tail[np_:].reshape(-1, 2)
    assert len(tail) == np_ + 2 * (np_ // 32) and sorted(perm[:n]) == list(range(n)) and list(perm[n:]) == list(range(n, np_))
    assert np.all(np.diff(mu_t[perm[:n]]) >= 0)
    vm = bout[3 * np_:3 * np_ + np_ * T].reshape(1, T, 64)[0, :, :n].T
    full = O.von_mises_peak1(angs[None, :], mu_t[:, None], sg_t[:, None])
    assert np.allclose(vm, full[perm[:n]], rtol=1e-6, atol=1e-30)
    for w, (th0, tlen) in enumerate(win):                   # outside the window every weight of the warp is < 2^-30
        cells = perm[32 * w:32 * w + 32]
        cells = cells[cells < n]
        inside = np.zeros(T, bool)
        inside[(th0 + np.arange(tlen)) % T] = True
        assert 0 <= th0 < T and 0 <= tlen <= T
        if len(cells):
            assert full[cells][:, ~inside].max(initial=0.0) < 2.0 ** -30 * (1 + 1e-6)
            assert tlen == T or (full[cells][:, th0].max() >= 2.0 ** -30 * (1 - 1e-6) and full[cells][:, (th0 + tlen - 1) % T].max() >= 2.0 ** -30 * (1 - 1e-6))
    ext = bout[3 * np_ + np_ * T:6 * np_ + np_ * T + 2 * T]  # egocentric extras: kap | cos mu | sin mu | cos theta | sin theta
    assert np.allclose(ext[:n], np.log2(np.e) / sg_t ** 2, rtol=1e-6)
    assert np.allclose(ext[np_:np_ + n], np.cos(mu_t), atol=1e-7) and np.allclose(ext[2 * np_:2 * np_ + n], np.sin(mu_t), atol=1e-7)
    assert np.allclose(ext[3 * np_:3 * np_ + T], np.cos(angs), atol=1e-7) and len(ext) == 3 * np_ + 2 * T
    assert lib.riab_bvc_scratch_floats(33, T) == 2 * T * 32


def test_environment_mirror_matches_oracle_and_reference(golden):
    """The reference's side is tests/golden/host_mirror.npz (oracle/gen_golden.py mirror)."""
    import ratinabox_b200 as rb
    E = rb.Environment({"aspect": 2, "scale": 1})
    E.add_wall([[1, 0], [1, 0.35]])
    E.add_wall([[1, 0.65], [1, 1]])
    env = O.OracleEnvironment(scale=1, aspect=2, walls=[[[1, 0], [1, 0.35]], [[1, 0.65], [1, 1]]])
    assert np.array_equal(E.walls, env.walls) and np.array_equal(E.extent, env.extent)
    assert E.check_if_position_is_in_environment([0.5, 0.5]) and not E.check_if_position_is_in_environment([2.0, 0.5])
    R = golden("host_mirror.npz")
    assert np.array_equal(R["walls"], E.walls) and np.array_equal(R["extent"], E.extent)
    assert np.array_equal(R["flattened_discrete_coords"], E.flattened_discrete_coords)
    for method, n in (("uniform_jitter", 100), ("uniform", 30), ("random", 7), ("uniform_jitter", 1024)):
        np.random.seed(5); b = E.sample_positions(n=n, method=method)
        assert np.array_equal(R[f"sample_{method}_{n}"], b), method


def test_set_up_helpers_match_reference(golden):
    """The reference's side is tests/golden/host_mirror.npz (oracle/gen_golden.py mirror)."""
    from ratinabox_b200 import utils as U
    R = golden("host_mirror.npz")
    for name, prm, shape in (("uniform", (0.2, 1.0), (9,)), ("modules", (0.3, 0.5, 0.8), (10,)), ("rayleigh", (0.3,), (5,)),
                             ("normal", (0, 1), (4, 2)), ("logarithmic", (0.1, 1.0), (6,)), ("delta", (0.4,), (3,))):
        np.random.seed(3); b = U.distribution_sampler(name, prm, shape)
        assert np.array_equal(R[f"dist_{name}"], b), name
    np.random.seed(4); b = U.create_random_assembly(n=12)
    assert len(b) == len(R["assembly_n12"])
    for x, y in zip(R["assembly_n12"], b):
        assert np.array_equal(x, y)
    assert np.array_equal(R["rotate"], U.rotate(np.array([1, 0]), 0.3))


def test_product_path_never_imports_the_oracle():
    import ast
    pkg = os.path.join(ROOT, "ratinabox_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            tree = ast.parse(open(os.path.join(pkg, fn)).read())
            for node in ast.walk(tree):
                names = []
                if isinstance(node, ast.Import):
                    names = [a.name for a in node.names]
                elif isinstance(node, ast.ImportFrom):
                    names = [node.module or ""]
                assert not any("oracle" in n or "ref_shim" in n for n in names), (fn, names)


def _gloo_worker(rank, world, port, n_total, q):
    import torch
    import torch.distributed as dist
    from ratinabox_b200.distributed import shard_range, gather_agent_axis, agent_params_for_rank
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    s, e = shard_range(n_total, rank, world)
    p = agent_params_for_rank({"dt": 0.01}, n_total, rank, world)
    assert p["n_agents"] == e - s and p["id_offset"] == s
    full = np.arange(5 * n_total * 2, dtype=np.float32).reshape(5, n_total, 2)      # (steps, agents, 2) history slab
    got = gather_agent_axis(full[:, s:e], n_total, axis=1, dst=0)
    ok = (got is None) if rank != 0 else np.array_equal(got, full)
    t = torch.tensor([1.0 + rank])
    dist.all_reduce(t, op=dist.ReduceOp.MAX)                                           # the bench's max-over-ranks timing
    ok = ok and float(t) == float(world)
    q.put((rank, bool(ok)))
    dist.destroy_process_group()


def test_sharding_and_history_gather_gloo_world2():
    import torch.multiprocessing as mp
    from ratinabox_b200.distributed import shard_range
    assert [shard_range(10, r, 3) for r in range(3)] == [(0, 4), (4, 7), (7, 10)]
    assert shard_range(65536, 7, 8) == (57344, 65536)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, 11, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert res == [(0, True), (1, True)]


def test_environment_mirror_polygon_and_holes_host_logic(golden):
    """Host side of polygon boundaries / holes: wall order (boundary, `walls`, holes, later add_wall), the strict
    in-environment test and sample_positions (Environment.py:560-633) -- the latter bit-equal to the live reference
    under the same np.random seed (tests/golden/polygon.npz)."""
    from ratinabox_b200.Environment import Environment
    g = golden("polygon.npz")
    cases = {"lroom": {"boundary": [[0, 0], [1, 0], [1, 0.5], [0.5, 0.5], [0.5, 1], [0, 1]], "walls": [[[0.25, 0.0], [0.25, 0.3]]]},
             "holed": {"holes": [[[0.4, 0.4], [0.6, 0.4], [0.6, 0.6], [0.4, 0.6]]], "walls": [[[0.8, 0.0], [0.8, 0.35]]]}}
    for name, params in cases.items():
        E = Environment(dict(params))
        assert np.array_equal(E.walls, g[f"{name}_walls"]) and E.is_polygonal
        assert E.los_skip == 4                                  # Environment.py:715-717
        np.random.seed(3)
        assert np.array_equal(E.sample_positions(n=50, method="uniform_jitter"), g[f"{name}_samples_uj"])
        assert all(E.check_if_position_is_in_environment(p) for p in g[f"{name}_pos"][::25])
    E = Environment(dict(cases["holed"]))
    assert (E.hole_wall0, E.n_hole_walls, E.n_boundary_walls) == (5, 4, 4)
    E.add_wall([[0.1, 0.1], [0.2, 0.1]])                        # appended AFTER the hole walls, like the reference
    assert len(E.walls) == 10 and (E.hole_wall0, E.n_hole_walls) == (5, 4)
    assert not E.check_if_position_is_in_environment([0.5, 0.5])        # in the hole
    assert E.check_if_position_is_in_environment([0.4, 0.5])            # on the hole's edge: not strictly inside the hole
    L = Environment(dict(cases["lroom"]))
    assert L.check_if_position_is_in_environment([0.25, 0.75]) and not L.check_if_position_is_in_environment([0.75, 0.75])
    assert not L.check_if_position_is_in_environment([0.5, 0.75])       # exactly on a boundary edge: not inside


def test_mirror_default_params_match_the_reference():
    """Every default_params key of the reference's classes on the path exists in the host mirror with the same default
    (tests/golden/api_defaults.json, written from the live reference by oracle/gen_golden.py api); the mirror only ADDS
    the batch-engine knobs."""
    import json
    import ratinabox_b200 as rb
    ref = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "api_defaults.json")))

    def merged(cls):
        d = {}
        for c in reversed(cls.__mro__):
            d.update(getattr(c, "default_params", {}))
        return d

    def same(a, b):
        if isinstance(a, (list, tuple, np.ndarray)) or isinstance(b, (list, tuple, np.ndarray)):
            return np.allclose(np.asarray(a, dtype=float), np.asarray(b, dtype=float))
        return a == b

    pairs = {"Environment": (rb.Environment, ["Environment"]), "Agent": (rb.Agent, ["Agent"]),
             "PlaceCells": (rb.PlaceCells, ["Neurons", "PlaceCells"]), "GridCells": (rb.GridCells, ["Neurons", "GridCells"]),
             "BoundaryVectorCells": (rb.BoundaryVectorCells, ["Neurons", "VectorCells", "BoundaryVectorCells"]),
             "FieldOfViewBVCs": (rb.FieldOfViewBVCs, ["Neurons", "VectorCells", "BoundaryVectorCells", "FieldOfViewBVCs"]),
             "ObjectVectorCells": (rb.ObjectVectorCells, ["Neurons", "VectorCells", "ObjectVectorCells"]),
             "FieldOfViewOVCs": (rb.FieldOfViewOVCs, ["Neurons", "VectorCells", "ObjectVectorCells", "FieldOfViewOVCs"])}
    added = {"Agent": {"n_agents", "seed", "id_offset", "history_bytes_limit", "fused_step"}, "Neurons": {"save_spikes", "history_bytes_limit"}}
    for name, (cls, chain) in pairs.items():
        want = {}
        for c in chain:
            want.update(ref[c])
        have = merged(cls)
        for k, v in want.items():
            if k == "color":
                continue                                   # plotting only
            assert k in have, (name, k)
            assert same(have[k], v), (name, k, have[k], v)
        extra = set(have) - set(want) - {"color"}
        allowed = added.get(name, set()) | added["Neurons"] | {"dtheta", "name", "n", "min_fr", "max_fr"}
        if name in ("Environment", "Agent"):
            allowed = added.get(name, set())
        assert extra <= allowed | set(ref.get("BoundaryVectorCells", {})), (name, sorted(extra - allowed))


def test_host_helpers_match_the_reference(golden):
    """Host-side helpers the mirror re-implements, under the same np.random seeds as the live reference
    (tests/golden/host_utils.npz): Environment.sample_positions in a 1.6 x 0.8 box, utils.distribution_sampler, and the
    random / uniform / diverging vector-cell assemblies."""
    from ratinabox_b200.Environment import Environment
    from ratinabox_b200 import utils as U
    g = golden("host_utils.npz")
    Env = Environment({"aspect": 2, "scale": 0.8})
    for method in ("random", "uniform", "uniform_jitter"):
        for n in (7, 40, 100):
            np.random.seed(5)
            assert np.array_equal(Env.sample_positions(n=n, method=method), g[f"sample_{method}_{n}"]), (method, n)
    for name, prm in (("uniform", (0.1, 0.4)), ("rayleigh", (0.2,)), ("normal", (1.0, 0.3)), ("logarithmic", (0.05, 1.0)),
                      ("delta", (0.7,)), ("modules", (0.3, 0.5, 0.8)), ("truncnorm", (0.0, 1.0, 0.5, 0.2))):
        np.random.seed(9)
        assert np.array_equal(np.asarray(U.distribution_sampler(name, prm, (23,))), g[f"dist_{name}"]), name
    np.random.seed(4)
    assert np.array_equal(np.stack(U.create_random_assembly(n=17)), g["assembly_random"])
    np.random.seed(4)
    assert np.array_equal(np.stack(U.create_random_assembly(tuning_distance=[0.1, 0.2, 0.3], sigma_angle=[10.0, 20.0, 30.0])),
                          g["assembly_random_lists"])
    assert np.array_equal(np.stack(U.create_uniform_radial_assembly(distance_range=[0.02, 0.3], angle_range=[0, 60],
                                                                    spatial_resolution=0.04)), g["assembly_uniform"])
    assert np.array_equal(np.stack(U.create_diverging_radial_assembly(distance_range=[0.02, 0.4], angle_range=[0, 75],
                                                                      spatial_resolution=0.02, beta=5)), g["assembly_diverging"])


def test_environment_mirror_like_the_reference_suite():
    """The 2D cases of the reference's own tests/test_environment.py (:20-23 add_wall, :31-36 sample_positions,
    :38-41 discretise_environment) against the host mirror; 1D is refused loudly."""
    from ratinabox_b200.Environment import Environment
    Env2D = Environment(params={"dimensionality": "2D"})
    assert type(Env2D) == Environment
    n_walls = len(Env2D.walls)
    Env2D.add_wall([[0.2, 0.2], [0.2, 0.2]])                 # the reference's test adds this zero-length wall
    assert len(Env2D.walls) == n_walls + 1
    for method_ in ["uniform", "random", "uniform_random"]:
        assert Env2D.sample_positions(5, method=method_).shape == (5, 2)
    coords = Env2D.discretise_environment(dx=0.01)
    assert type(coords) is np.ndarray and coords.shape == (100, 100, 2)
    with pytest.raises(NotImplementedError):
        Environment(params={"dimensionality": "1D"})


def test_ctypes_structs_have_the_headers_layout(tmp_path):
    """Compile a C program against include/riab_b200.h (gcc: the header is plain C) that prints sizeof / selected
    offsetof of every POD struct, and compare with the ctypes mirrors in ratinabox_b200/_lib.py."""
    import shutil
    import subprocess
    from ratinabox_b200 import _lib
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    pairs = {"riab_env": _lib.Env, "riab_agents": _lib.Agents, "riab_motion_params": _lib.MotionParams,
             "riab_step_io": _lib.StepIO, "riab_place_cells": _lib.PlaceCells, "riab_grid_cells": _lib.GridCells,
             "riab_bvc_cells": _lib.BvcCells, "riab_ovc_cells": _lib.OvcCells, "riab_neuron_noise": _lib.NeuronNoise,
             "riab_rates_out": _lib.RatesOut, "riab_population": _lib.Population, "riab_agent_history": _lib.AgentHistory,
             "riab_history_view": _lib.HistoryView}
    last = {name: cls._fields_[-1][0] for name, cls in pairs.items()}
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "riab_b200.h"', "int main(void) {"]
    for name in pairs:
        src.append(f'  printf("{name} %zu %zu\\n", sizeof({name}), offsetof({name}, {last[name]}));')
    src += ["  return 0;", "}"]
    c = tmp_path / "sizes.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "sizes"
    subprocess.run([gcc, "-std=c11", "-I", os.path.join(ROOT, "include"), str(c), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    for line in out.strip().splitlines():
        name, size, off = line.split()
        cls = pairs[name]
        assert C.sizeof(cls) == int(size), (name, C.sizeof(cls), size)
        assert getattr(cls, last[name]).offset == int(off), (name, last[name])


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm: the live reference staged in oracle/_ref -- or the NumPy port when it is
    absent -- on the host cores) prints ONE JSON line with the keys the driver reads, and its `steps x ms_per_step` is the
    time it really measured; it needs no GPU, so it is checked here."""
    import json
    import subprocess
    env = dict(os.environ, OMP_NUM_THREADS="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.strip().splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "agent-steps/sec" and d["value"] > 0
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_shim
    want_kind = "reference" if ref_shim.reference_root() is not None else "port"
    assert d["cpu_baseline"]["kind"] == want_kind and d["cpu_baseline"]["cores"] >= 1
    assert d["steps"] * d["ms_per_step"] * 1e-3 <= d["wall_s"]          # the timed region fits inside the run
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "c2" in d["config"]["workload"]


def test_step_kernels_got_the_launch_registers_the_setmaxnreg_split_assumes():
    """k_step re-balances registers between its producer and consumer warps with setmaxnreg, which can only move registers
    inside what the launch allocated per SM sub-partition (riab_b200.cu: StepCfg::REGS_LAUNCH, step_cfg_fits): if ptxas gave a
    kernel FEWER registers than the model assumes, the consumers' setmaxnreg.inc never completes and the kernel hangs (a
    6-producer variant did exactly that in round 2: 704 threads get 80 registers, not 88).  Every instantiation in the built
    library must therefore carry its configuration's launch count: 96 for StepCfg<4> (20 warps, 5 per sub-partition), 80 for
    StepCfg<8> and StepCfg<12> (24 warps, 6 per sub-partition), and fit the 48 KB of static shared memory."""
    import shutil
    import subprocess
    from ratinabox_b200 import _lib
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    txt = subprocess.run([tool, "--dump-resource-usage", _lib.lib_path()], capture_output=True, text=True, check=True).stdout
    found = re.findall(r"Function (\S*6k_stepI\S*?7StepCfgILi(\d+)E\S*):\s*\n\s*REG:(\d+) STACK:\d+ SHARED:(\d+)", txt)
    assert len(found) > 50, len(found)
    want = {"4": 96, "8": 80, "12": 80}
    seen = set()
    for name, cfg, reg, shared in found:
        assert int(reg) == want[cfg], (name[:120], cfg, reg)
        assert int(shared) <= 48 * 1024, (name[:120], shared)
        seen.add(cfg)
    assert seen == {"4", "8", "12"}
