#!/usr/bin/env python
"""bench.py -- agent-steps/sec of the RatInABox per-step hot path on B200.

One "step" = Agent.update() + Neurons.update() of every population for every agent
(BASELINE.json metric).  Default workload = BASELINE.json configs[1]:
65 536 agents, 1x1 m box + 2 internal walls, 1 024 Gaussian PlaceCells with the
reference's default wall geometry for that box (geodesic -> line_of_sight,
ratinabox/Neurons.py:922-928), dt = 10 ms, history + spikes on (reference defaults).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c2e|c3|c4]
                  [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); agents are sharded (weak scaling:
65 536 agents per GPU), there is no collective on the step path.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BOX_WALLS = [[[0.3, 0.0], [0.3, 0.5]], [[0.7, 1.0], [0.7, 0.5]]]       # SURVEY.md section 8(d)


def maze_walls(n=8, length=0.6):
    out = []
    for k in range(1, n + 1):
        x = k / (n + 1)
        out.append([[x, 0.0], [x, length]] if k % 2 else [[x, 1.0], [x, 1.0 - length]])
    return out


WORKLOADS = {
    # name: (agents per GPU, walls, population spec, description)
    "c2": dict(agents=65536, walls=BOX_WALLS, cells=("place", 1024, "line_of_sight"),
               desc="configs[1]: 65536 agents, box+2 walls, 1024 Gaussian PlaceCells (reference-default line_of_sight), dt=10ms"),
    "c2e": dict(agents=65536, walls=BOX_WALLS, cells=("place", 1024, "euclidean"),
                desc="configs[1] with wall_geometry='euclidean'"),
    "c3": dict(agents=65536, walls=[], cells=("grid", 1024, None),
               desc="configs[2]: 65536 agents, 1024 GridCells, box"),
    "c4": dict(agents=16384, walls=maze_walls(), cells=("bvc", 512, None),
               desc="configs[3]: 16384 agents, 512 BVCs, 8-wall maze (4 boundary + 8 internal)"),
    # configs[4] is a STRONG-scaling case: 262144 agents in total, divided over the ranks
    "c5": dict(agents=262144, strong=True, walls=BOX_WALLS,
               cells=[("place", 512, "line_of_sight"), ("grid", 512, None), ("bvc", 256, None)],
               desc="configs[4]: 262144 agents in total, 512 Place + 512 Grid + 256 BVC populations, box+2 walls"),
}


def cells_of(wl):
    c = wl["cells"]
    return list(c) if isinstance(c, list) else [c]


def agents_per_rank(wl, world):
    return wl["agents"] // world if wl.get("strong") else wl["agents"]


def synthetic_cells(kind, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "place":
        g = int(round(np.sqrt(n)))
        delta = 1.0 / g
        xs = np.linspace(delta / 2, 1 - delta / 2, g)
        c = np.array(np.meshgrid(xs, xs)).reshape(2, -1).T[:n]
        c = c + rng.uniform(-0.45 * delta, 0.45 * delta, c.shape)      # uniform_jitter (Environment.py:601-631)
        return dict(centres=c, widths=0.2 * np.ones(len(c)))
    if kind == "grid":
        return dict(gridscales=rng.uniform(0.2, 1.0, n), orientations=rng.uniform(0, np.pi / 3, n),
                    phase_offsets=rng.uniform(0, 2 * np.pi, (n, 2)))
    if kind == "bvc":
        mu_d = rng.uniform(0.05, 0.3, n)
        sg_t = rng.uniform(10, 30, n)                    # the reference's default angular spread (utils.py:1129-1131)
        if os.environ.get("RIAB_BENCH_BVC_SIGMA_DEG"):   # experiment: one narrow angular tuning for all cells
            sg_t = np.full(n, float(os.environ["RIAB_BENCH_BVC_SIGMA_DEG"]))
        return dict(mu_d=mu_d, sg_d=0.08 + mu_d / 12, mu_t=rng.uniform(0, 360, n), sg_t=sg_t)
    raise ValueError(kind)


def synthetic_agents(n, walls, seed):
    rng = np.random.default_rng(seed)
    pos = rng.uniform(0.02, 0.98, (n, 2))
    ang = rng.uniform(0, 2 * np.pi, n)
    vel = 0.08 * np.stack((np.cos(ang), np.sin(ang)), axis=1)
    return pos, vel


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed regions: one streaming
    `nvidia-smi -lms 50` process (per-call start-up would miss short regions)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self._p, self._t = index, [], None, None

    def _pump(self):
        try:
            for line in self._p.stdout:
                parts = [x.strip() for x in line.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
        except Exception:
            pass

    def start(self):
        try:
            self._p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                        "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE,
                                       stderr=subprocess.DEVNULL, text=True)
            self._t = threading.Thread(target=self._pump, daemon=True)
            self._t.start()
            time.sleep(0.3)            # let the first samples arrive before the timed region starts
            self.rows.clear()
        except Exception:
            self._p = None

    def stop(self):
        if self._p is not None:
            time.sleep(0.06)
            self._p.terminate()
            try:
                self._p.wait(timeout=5)
            except Exception:
                self._p.kill()
            if self._t:
                self._t.join(timeout=2)
        num = lambda x: x.replace(".", "", 1).isdigit()
        sm = [float(r[0]) for r in self.rows if num(r[0])]
        mx = [float(r[1]) for r in self.rows if num(r[1])]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------- CPU legs: the live reference (or its NumPy port)
def ref_population_specs(wl):
    """(kind, params, attrs) per population for oracle/ref_driver.build: the same synthetic cells as the GPU arm."""
    out = []
    for k, (kind, n, geom) in enumerate(cells_of(wl)):
        cp = synthetic_cells(kind, n, k)
        if kind == "place":
            out.append(("place", {"n": n, "place_cell_centres": cp["centres"], "widths": 0.2, "description": "gaussian",
                                  "wall_geometry": geom}, None))
        elif kind == "grid":
            out.append(("grid", {"n": n, "gridscale": cp["gridscales"], "orientation": cp["orientations"],
                                 "phase_offset": cp["phase_offsets"]}, None))
        else:
            out.append(("bvc", {"n": n}, {"tuning_distances": np.asarray(cp["mu_d"], float), "tuning_angles": np.radians(cp["mu_t"]),
                                          "sigma_distances": np.asarray(cp["sg_d"], float), "sigma_angles": np.radians(cp["sg_t"])}))
    return out


def cpu_kind():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_driver
    return "reference" if ref_driver.available() else "port"


_W = {}


def _cpu_worker_init(wl_name, kind):
    """One process = one reference-style Agent + populations stepped in a Python loop (how the reference runs:
    SURVEY.md section 3.1).  kind "reference": the unmodified RatInABox staged by oracle/make_ref.py; "port": the NumPy
    restatement oracle/riab_oracle.py (only when the staged reference is absent)."""
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[v] = "1"
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    wl = WORKLOADS[wl_name]
    seed = os.getpid() % 100003
    pos, vel = synthetic_agents(1, wl["walls"], seed)
    if kind == "reference":
        import ref_driver
        _, _, ag, pops = ref_driver.build(wl["walls"], ref_population_specs(wl), pos=pos[0], vel=vel[0], dt=0.01, seed=seed)
        _W["step"] = lambda n: ref_driver.step(ag, pops, n)
    else:
        import riab_oracle as O
        np.random.seed(seed)
        env = O.OracleEnvironment(walls=wl["walls"])
        ag = O.OracleAgent(env, pos[0], vel[0], {"dt": 0.01})
        rng = O.GlobalRNG()

        def population(kind_, n, geom, k):
            cp = synthetic_cells(kind_, n, k)
            if kind_ == "place":
                return O.OracleNeurons(ag, n, lambda p, r: O.place_cells_get_state(env, cp["centres"], cp["widths"], p, r,
                                                                                   "gaussian", geom))
            if kind_ == "grid":
                w = O.grid_cells_w(cp["orientations"])
                return O.OracleNeurons(ag, n, lambda p, r: O.grid_cells_get_state(cp["gridscales"], cp["phase_offsets"], w, p))
            return O.OracleNeurons(ag, n, lambda p, r: O.bvc_get_state(env, cp["mu_d"], np.radians(cp["mu_t"]), cp["sg_d"],
                                                                       np.radians(cp["sg_t"]), p, r))
        pops = [population(kind_, n, geom, k) for k, (kind_, n, geom) in enumerate(cells_of(wl))]

        def step(n):
            for _ in range(n):
                ag.update(rng)
                for ns in pops:
                    ns.update(rng)
        _W["step"] = step
    _W["step"](3)


def _cpu_worker_run(n):
    t0 = time.perf_counter()
    _W["step"](n)
    return n, time.perf_counter() - t0


def host_cores():
    """Usable host cores: the affinity mask capped by the cgroup CPU quota (containers on shared hosts)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


# agent-steps one worker runs per sample pass: ~0.5 .. 1 s of the reference per pass
CPU_STEPS_PER_PASS = {"c2": 400, "c2e": 500, "c3": 450, "c4": 70, "c5": 60}


# -------------------------------------------------------------------------------- main
def build_populations(rb, Ag, wl):
    return [build_population(rb, Ag, kind, n, geom, k) for k, (kind, n, geom) in enumerate(cells_of(wl))]


def build_population(rb, Ag, kind, n, geom, k=0):
    cp = synthetic_cells(kind, n, k)
    if kind == "place":
        return rb.PlaceCells(Ag, {"place_cell_centres": cp["centres"], "widths": 0.2, "description": "gaussian",
                                  "wall_geometry": geom})
    if kind == "grid":
        return rb.GridCells(Ag, {"gridscale": cp["gridscales"], "orientation": cp["orientations"],
                                 "phase_offset": cp["phase_offsets"]})
    # The reference's VectorCells declare `angular_spread` in default_params but hand **params to
    # utils.create_random_assembly, which reads `sigma_angle` (ratinabox/Neurons.py:1315 vs utils.py:1124-1131): a
    # `sigma_angle` key works but warns, an `angular_spread` key is silently ignored.  The tuning is therefore set the way
    # the reference tells its users to (Neurons.py:1612): by assigning the arrays after construction.
    B = rb.BoundaryVectorCells(Ag, {"n": n})
    B.tuning_distances, B.tuning_angles = np.asarray(cp["mu_d"], float), np.radians(cp["mu_t"])
    B.sigma_distances, B.sigma_angles = np.asarray(cp["sg_d"], float), np.radians(cp["sg_t"])
    return B


def algorithmic_bytes_per_agent_step(n_cells, spikes):
    """DESIGN.md 'bytes per unit': float64 state in+out (12 doubles each), float32 agent
    history row (8), one float32 write per rate, bit-packed spikes."""
    return 2 * 12 * 8 + 8 * 4 + 4 * n_cells + (n_cells // 8 if spikes else 0)


DUMP_BYTES = 60_000_000           # all arrays together, .npy headers aside: under 64 MB
DUMP_STATE = ("pos", "velocity", "rotational_velocity", "measured_velocity", "measured_rotational_velocity", "head_direction",
              "distance_travelled", "distance_to_closest_wall")


def dump_outputs(out_dir, Ag, pops, spikes):
    """What a caller of Agent.run() receives after its last step, as <out_dir>/<name>.npy: the Agent's state (float64) and,
    per population k, that step's firing rates (rates_<k>, float32) and spikes (spikes_<k>, 0 / 1 as float32).  Arrays of
    every agent while they fit in DUMP_BYTES, else the rows of a fixed seeded sample of agents (agent_rows.npy)."""
    import torch
    from ratinabox_b200.Neurons import _unpack_spikes
    os.makedirs(out_dir, exist_ok=True)
    A = Ag.n_agents
    state = {name: Ag.state_view(name) for name in DUMP_STATE}          # (A, ...) float64, read-only views
    per_agent = 8 * (1 + sum(v[0].size for v in state.values())) + 4 * sum(ns.n for ns in pops) * (2 if spikes else 1)
    n_rows = min(A, DUMP_BYTES // per_agent)
    rows = np.arange(A) if n_rows == A else np.sort(np.random.default_rng(0).choice(A, n_rows, replace=False))
    idx = torch.as_tensor(rows, device=Ag.device)
    out = {"agent_rows": rows.astype(np.float64)}
    for name, v in state.items():
        out[name] = np.array(v[rows], dtype=np.float64)
    for k, ns in enumerate(pops):
        out[f"rates_{k}"] = ns._hist[ns._last_slot][idx, : ns.n].cpu().numpy()
        if spikes:
            out[f"spikes_{k}"] = _unpack_spikes(ns._spk[ns._last_slot][idx].cpu().numpy(), ns.n).astype(np.float32)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), arr)


def measure(rb, lib, torch, dist, name, steps, warmup, rank, world, local_rank, spikes=True, total_agents=None, e2e=True,
            keep=False, dump=None):
    """Device-resident throughput (riab_run, CUDA events, max over ranks) and the stepped-API e2e number of one workload.
    total_agents: strong-scaling variant (that many agents in total, split over the ranks).  dump: directory that receives
    rank 0's outputs of the last timed step (dump_outputs)."""
    wl = WORKLOADS[name]
    if total_agents is not None:
        A, scaling = total_agents // world, "strong"
    else:
        A, scaling = agents_per_rank(wl, world), ("strong" if wl.get("strong") else "weak")
    cl = cells_of(wl)
    n_cells = sum(n for _, n, _ in cl)
    np.random.seed(1234 + rank)
    Env = rb.Environment()
    for w in wl["walls"]:
        Env.add_wall(w)
    Ag = rb.Agent(Env, {"dt": 0.01, "n_agents": A, "seed": 7, "id_offset": rank * A,
                        "fused_step": os.environ.get("RIAB_BENCH_FUSED_STEP") == "1"})
    pos, vel = synthetic_agents(A, wl["walls"], 100 + rank)
    Ag.pos, Ag.velocity = pos, vel
    Ag.measured_velocity = vel
    pops = build_populations(rb, Ag, wl)
    if not spikes:
        for ns in pops:
            ns.save_spikes = False

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    Ag.run(warmup)
    barrier()
    l0 = lib.riab_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    Ag.run(steps)
    ev1.record()
    barrier()
    launches = lib.riab_launch_count() - l0
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    if dump is not None and rank == 0:
        dump_outputs(dump, Ag, pops, spikes)
    res = {"agents_per_gpu": A, "agents_total": A * world, "n_cells": n_cells, "scaling": scaling, "steps": steps,
           "ms_per_step": ms / steps, "value": world * A * steps / (ms * 1e-3), "gpu_launches": int(launches)}
    bytes_unit = algorithmic_bytes_per_agent_step(n_cells, spikes)
    res["bytes_per_agent_step"] = bytes_unit
    res["achieved_gbs"] = bytes_unit * A / (ms / steps * 1e-3) / 1e9
    n_bvc = sum(n for k, n, _ in cl if k == "bvc")
    if n_bvc:
        res["ex2_per_step"] = A * n_bvc * 180
    if e2e:
        # the Python API with HOST buffers each step (drift in, positions out)
        e2e_steps = max(10, min(steps, 500))
        drift = (0.05 * torch.randn((A, 2), dtype=torch.float64)).pin_memory()       # a policy's velocity commands
        for _ in range(3):
            Ag.update(drift_velocity=drift)
            for ns in pops:
                ns.update()
            _ = Ag.state_view("pos")
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            Ag.update(drift_velocity=drift)          # H2D: A*2*8 B read from pinned host memory by the motion kernel, every step
            for ns in pops:
                ns.update()                          # rates of every population at the new positions
            p = Ag.state_view("pos")                 # D2H: A*2*8 B posted to pinned host memory by the motion kernel; blocks until
                                                     # the whole step has finished (`Ag.pos` = a private copy of it)
        barrier()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        res["e2e"] = {"value": world * A * e2e_steps / e2e_s, "unit": "agent-steps/s", "h2d_bytes_per_step": A * 16,
                      "d2h_bytes_per_step": A * 16, "steps": e2e_steps,
                      "api": "Agent.update(drift_velocity=<pinned host tensor>) + Neurons.update() + Agent.state_view('pos') "
                             "(host positions), per step; the rates stay in the device history ring (268 MB/step at c2 cannot "
                             "cross PCIe)"}
    if keep:
        res["_objects"] = (Env, Ag, pops)
    else:
        del pops, Ag, Env
        import gc
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    return res


def gather_check(torch, dist, Ag, pops, rank, world):
    """The one collective of the design: all_gather of a history slab (here the last rate row of population 0 and the
    positions) over NCCL.  Device-timed, and rank 0 re-evaluates a sample of ANOTHER rank's rows from the gathered positions
    on its own GPU: the gathered rates must equal them bit for bit (same kernels, same cell parameters, same positions)."""
    from ratinabox_b200.distributed import gather_agent_axis
    ns = pops[0]
    A = Ag.n_agents
    row = ns._hist[ns._last_slot]                               # (A, ld) float32, the step's rates
    pos = Ag._s["pos"]
    gather_agent_axis(row[:64], 64 * world, axis=0, dst=0)      # untimed: NCCL sets its channels up on the first collective
    torch.cuda.synchronize(); dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    full = gather_agent_axis(row, A * world, axis=0, dst=0)
    ev1.record()
    torch.cuda.synchronize()
    t = torch.tensor([ev0.elapsed_time(ev1)], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    allpos = gather_agent_axis(pos, A * world, axis=0, dst=0)
    out = {"what": f"all_gather of the last rate row ({row.numel() * 4 / 1e6:.0f} MB per rank) to every rank, NCCL",
           "ms": ms, "bytes_received_per_rank": int(row.numel() * 4 * (world - 1)),
           "gbs_per_rank": row.numel() * 4 * (world - 1) / (ms * 1e-3) / 1e9}
    if rank == 0:
        other, n_chk = world - 1, min(A, 2048)
        lo = other * A
        again = ns.get_state(evaluate_at=None, pos=allpos[lo:lo + n_chk], return_tensor=True)
        got = full[lo:lo + n_chk, : ns.n]
        out["rows_checked"] = int(n_chk)
        out["equal_to_local_recompute"] = bool(torch.equal(again, got))
        out["own_shard_equal"] = bool(torch.equal(full[:A], row))
    return out


def reference_arm(args, config, scaling, A_rank, world):
    """`--impl reference`: the reference's own CPU implementation on all usable host cores (rank 0 only).  One "step" of this
    arm = one bounded sample pass: every worker process steps its own reference Agent CPU_STEPS_PER_PASS times."""
    kind = cpu_kind()
    cores = host_cores()
    per = CPU_STEPS_PER_PASS[args.workload]
    ctx = mp.get_context("spawn")
    t_all = time.perf_counter()
    with ctx.Pool(cores, initializer=_cpu_worker_init, initargs=(args.workload, kind)) as pool:
        for _ in range(max(1, args.warmup)):
            pool.map(_cpu_worker_run, [max(5, per // 10)] * cores)
        passes = []
        for _ in range(max(1, args.steps)):
            t0 = time.perf_counter()
            res = pool.map(_cpu_worker_run, [per] * cores)
            passes.append((sum(r[0] for r in res), time.perf_counter() - t0))
    n_steps = sum(p[0] for p in passes)
    secs = sum(p[1] for p in passes)
    value = n_steps / secs
    what = ("the unmodified RatInABox reference (oracle/_ref, staged by oracle/make_ref.py; matplotlib / shapely stand-ins from "
            "oracle/ref_shim.py)" if kind == "reference" else "the NumPy port oracle/riab_oracle.py (the staged reference is absent)")
    sample = f"{cores} processes x 1 agent x {per} agent-steps per pass, {len(passes)} timed passes of {what}"
    line = {"impl": "reference", "metric": "agent-steps/sec", "value": value, "unit": "agent-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * secs / len(passes), "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "step_definition": "one sample pass (see cpu_baseline.sample); value = agent-steps of all passes / their wall time",
            "wall_s": time.perf_counter() - t_all}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-spikes", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the `workloads` / `strong` / `gather` objects")
    ap.add_argument("--agents", type=int, default=None,
                    help="experiments only: agents per GPU instead of the workload's (the line's config says so)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed run computed in its last step to DIR/<name>.npy (agent state, rates, spikes)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.agents is not None:                          # experiment: same workload at another batch size
        w0 = WORKLOADS[args.workload]
        WORKLOADS[args.workload] = dict(w0, agents=args.agents, desc=w0["desc"] + f" [--agents {args.agents}: NOT the configuration]")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cl = cells_of(wl)
    n_cells = sum(n for _, n, _ in cl)
    kind = "+".join(k for k, _, _ in cl)
    geom = cl[0][2]
    A_rank = agents_per_rank(wl, world)
    scaling = "strong" if wl.get("strong") else "weak"
    config = {"workload": f"{args.workload}: {wl['desc']}", "agents_per_gpu": A_rank, "n_cells": n_cells,
              "cells": kind, "wall_geometry": geom, "n_walls": 4 + len(wl["walls"]), "dt": 0.01,
              "spikes": not args.no_spikes,
              "spike_stream": (None if args.no_spikes else
                               {"place": "dense Philox4x32-7 stream in the pair loop", "grid": "thinned (Binomial candidates per 128-cell block)",
                                "bvc": "dense, in the integration kernel's epilogue"}.get(kind, "per population: place dense / grid thinned / bvc dense")),
              "history": "device rings (rates: last rows within 8 GiB; agent rows: all)",
              "l2": "each step writes >= 2x L2 of fresh rate rows (inputs larger than L2)",
              "parallelism": f"agents sharded x{world}, no step-path collective"}

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, config, scaling, A_rank, world)
        return

    # ----------------------------------------------------------------------- our arm
    import torch
    import ratinabox_b200 as rb
    from ratinabox_b200 import _lib
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.load()
    spikes = not args.no_spikes
    sampler = ClockSampler(local_rank)
    sampler.start()
    head = measure(rb, lib, torch, dist, args.workload, args.steps, args.warmup, rank, world, local_rank, spikes=spikes,
                   keep=(world > 1 and not args.no_extra), dump=args.dump_outputs)
    clocks = sampler.stop()        # sampled across the device-resident and the e2e timed regions of the headline workload
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json (measured)" if peaks else "fallback 6650 GB/s"
    sm_mhz = clocks.get("sm_mhz") or 1965.0

    def roofline_of(name, r):
        rf = {"bound": "hbm", "achieved": r["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": r["achieved_gbs"] / peak,
              "traffic": None, "peak_source": peak_src, "bytes_per_agent_step": r["bytes_per_agent_step"],
              "kernel_ms": r["ms_per_step"]}
        if "ex2_per_step" in r:
            # BoundaryVectorCells are bound by the special-function unit, not by HBM: one ex2 per (agent, cell, test angle)
            # in the angular integral (T = 180) against 16 MUFU results per clock per SM (148 SMs at the sampled SM clock)
            ex2 = r["ex2_per_step"] / (r["ms_per_step"] * 1e-3)
            peak_ex2 = 148 * 16 * sm_mhz * 1e6
            rf["mufu"] = {"achieved_ex2_per_s": ex2, "peak_ex2_per_s": peak_ex2, "frac": ex2 / peak_ex2,
                          "note": "share of the whole step (motion, rays, other populations included) spent at the ex2 rate"}
        prof = os.path.join(ROOT, "profiles", f"traffic_{name}.json")
        if os.path.exists(prof):
            try:
                t = json.load(open(prof))
                rf["traffic"] = t.get("dram_bytes_per_step")
                rf["traffic_source"] = t.get("source")
            except Exception:
                pass
        return rf

    extra = {}
    if not args.no_extra:
        # every other BASELINE.json config so that the driver's one line carries them (100 steps for the whole-run
        # single-population workloads, whose one launch per run pays ~50 us of ramp; 20 for the millisecond steps)
        wls = {}
        for name in ("c2e", "c3", "c4", "c5"):
            if name == args.workload:
                continue
            r = measure(rb, lib, torch, dist, name, 100 if name in ("c2e", "c3") else 20, 5, rank, world, local_rank, spikes=spikes)
            wls[name] = {"workload": WORKLOADS[name]["desc"], "agents_per_gpu": r["agents_per_gpu"], "scaling": r["scaling"],
                         "ms_per_step": r["ms_per_step"], "value": r["value"], "unit": "agent-steps/s", "steps": r["steps"],
                         "gpu_launches": r["gpu_launches"], "roofline": roofline_of(name, r), "e2e": r["e2e"]}
        extra["workloads"] = wls
        if world > 1:
            # strong scaling of the headline workload: configs[1]'s 65 536 agents IN TOTAL (north_star's 8-GPU target)
            r = measure(rb, lib, torch, dist, "c2", 200, 10, rank, world, local_rank, spikes=spikes, total_agents=65536)
            extra["strong"] = {"c2": {"agents_total": 65536, "agents_per_gpu": r["agents_per_gpu"], "ms_per_step": r["ms_per_step"],
                                      "value": r["value"], "unit": "agent-steps/s", "steps": r["steps"], "e2e": r["e2e"],
                                      "note": "efficiency = value(N) / (N * value(1) of the same 65 536-agent job): divide by the "
                                              "N=1 headline value"},
                               "c5": {"agents_total": 262144, "see": "workloads.c5 (configs[4] is a strong-scaling job)"}}
            Env, Ag, pops = head.pop("_objects")
            extra["gather"] = gather_check(torch, dist, Ag, pops, rank, world)
            del pops, Ag, Env
    head.pop("_objects", None)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:          # a reported baseline, timed at N=1 only
        kind_cpu = cpu_kind()
        per = 36 * CPU_STEPS_PER_PASS[args.workload]         # ~12 s of CPU work on the GPU box's host (bounded sample)
        _cpu_worker_init(args.workload, kind_cpu)
        n, secs = _cpu_worker_run(per)
        cpu_baseline = {"value": n / secs, "unit": "agent-steps/s", "cores": 1, "kind": kind_cpu,
                        "sample": f"1 agent x {per} steps of " + ("the unmodified RatInABox reference (oracle/_ref)" if kind_cpu == "reference"
                                                                  else "oracle/riab_oracle.py (NumPy port)") + f", {secs:.1f} s"}
    line = {"metric": "agent-steps/sec", "value": head["value"], "unit": "agent-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32 rates / f64 agent state", "data": "synthetic", "config": config,
            "clocks": clocks, "e2e": head["e2e"], "gpu_launches": head["gpu_launches"],
            "roofline": roofline_of(args.workload, head), "cpu_baseline": cpu_baseline}
    line.update(extra)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
