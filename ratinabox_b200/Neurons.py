"""Host mirror of ``ratinabox.Neurons`` for PlaceCells, GridCells and allocentric
BoundaryVectorCells: ``update()`` and ``get_state()`` run on the GPU through
libriab_b200 (C ABI: include/riab_b200.h).

API parity (ratinabox/Neurons.py): ``Neurons(Agent, params)`` registers itself in
``Agent.Neurons`` (:111-112); ``update(**kwargs)`` (:145-171) refreshes
``firingrate`` (OU noise + ``get_state`` + optional spikes) and appends to
``history`` (``t``, ``firingrate``, ``spikes``; :681-687); ``get_state(evaluate_at=
"agent"|"all"|None, pos=...)`` returns ``(n_cells, n_pos)`` like the reference.
Parameter arrays (``place_cell_centres``, ``gridscales`` ...) are plain NumPy
attributes the user may overwrite or mutate between steps
(tests/test_advanced.py:59): they are re-packed when their bytes change.

With ``n_agents > 1`` ``firingrate`` is ``(n_agents, n)`` and history arrays are
``(steps, n_agents, n)``.  Rates are float32 on the device (history rows double as
the step's output: one write per rate).
"""
import copy
import ctypes as C
import warnings

import numpy as np

from . import _lib
from .Agent import _HistoryView


def _f64p(a):
    return a.ctypes.data_as(_lib.c_double_p)


def _unpack_spikes(words, n):
    """Spike words (..., W) int32 of the device rings -> (..., n) bool."""
    lead = words.shape[:-1]
    bits = np.unpackbits(words.view(np.uint8), axis=-1, bitorder="little")
    # bit L of word 4B+i = cell 128B + 4L + i  (one warp ballot per cell slot i)
    bits = bits.reshape(*lead, -1, 4, 32).swapaxes(-1, -2).reshape(*lead, -1)
    return bits[..., :n].astype(bool)


class Neurons:
    default_params = {                                              # ratinabox/Neurons.py:90-99
        "n": 10,
        "name": "Neurons",
        "color": None,
        "noise_std": 0,
        "noise_coherence_time": 0.5,
        "min_fr": 0.0,
        "max_fr": 1.0,
        "save_history": True,
        # ---- batch-engine additions
        "save_spikes": True,          # the reference draws spikes whenever save_history is True (:681-684)
        "history_bytes_limit": 8 << 30,
    }
    _cells_kind = None

    def __init__(self, Agent, params={}):
        import torch
        self._lib = _lib.load()
        self.Agent = Agent
        self.Agent.Neurons.append(self)
        self._population_id = len(self.Agent.Neurons) - 1
        all_defaults = {}
        for cls in reversed(type(self).__mro__):                    # utils.collect_all_params, utils.py:821-874
            all_defaults.update(getattr(cls, "default_params", {}))
        unexpected = [k for k in params if k not in all_defaults]
        if unexpected:
            warnings.warn(f"Found {len(unexpected)} unexpected params key(s) while initializing "
                          f"{type(self).__name__}: {unexpected}")
        self.params = copy.deepcopy(all_defaults)
        self.params.update(params)
        for k, v in self.params.items():
            setattr(self, k, v)
        self.device = Agent.device
        self._torch = torch
        self._sig = None
        self._packed = None
        self._keep = []
        self._hist = None
        self._hist_cap = 0
        self._hist_rows = 0
        self._spk = None
        self._noise = None
        self._t_hist = []
        self._last_slot = None
        self._upd = 0              # updates of THIS population so far: keys its OU-noise / spike Philox streams
        self._history_view = _HistoryView(self)
        self._last_history_array_cache_time = None
        self._history_arrays = {}
        self._out = _lib.RatesOut()
        self._nz = _lib.NeuronNoise()
        self.colormap = "inferno"

    # ---------------------------------------------------------------- subclass API
    def _signature(self):
        raise NotImplementedError

    def _pack(self):
        """(re)build the device parameter block + C struct; returns the struct."""
        raise NotImplementedError

    def _cells(self):
        sig = self._signature()
        if sig != self._sig:
            self._cstruct = self._pack()
            self._sig = sig
        return self._cstruct

    def _rates_from_positions(self, pos_dev, n_pos, out):
        raise NotImplementedError

    # ------------------------------------------------------------------- helpers
    def _ld(self):
        return (self.n + 3) // 4 * 4

    def _upload(self, host, dtype=None):
        t = self._torch.as_tensor(np.ascontiguousarray(host), device=self.device)
        return t

    def _row_buffers(self):
        """Next history row (rates [+ spikes]) on the device; grows / wraps like Agent's ring."""
        torch = self._torch
        A, ld = self.Agent.n_agents, self._ld()
        words = 4 * ((self.n + 127) // 128)           # 4 ballot words per 128 cells (riab_b200.h, riab_rates_out)
        row_bytes = A * ld * 4
        if self._hist is None:
            cap = int(max(1, min(256, self.history_bytes_limit // row_bytes))) if self.save_history else 1
            self._hist = torch.empty((cap, A, ld), dtype=torch.float32, device=self.device)
            self._spk = torch.zeros((cap, A, words), dtype=torch.int32, device=self.device)
            self._hist_cap = cap
        elif self.save_history and self._hist_rows == self._hist_cap and 2 * self._hist_cap * row_bytes <= self.history_bytes_limit:
            cap = self._hist_cap
            new = torch.empty((2 * cap, A, ld), dtype=torch.float32, device=self.device)
            new[:cap].copy_(self._hist)
            spk = torch.zeros((2 * cap, A, words), dtype=torch.int32, device=self.device)
            spk[:cap].copy_(self._spk)
            self._hist, self._spk, self._hist_cap = new, spk, 2 * cap
        slot = self._hist_rows % self._hist_cap
        self._hist_rows += 1
        self._last_slot = slot
        # raw pointers of the slot (no tensor views on the per-step path)
        return (self._hist.data_ptr() + slot * row_bytes, self._spk.data_ptr() + slot * A * words * 4)

    def _reserve_history(self, n_more):
        """Grow the ring (within history_bytes_limit) so n_more further rows fit without wrapping if possible."""
        torch = self._torch
        A, ld = self.Agent.n_agents, self._ld()
        words = 4 * ((self.n + 127) // 128)           # 4 ballot words per 128 cells (riab_b200.h, riab_rates_out)
        row_bytes = A * ld * 4
        limit_rows = max(1, self.history_bytes_limit // row_bytes)
        need = self._hist_rows + n_more if self.save_history else 1
        if self._hist is None:
            cap = int(max(1, min(max(256, need), limit_rows))) if self.save_history else 1
            self._hist = torch.empty((cap, A, ld), dtype=torch.float32, device=self.device)
            self._spk = torch.zeros((cap, A, words), dtype=torch.int32, device=self.device)
            self._hist_cap = cap
        elif need > self._hist_cap and self._hist_rows <= self._hist_cap:
            cap = int(min(max(need, 2 * self._hist_cap), limit_rows))
            if cap > self._hist_cap:
                new = torch.empty((cap, A, ld), dtype=torch.float32, device=self.device)
                new[: self._hist_cap].copy_(self._hist)
                spk = torch.zeros((cap, A, words), dtype=torch.int32, device=self.device)
                spk[: self._hist_cap].copy_(self._spk)
                self._hist, self._spk, self._hist_cap = new, spk, cap

    # -------------------------------------------------------------------- update
    def _fill_out_structs(self, row, spk):
        ag = self.Agent
        out, nz = self._out, self._nz
        out.rates_row = row
        out.ld = self._ld()
        want_spikes = bool(self.save_history and self.save_spikes)
        out.spikes_row = spk if (want_spikes and spk is not None) else None
        out.noise_state = None
        if self.noise_std != 0:
            if self._noise is None:
                self._noise = self._torch.zeros((ag.n_agents, self._ld()), dtype=self._torch.float32, device=self.device)
            out.noise_state = self._noise.data_ptr()
        out.bvc_scratch = self._scratch_ptr(ag.n_agents)
        nz.noise_std = float(self.noise_std)
        nz.noise_coherence_time = float(self.noise_coherence_time)
        nz.dt = float(ag.dt)
        nz.seed = int(ag.seed) & 0xFFFFFFFFFFFFFFFF
        nz.step = self._upd
        nz.id_offset = int(ag.id_offset)
        nz.population_id = self._population_id
        return out, nz

    def update(self, **kwargs):
        """Neurons.update (ratinabox/Neurons.py:145-171)."""
        ag = self.Agent
        cells = self._cells()
        ag._sync_user_writes()                 # in-place edits of Ag.pos etc. since they were read
        saved = (self._hist_rows, self._last_slot)
        row, spk = self._row_buffers()
        out, nz = self._fill_out_structs(row, spk)
        fused = ag._take_pending()
        try:
            if fused:
                _lib.check(self._lib.riab_step_fused(C.byref(ag._agents_c), C.byref(ag._env_struct()), C.byref(ag._mp),
                                                     C.byref(ag._io), self._cells_kind, C.byref(cells), C.byref(nz),
                                                     C.byref(out), ag._stream()))
            else:
                self._update_unfused(cells, out, nz)
        except Exception:
            # the library refused the call (validation): nothing ran -- keep the queued motion step and the ring as they were
            self._hist_rows, self._last_slot = saved
            if fused:
                ag._pending = True
            raise
        self._upd += 1
        if self.save_history:
            self._t_hist.append(ag.t)

    def _update_unfused(self, cells, out, nz):
        """Rates for the agents' current positions (no queued motion step to fuse with)."""
        ag = self.Agent
        _lib.check(self._lib.riab_neurons_update(C.byref(ag._agents_c), C.byref(ag._env_struct()), self._cells_kind,
                                                 C.byref(cells), C.byref(nz), C.byref(out), ag._stream()))

    def _scratch_ptr(self, n):
        return None

    # ----------------------------------------------------------------- get_state
    def get_state(self, evaluate_at="agent", **kwargs):
        """(n_cells, n_pos) firing rates, float64 NumPy (pass ``return_tensor=True``
        for the (n_pos, n_cells) float32 device tensor)."""
        torch = self._torch
        self._cells()
        if evaluate_at == "agent":
            self.Agent._flush_pending()
            self.Agent._sync_user_writes()
            pos_dev = self.Agent._s["pos"]
        else:
            pos = self.Agent.Environment.flattened_discrete_coords if evaluate_at == "all" else kwargs["pos"]
            if isinstance(pos, torch.Tensor):
                pos_dev = pos.to(device=self.device, dtype=torch.float64).reshape(-1, 2).contiguous()
            else:
                pos_dev = torch.as_tensor(np.ascontiguousarray(np.asarray(pos, dtype=np.float64).reshape(-1, 2)),
                                          device=self.device)
        n_pos = int(pos_dev.shape[0])
        out = torch.empty((n_pos, self._ld()), dtype=torch.float32, device=self.device)
        self._rates_from_positions(pos_dev, n_pos, out)
        if kwargs.get("return_tensor", False):
            return out[:, : self.n]
        return out[:, : self.n].T.contiguous().cpu().numpy().astype(np.float64)

    # ------------------------------------------------------------------ firingrate
    @property
    def firingrate(self):
        if self._last_slot is None:
            return np.zeros(self.n)
        r = self._hist[self._last_slot][:, : self.n].cpu().numpy().astype(np.float64)
        return r[0] if self.Agent.n_agents == 1 else r

    # --------------------------------------------------------------------- history
    def _history_keys(self):
        return ["t", "firingrate", "spikes"]

    @property
    def history(self):
        return self._history_view

    def get_history_arrays(self):                                   # Neurons.py:812-821
        key = (self.Agent.t, self._hist_rows)
        if self._last_history_array_cache_time != key:
            self._last_history_array_cache_time = key
            torch = self._torch
            n = min(self._hist_rows, self._hist_cap) if self.save_history else 0
            A = self.Agent.n_agents
            if n == 0:
                fr = np.zeros((0, A, self.n))
                sp = np.zeros((0, A, self.n), dtype=bool)
            else:
                start = self._hist_rows % self._hist_cap if self._hist_rows > self._hist_cap else 0
                idx = (torch.arange(n, device=self.device) + start) % self._hist_cap
                fr = self._hist[idx][:, :, : self.n].cpu().numpy().astype(np.float64)
                sp = _unpack_spikes(self._spk[idx].cpu().numpy(), self.n)
            if A == 1:
                fr, sp = fr[:, 0], sp[:, 0]
            self.history_dropped = self._hist_rows - n
            self._history_arrays = {"t": np.array(self._t_hist[len(self._t_hist) - n:]), "firingrate": fr, "spikes": sp}
        return self._history_arrays

    def get_history_rate_maps(self, dx=None, return_zero_bins=False):
        """Rate maps from the history, the data of ``plot_rate_map(method="history")`` (Neurons.py:470-490): for every
        cell ``utils.bin_data_for_histogramming(pos, extent, dx, weights=rate, norm_by_bincount=True)`` over the history of
        ALL agents, binned on the device (riab_history_rate_maps).  Returns (n_cells, ny, nx) [and the empty-bin mask]."""
        count, ssum = self.Agent._history_maps(dx, neurons=self)
        zero = (count == 0)
        c = count.copy()
        c[zero] = 1
        maps = (ssum / c[:, :, None]).transpose(2, 1, 0)[:, ::-1, :]            # per cell: heatmap.T[::-1, :]
        if return_zero_bins:
            return maps, zero.T[::-1, :]
        return maps

    def reset_history(self):                                        # Neurons.py:689-692
        self._hist_rows = 0
        self._t_hist = []
        self._last_history_array_cache_time = None


# =============================================================================
class PlaceCells(Neurons):
    default_params = {                                              # ratinabox/Neurons.py:857-867
        "n": 10,
        "name": "PlaceCells",
        "description": "gaussian",
        "widths": 0.20,
        "place_cell_centres": None,
        "wall_geometry": "geodesic",
        "min_fr": 0,
        "max_fr": 1,
    }
    _cells_kind = _lib.CELLS_PLACE

    def __init__(self, Agent, params={}):
        params = dict(params)
        p = copy.deepcopy(__class__.default_params)
        p.update(params)
        env = Agent.Environment
        if p["place_cell_centres"] is None:                         # Neurons.py:881-901
            p["place_cell_centres"] = env.sample_positions(n=p["n"], method="uniform_jitter")
        elif type(p["place_cell_centres"]) is str:
            if p["place_cell_centres"] in ["random", "uniform", "uniform_jitter"]:
                p["place_cell_centres"] = env.sample_positions(n=p["n"], method=p["place_cell_centres"])
            else:
                raise ValueError("self.params['place_cell_centres'] must be None, an array of locations or one of "
                                 "the instructions ['random', 'uniform', 'uniform_jitter']")
        else:
            p["place_cell_centres"] = np.array(p["place_cell_centres"], dtype=float)
            p["n"] = p["place_cell_centres"].shape[0]
        params["place_cell_centres"], params["n"] = p["place_cell_centres"], p["n"]
        super().__init__(Agent, params)
        self.place_cell_widths = self.widths * np.ones(self.n)
        if self.description not in _lib.PC_DESCRIPTIONS:
            raise ValueError(f"unknown PlaceCells description {self.description!r}")
        if self.wall_geometry in ("line_of_sight", "geodesic") and env.boundary_conditions == "periodic":   # Neurons.py:907-921
            print(f"{self.wall_geometry} wall geometry only possible in 2D when the boundary conditions are solid. "
                  "Using 'euclidean' instead.")
            self.wall_geometry = "euclidean"
        if (self.wall_geometry == "geodesic") and (len(env.walls) > 5):   # Neurons.py:922-928
            print("'geodesic' wall geometry only supported for enivironments with 1 additional wall "
                  "(4 bounding walls + 1 additional). Sorry. Using 'line_of_sight' instead.")
            self.wall_geometry = "line_of_sight"

    def _effective_geometry(self):
        n_inner = len(self.Agent.Environment.walls) - self.Agent.Environment.los_skip
        if self.wall_geometry not in _lib.WALL_GEOMETRIES:
            raise ValueError(f"unknown wall_geometry {self.wall_geometry!r}")
        if self.wall_geometry == "geodesic":
            if self.Agent.Environment.is_polygonal:
                raise NotImplementedError("geodesic distances in polygon / holed environments are outside the CUDA hot path")
            assert n_inner <= 1, ("unfortunately geodesic geometry is only defined in closed rooms with one "
                                  "additional wall (Environment.py:736-739)")
        if n_inner == 0:
            return "euclidean"          # line_of_sight / geodesic without inner walls are plain distances
        return self.wall_geometry

    def _signature(self):
        env = self.Agent.Environment
        return (np.ascontiguousarray(self.place_cell_centres, dtype=np.float64).tobytes(),
                np.ascontiguousarray(self.place_cell_widths, dtype=np.float64).tobytes(),
                env._walls_signature(), self.description, self.wall_geometry, float(self.min_fr), float(self.max_fr),
                float(self.widths) if np.isscalar(self.widths) else None, self.n)

    def _pack(self):
        env = self.Agent.Environment
        centres = np.ascontiguousarray(self.place_cell_centres, dtype=np.float64).reshape(-1, 2)
        widths = np.ascontiguousarray(self.place_cell_widths, dtype=np.float64).reshape(-1)
        self.n = centres.shape[0]
        assert widths.shape[0] == self.n
        geom = _lib.WALL_GEOMETRIES[self._effective_geometry()]
        walls = np.ascontiguousarray(env.walls, dtype=np.float64)
        n_inner = 0 if geom == 0 else walls.shape[0] - env.los_skip
        c = _lib.PlaceCells()
        nfl = self._lib.riab_place_pack_floats(self.n, n_inner)
        host = np.zeros(nfl, dtype=np.float32)
        ext = np.ascontiguousarray(env.extent, dtype=np.float64)
        _lib.check(self._lib.riab_place_pack(_f64p(centres), _f64p(widths), self.n, _f64p(walls), walls.shape[0],
                                             env.los_skip, _f64p(ext), geom, C.byref(c),
                                             host.ctypes.data_as(_lib.c_float_p)))
        self._packed = self._upload(host)
        self._centres_dev = self._upload(centres)
        c.n_cells, c.description, c.wall_geometry = self.n, _lib.PC_DESCRIPTIONS[self.description], geom
        c.min_fr, c.max_fr = float(self.min_fr), float(self.max_fr)
        c.top_hat_width = float(self.widths) if np.isscalar(self.widths) else float(np.asarray(self.widths).reshape(-1)[0])
        c.packed_dev, c.centres_dev = self._packed.data_ptr(), self._centres_dev.data_ptr()
        return c

    def _rates_from_positions(self, pos_dev, n_pos, out):
        ag = self.Agent
        _lib.check(self._lib.riab_place_rates(pos_dev.data_ptr(), n_pos, C.byref(ag._env_struct()),
                                              C.byref(self._cells()), out.data_ptr(), out.stride(0), ag._stream()))


# =============================================================================
class GridCells(Neurons):
    default_params = {                                              # ratinabox/Neurons.py:1055-1068
        "n": 30,
        "gridscale_distribution": "modules",
        "gridscale": (0.3, 0.5, 0.8),
        "orientation_distribution": "modules",
        "orientation": (0, 0.1, 0.2),
        "phase_offset_distribution": "uniform",
        "phase_offset": (0, 2 * np.pi),
        "description": "rectified_cosines",
        "width_ratio": 4 / (3 * np.sqrt(3)),
        "min_fr": 0,
        "max_fr": 1,
        "name": "GridCells",
    }
    _cells_kind = _lib.CELLS_GRID

    def __init__(self, Agent, params={}):
        from .utils import distribution_sampler, rotate
        params = dict(params)
        p = copy.deepcopy(__class__.default_params)
        p.update(params)
        if p["description"] in ("three_rectified_cosines", "three_shifted_cosines"):   # Neurons.py:1091-1095
            p["description"] = p["description"][6:]
            params["description"] = p["description"]
        if type(p["gridscale"]) in (list, np.ndarray):              # Neurons.py:1098-1113
            gridscales = np.array(p["gridscale"], dtype=float)
            p["n"] = len(gridscales)
        else:
            gridscales = distribution_sampler(p["gridscale_distribution"], p["gridscale"], (p["n"],))
        params["n"] = p["n"]
        super().__init__(Agent, params)
        self.gridscales = gridscales
        if type(self.params["phase_offset"]) in (list, np.ndarray) and np.array(self.params["phase_offset"]).ndim == 2:
            self.phase_offsets = np.array(self.params["phase_offset"], dtype=float)
            assert len(self.phase_offsets) == self.n, "number of phase offsets supplied incompatible with number of neurons"
        else:
            if self.params["phase_offset_distribution"] == "grid":
                raise NotImplementedError("phase_offset_distribution='grid' is host set-up outside the hot path")
            self.phase_offsets = distribution_sampler(self.params["phase_offset_distribution"],
                                                      self.params["phase_offset"], (self.n, 2))
        if type(self.params["orientation"]) in (list, np.ndarray):
            self.orientations = np.array(self.params["orientation"], dtype=float)
            assert len(self.orientations) == self.n, "number of orientations supplied incompatible with number of neurons"
        else:
            self.orientations = distribution_sampler(self.params["orientation_distribution"],
                                                     self.params["orientation"], (self.n,))
        w = []
        for i in range(self.n):                                     # Neurons.py:1154-1161
            w1 = rotate(np.array([1, 0]), self.orientations[i])
            w.append(np.array([w1, rotate(w1, np.pi / 3), rotate(w1, 2 * np.pi / 3)]))
        self.w = np.array(w)
        if self.description == "rectified_cosines":
            assert self.width_ratio > 0 and self.width_ratio <= 1, "width_ratio must be between 0 and 1"
        if self.description not in _lib.GC_DESCRIPTIONS:
            raise ValueError(f"unknown GridCells description {self.description!r}")

    def _signature(self):
        return (np.ascontiguousarray(self.gridscales, dtype=np.float64).tobytes(),
                np.ascontiguousarray(self.phase_offsets, dtype=np.float64).tobytes(),
                np.ascontiguousarray(self.w, dtype=np.float64).tobytes(),
                self.description, float(self.width_ratio), float(self.min_fr), float(self.max_fr))

    def _pack(self):
        env = self.Agent.Environment
        gs = np.ascontiguousarray(self.gridscales, dtype=np.float64).reshape(-1)
        ph = np.ascontiguousarray(self.phase_offsets, dtype=np.float64).reshape(-1, 2)
        w = np.ascontiguousarray(self.w, dtype=np.float64).reshape(-1, 3, 2)
        self.n = gs.shape[0]
        c = _lib.GridCells()
        host = np.zeros(self._lib.riab_grid_pack_floats(self.n), dtype=np.float32)
        ext = np.ascontiguousarray(env.extent, dtype=np.float64)
        _lib.check(self._lib.riab_grid_pack(_f64p(gs), _f64p(ph), _f64p(w), self.n, _f64p(ext), C.byref(c),
                                            host.ctypes.data_as(_lib.c_float_p)))
        self._packed = self._upload(host)
        c.n_cells, c.description = self.n, _lib.GC_DESCRIPTIONS[self.description]
        c.width_ratio, c.min_fr, c.max_fr = float(self.width_ratio), float(self.min_fr), float(self.max_fr)
        c.packed_dev = self._packed.data_ptr()
        return c

    def _rates_from_positions(self, pos_dev, n_pos, out):
        ag = self.Agent
        _lib.check(self._lib.riab_grid_rates(pos_dev.data_ptr(), n_pos, C.byref(ag._env_struct()),
                                             C.byref(self._cells()), out.data_ptr(), out.stride(0), ag._stream()))


# =============================================================================
class BoundaryVectorCells(Neurons):
    default_params = {                                              # Neurons.py:1303-1316 (VectorCells) + :1549-1555
        "n": 10,
        "name": "BoundaryVectorCells",
        "reference_frame": "allocentric",
        "cell_arrangement": "random",
        "tuning_distance_distribution": "uniform",
        "tuning_distance": (0.05, 0.3),
        "sigma_distance_distribution": "diverging",
        "sigma_distance": (0.08, 12),
        "tuning_angle_distribution": "uniform",
        "tuning_angle": (0.0, 360),
        "angular_spread_distribution": "uniform",
        "angular_spread": (10, 30),
        "dtheta": 2,
        "max_fr": 1.0,
        "min_fr": 0.0,
    }
    _cells_kind = _lib.CELLS_BVC
    _egocentric_warning = "BVCs in egocentric plane require a head direction vector but none was passed. Using [1,0]"

    def _init_vector_tuning(self):
        """VectorCells.set_tuning_parameters (Neurons.py:1388-1437): tuning_distances / tuning_angles /
        sigma_distances / sigma_angles from ``cell_arrangement``."""
        from .utils import (create_random_assembly, create_uniform_radial_assembly,
                            create_diverging_radial_assembly)
        if self.reference_frame not in ("allocentric", "egocentric"):
            raise ValueError(f"unknown reference_frame {self.reference_frame!r}")
        arr = self.cell_arrangement                                   # VectorCells.set_tuning_parameters, Neurons.py:1388-1437
        if callable(arr):
            tuning = arr(**self.params)
        elif arr is None or (isinstance(arr, str) and arr[:6] == "random"):
            tuning = create_random_assembly(**self.params)
        elif arr == "uniform_manifold":
            tuning = create_uniform_radial_assembly(**self.params)
        elif arr == "diverging_manifold":
            tuning = create_diverging_radial_assembly(**self.params)
        else:
            raise ValueError("cell_arrangement must be either 'uniform_manifold' or 'diverging_manifold' or a function")
        (self.tuning_distances, self.tuning_angles, self.sigma_distances,
         self.sigma_angles) = (np.array(x, dtype=float) for x in tuning)
        assert len(self.tuning_distances) == len(self.tuning_angles) == len(self.sigma_distances) == len(self.sigma_angles), \
            "All manifold tuning parameters must be of the same length"
        self.n = len(self.tuning_distances)

    def __init__(self, Agent, params={}):
        from .utils import rotate
        super().__init__(Agent, params)
        assert self.Agent.Environment.boundary_conditions == "solid", \
            "boundary cells only possible with solid boundary conditions"      # Neurons.py:1580-1582
        self._init_vector_tuning()
        test_direction = np.array([1, 0])                           # Neurons.py:1584-1596 (duplicated-0 quirk kept)
        dirs, angs = [test_direction], [0]
        self.n_test_angles = int(360 / self.dtheta)
        for i in range(self.n_test_angles - 1):
            dirs.append(rotate(test_direction, 2 * np.pi * i * self.dtheta / 360))
            angs.append(2 * np.pi * i * self.dtheta / 360)
        self.test_directions = np.array(dirs, dtype=float)
        self.test_angles = np.array(angs, dtype=float)
        kappa = 1 / (self.sigma_angles.reshape(-1, 1) ** 2)         # Neurons.py:1599-1604
        self.cell_fr_norm = (np.exp(kappa * np.cos(self.test_angles.reshape(1, -1))) * (1 / np.exp(kappa))).sum(axis=1)
        self._scratch = None

    def _signature(self):
        return tuple(np.ascontiguousarray(a, dtype=np.float64).tobytes() for a in (
            self.tuning_distances, self.tuning_angles, self.sigma_distances, self.sigma_angles, self.test_angles,
            self.test_directions)) + (float(self.min_fr), float(self.max_fr), self.reference_frame)

    def _pack(self):
        arrs = [np.ascontiguousarray(a, dtype=np.float64).reshape(-1) for a in (
            self.tuning_distances, self.tuning_angles, self.sigma_distances, self.sigma_angles)]
        self.n = arrs[0].shape[0]
        angs = np.ascontiguousarray(self.test_angles, dtype=np.float64)
        T = angs.shape[0]
        c = _lib.BvcCells()
        host = np.zeros(self._lib.riab_bvc_pack_floats(self.n, T), dtype=np.float32)
        _lib.check(self._lib.riab_bvc_pack(*[_f64p(a) for a in arrs], self.n, _f64p(angs), T, C.byref(c),
                                           host.ctypes.data_as(_lib.c_float_p)))
        self._packed = self._upload(host)
        self._dirs_dev = self._upload(np.ascontiguousarray(self.test_directions, dtype=np.float64))
        c.n_cells, c.n_test_angles = self.n, T
        c.egocentric = 1 if self.reference_frame == "egocentric" else 0
        c.min_fr, c.max_fr = float(self.min_fr), float(self.max_fr)
        c.packed_dev, c.test_dirs_dev = self._packed.data_ptr(), self._dirs_dev.data_ptr()
        return c

    def _scratch_for(self, n):
        need = self._lib.riab_bvc_scratch_floats(n, len(self.test_angles))
        if self._scratch is None or self._scratch.numel() < need:
            self._scratch = self._torch.empty(need, dtype=self._torch.float32, device=self.device)
        return self._scratch

    def _scratch_ptr(self, n):
        return self._scratch_for(n).data_ptr()

    def _rates_from_positions(self, pos_dev, n_pos, out, first_wall=None, head_dir=None):
        ag = self.Agent
        scratch = self._scratch_for(n_pos)
        _lib.check(self._lib.riab_bvc_rates(pos_dev.data_ptr(), n_pos, C.byref(ag._env_struct()),
                                            C.byref(self._cells()), scratch.data_ptr(),
                                            first_wall.data_ptr() if first_wall is not None else None,
                                            head_dir.data_ptr() if head_dir is not None else None,
                                            out.data_ptr(), out.stride(0), ag._stream()))

    def get_state(self, evaluate_at="agent", **kwargs):
        """BoundaryVectorCells.get_state (Neurons.py:1617-1744).  Egocentric cells take the Agent's
        head_direction with evaluate_at="agent", else the ``head_direction`` kwarg (one vector for all
        positions, or one per position), else [1,0] with the reference's warning (Neurons.py:1693-1706)."""
        if self.reference_frame != "egocentric":
            return super().get_state(evaluate_at, **kwargs)
        torch = self._torch
        self._cells()
        if evaluate_at == "agent":
            self.Agent._flush_pending()
            pos_dev, hd_dev = self.Agent._s["pos"], self.Agent._s["head_direction"]
        else:
            pos = self.Agent.Environment.flattened_discrete_coords if evaluate_at == "all" else kwargs["pos"]
            pos_dev = torch.as_tensor(np.ascontiguousarray(np.asarray(pos, dtype=np.float64).reshape(-1, 2)), device=self.device)
            if "head_direction" in kwargs:
                hd = np.array(kwargs["head_direction"], dtype=np.float64)       # own, writable copy
            elif "vel" in kwargs:
                warnings.warn("'vel' kwarg deprecated in favour of 'head_direction'")
                hd = np.asarray(kwargs["vel"], dtype=np.float64)
            else:
                warnings.warn(self._egocentric_warning)
                hd = np.array([1.0, 0.0])
            hd = np.array(np.broadcast_to(hd.reshape(-1, 2), (pos_dev.shape[0], 2)), order="C")   # own, writable, C-contiguous
            hd_dev = torch.as_tensor(hd, device=self.device)
        n_pos = int(pos_dev.shape[0])
        out = torch.empty((n_pos, self._ld()), dtype=torch.float32, device=self.device)
        if n_pos:
            self._rates_from_positions(pos_dev, n_pos, out, head_dir=hd_dev)
        if kwargs.get("return_tensor", False):
            return out[:, : self.n]
        return out[:, : self.n].T.contiguous().cpu().numpy().astype(np.float64)


class FieldOfViewBVCs(BoundaryVectorCells):
    """Egocentric BVCs tiling the agent's field of view (ratinabox/Neurons.py:1847-1887)."""
    default_params = {
        "distance_range": [0.02, 0.4],
        "angle_range": [0, 75],
        "spatial_resolution": 0.02,
        "cell_arrangement": "diverging_manifold",
        "beta": 5,
        "color": [0.3, 0.3, 0.3, 1],
    }

    def __init__(self, Agent, params={}):
        p = copy.deepcopy(__class__.default_params)
        p.update(params)
        p["reference_frame"] = "egocentric"
        assert p["cell_arrangement"] is not None, "cell_arrangement must be set for FoV Neurons"
        super().__init__(Agent, p)


class ObjectVectorCells(BoundaryVectorCells):
    """ratinabox.ObjectVectorCells (Neurons.py:1892-2113): vector cells tuned to the objects of the Environment.
    Same tuning machinery as the other VectorCells (cell_arrangement, tuning_distance, ...); each cell responds to the
    objects of ONE type (``object_tuning_type``: "random", an int, or one int per cell).  The rates are evaluated by
    ``riab_ovc_*`` (csrc/riab_ovc.cuh): exact float64 agent-object geometry per agent, float32 tuning per cell."""
    default_params = {
        "n": 10,
        "name": "ObjectVectorCell",
        "walls_occlude": True,          # objects behind walls cannot be seen
        "object_tuning_type": "random",
    }
    _cells_kind = _lib.CELLS_OVC

    def __init__(self, Agent, params={}):
        p = copy.deepcopy(__class__.default_params)
        p.update(params)
        env = Agent.Environment
        if len(env.objects["objects"]) == 0:                       # Neurons.py:1921-1923
            raise RuntimeError(f"Cannot initialize {p['name']}, as there are no objects in the environment.")
        if len(env.objects["objects"]) > _lib.MAX_OBJECTS:
            raise NotImplementedError(f"at most {_lib.MAX_OBJECTS} objects per environment on the CUDA path")
        Neurons.__init__(self, Agent, p)
        self._init_vector_tuning()
        self.object_locations = env.objects["objects"]
        self.tuning_types = None
        self.set_tuning_types(self.object_tuning_type)
        self.wall_geometry = "line_of_sight" if self.walls_occlude == True else "euclidean"      # Neurons.py:1937-1940

    def set_tuning_types(self, tuning_types=None):                  # Neurons.py:1962-1986
        if isinstance(tuning_types, str) and tuning_types == "random":
            self.object_types = self.Agent.Environment.objects["object_types"]
            self.tuning_types = np.random.choice(np.unique(self.object_types), replace=True, size=(self.n,))
        else:
            if isinstance(tuning_types, (int, np.integer)):
                tuning_types = np.repeat(tuning_types, self.n)
            elif isinstance(tuning_types, list):
                tuning_types = np.array(tuning_types)
            assert isinstance(tuning_types, np.ndarray), "tuning_types must be an integer, list or numpy array"
            assert tuning_types.shape[0] == self.n, \
                f"Tuning types must be a vector of length of the number of neurons: ({self.n},)"
            self.tuning_types = tuning_types

    def _signature(self):
        env = self.Agent.Environment
        return tuple(np.ascontiguousarray(a, dtype=np.float64).tobytes() for a in (
            self.tuning_distances, self.tuning_angles, self.sigma_distances, self.sigma_angles,
            np.asarray(self.tuning_types, dtype=np.float64), env.objects["objects"],
            np.asarray(env.objects["object_types"], dtype=np.float64))) + (
            float(self.min_fr), float(self.max_fr), self.reference_frame, self.wall_geometry)

    def _pack(self):
        env = self.Agent.Environment
        arrs = [np.ascontiguousarray(a, dtype=np.float64).reshape(-1) for a in (
            self.tuning_distances, self.tuning_angles, self.sigma_distances, self.sigma_angles)]
        self.n = arrs[0].shape[0]
        types = np.ascontiguousarray(self.tuning_types, dtype=np.int32).reshape(-1)
        assert types.shape[0] == self.n
        objs = np.ascontiguousarray(env.objects["objects"], dtype=np.float64).reshape(-1, 2)
        otypes = np.asarray(env.objects["object_types"], dtype=np.int32).reshape(-1)
        if len(objs) > _lib.MAX_OBJECTS:
            raise NotImplementedError(f"at most {_lib.MAX_OBJECTS} objects per environment on the CUDA path")
        c = _lib.OvcCells()
        host = np.zeros(self._lib.riab_ovc_pack_floats(self.n), dtype=np.float32)
        _lib.check(self._lib.riab_ovc_pack(*[_f64p(a) for a in arrs], types.ctypes.data_as(C.POINTER(C.c_int32)), self.n,
                                           C.byref(c), host.ctypes.data_as(_lib.c_float_p)))
        self._packed = self._upload(host)
        c.n_cells, c.n_objects = self.n, len(objs)
        for o in range(len(objs)):
            c.objects[2 * o], c.objects[2 * o + 1] = float(objs[o, 0]), float(objs[o, 1])
            c.object_types[o] = int(otypes[o])
        c.walls_occlude = 1 if self.wall_geometry == "line_of_sight" else 0
        c.egocentric = 1 if self.reference_frame == "egocentric" else 0
        c.min_fr, c.max_fr = float(self.min_fr), float(self.max_fr)
        c.packed_dev = self._packed.data_ptr()
        return c

    def _scratch_ptr(self, n):
        return None

    def _rates_from_positions(self, pos_dev, n_pos, out, first_wall=None, head_dir=None):
        ag = self.Agent
        _lib.check(self._lib.riab_ovc_rates(pos_dev.data_ptr(), n_pos, C.byref(ag._env_struct()), C.byref(self._cells()),
                                            head_dir.data_ptr() if head_dir is not None else None,
                                            out.data_ptr(), out.stride(0), ag._stream()))

    _egocentric_warning = "OVCs in egocentric plane require a head direction vector but none was passed. Using [1,0]"


class FieldOfViewOVCs(ObjectVectorCells):
    """Egocentric ObjectVectorCells tiling the agent's field of view (ratinabox/Neurons.py:2116-2160)."""
    default_params = {
        "distance_range": [0.02, 0.4],
        "angle_range": [0, 75],
        "spatial_resolution": 0.02,
        "beta": 5,
        "cell_arrangement": "diverging_manifold",
        "object_tuning_type": None,
    }

    def __init__(self, Agent, params={}):
        p = copy.deepcopy(__class__.default_params)
        p.update(params)
        if p["object_tuning_type"] is None:
            warnings.warn("For FieldOfViewOVCs you must specify the object type they are selective for with the "
                          "'object_tuning_type' parameter. This can be 'random' (each cell in the field of view chooses a "
                          "random object type) or any integer (all cells have the same preference for this type). For now "
                          "defaulting to params['object_tuning_type'] = 0.")
            p["object_tuning_type"] = 0
        p["reference_frame"] = "egocentric"
        assert p["cell_arrangement"] is not None, "cell_arrangement must be set for FOV Neurons"
        super().__init__(Agent, p)
