"""BatchedFlexProvisionEnv -- N independent flex_provision environments on one B200.

Same verbs as the reference's MultiAgentEnv API (madrl/environments/multiagentenv.py:1-67,
implemented by flexibility_provision_env.py) with a leading env dimension on device
tensors:

    reset()            -> (obs[N, na, 6*history] f32, state[N, 3*nb+2*na+1] f32)
    step(actions)      -> (reward[N] f64, terminated[N] bool, info: dict[str, Tensor[N]])
    get_obs()          -> obs            (pushes the observation history, quirk Q7)
    get_state()        -> state
    get_avail_actions()-> ones[N, na, 4]

All compute happens in libflexgpu.so (hand-written sm_100a CUDA, include/flexgpu.h); torch
only owns device memory and the stream.  Output tensors are allocated once and overwritten
by the next call of the same verb.
"""
import ctypes as C
import warnings

import numpy as np
import torch

from . import _lib, sharding
from .config import convert, make_fp_config, normalize_args
from .network import Network, create_network
from .profiles import Profiles, csv_profiles_available, load_csv_profiles, synthetic_profiles


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class BatchedFlexProvisionEnv:
    def __init__(self, kwargs=None, n_envs=1, device="cuda:0", network=None, profiles=None,
                 seed=None, env_offset=0):
        self.args_dict = normalize_args(kwargs)
        self.args = convert(self.args_dict)
        self.n_envs = int(n_envs)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.FlexGpuError("BatchedFlexProvisionEnv needs a CUDA device; there is no CPU fallback")
        if not torch.cuda.is_available():
            raise _lib.FlexGpuError("no CUDA device available; there is no CPU fallback")
        self.base_powergrid = network if network is not None else create_network(
            self.args_dict, self.args_dict.get("data_path"))
        self.network = Network(self.base_powergrid)
        self.n_bus = self.network.n_bus
        self.n_lines = self.n_bus - 1
        self.n_agents = len(self.base_powergrid['buildings'])          # :66
        self.n_actions = 4                                             # :67
        self.agent_ids = self.base_powergrid['buildings']              # :68
        self.episode_limit = self.args_dict["episode_limit"]           # :61
        self.history = self.args_dict["history"]                       # :65
        self.obs_size = 6 * self.history if self.history > 1 else 6
        self.state_size = 3 * self.n_bus + 2 * self.n_agents + 1
        self.kernel_variant = self.args_dict["kernel_variant"]
        self.seed = int(self.args_dict["seed"] if seed is None else seed)
        self.env_offset = int(env_offset)

        self._lib = _lib.lib()
        self._cfg = make_fp_config(self.args_dict, self.network)
        self._h = C.c_void_p()
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", dev_index)    # the handle's device: torch's current device may change later
        _lib.check(self._lib.fp_create(C.byref(self._cfg), self.n_envs, dev_index, C.byref(self._h)),
                   None, "fp_create")
        self.profiles = None
        if profiles is None:
            # the reference's __init__ loads the four CSVs under data_path (:55-58); they ship as Git-LFS
            # pointers, so a checkout without the payloads has nothing to load -- say so instead of
            # silently training on made-up data
            data_path = self.args_dict.get("data_path")
            if csv_profiles_available(data_path):
                profiles = load_csv_profiles(data_path, self.args_dict)
            else:
                warnings.warn(f"no profile CSVs under data_path={data_path!r} (pv_active/load_active/load_reactive/"
                              "prices.csv missing or Git-LFS pointers): using SYNTHETIC profiles of the bundled "
                              "data's shape; pass profiles= or point data_path at the real files", stacklevel=2)
                profiles = synthetic_profiles(self.network, self.n_agents, seed=0, pv_scale=self.args_dict["pv_scale"])
        self.load_profiles(profiles)
        N, na, nb = self.n_envs, self.n_agents, self.n_bus
        dev = self.device
        self._reward = torch.empty(N, dtype=torch.float64, device=dev)
        self._done = torch.zeros(N, dtype=torch.bool, device=dev)      # one byte per env, written as uint8
        self._info = torch.empty(N, _lib.FP_INFO_STRIDE, dtype=torch.float64, device=dev)
        self._obs = {}
        self._state = {}
        self._stats = torch.zeros(_lib.FP_NSTATS, dtype=torch.float64, device=dev)
        self._avail = torch.ones(N, na, self.n_actions, dtype=torch.int64, device=dev)
        self._views = None
        self._inject = None
        self._host = None
        self._obs_views = {}
        self._reset_failed = None

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.fp_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        _lib.check(rc, self._h, what)

    # ------------------------------------------------------------------ data
    def load_profiles(self, profiles):
        """Replaces _load_*_data (:431-465): host arrays -> device dataset."""
        if isinstance(profiles, dict):
            profiles = Profiles(**profiles)
        if profiles.P.shape[1] != self.n_lines or profiles.PV.shape[1] != self.n_agents:
            raise ValueError("profile widths do not match the network")
        self.profiles = profiles
        self.time_delta = profiles.time_delta
        self._check(self._lib.fp_load_profiles(
            self._h, profiles.P.ctypes.data_as(C.c_void_p), profiles.Q.ctypes.data_as(C.c_void_p),
            profiles.PV.ctypes.data_as(C.c_void_p), profiles.price.ctypes.data_as(C.c_void_p),
            profiles.T), "fp_load_profiles")

    def max_start(self):
        """Largest valid episode start row (+1): the slice is episode_limit + history + 1 rows (:478)."""
        return self.profiles.T - (self.episode_limit + self.history + 1) + 1

    # ------------------------------------------------------------------ views on live state
    def _state_views(self):
        if self._views is None:
            ptrs = [C.c_void_p() for _ in range(6)]
            self._check(self._lib.fp_state_ptrs(self._h, *[C.byref(p) for p in ptrs]), "fp_state_ptrs")
            N, na, nb, nl = self.n_envs, self.n_agents, self.n_bus, self.n_lines

            def view(p, shape, dtype):
                if not p.value:
                    return None
                n = int(np.prod(shape))
                itemsize = torch.empty(0, dtype=dtype).element_size()
                holder = _ExternalCudaBuffer(p.value, n * itemsize, self.device.index or 0)
                return torch.as_tensor(holder, device=self.device).view(dtype).view(*shape)

            self._views = dict(
                rec=view(ptrs[0], (N, _lib.FP_REC_STRIDE), torch.int64),
                voltage=view(ptrs[1], (N, nb), torch.float64),
                setpoint=view(ptrs[2], (N, 4, na), torch.float64),
                pflow=view(ptrs[3], (N, nl), torch.float64),
                qflow=view(ptrs[4], (N, nl), torch.float64),
                isq=view(ptrs[5], (N, nl), torch.float64),
            )
        return self._views

    def keep_line_flows(self, keep=True):
        """Also store receiving-end P/Q and squared currents of every solve (utils/pf.py:109-110)."""
        self._check(self._lib.fp_set_keep_flows(self._h, 1 if keep else 0), "fp_set_keep_flows")
        self._views = None

    @property
    def rec(self):
        return self._state_views()["rec"]

    @property
    def voltages(self):
        """current_voltage, bus order [N, nb] (:146, :310)."""
        return self._state_views()["voltage"]

    @property
    def setpoints(self):
        """[N, 4, na]: power_reduction, ess_charging, ess_discharging, q_pv."""
        return self._state_views()["setpoint"]

    @property
    def line_flows(self):
        v = self._state_views()
        return v["pflow"], v["qflow"], v["isq"]

    @property
    def ess_energy(self):
        na = self.n_agents
        return self.rec[:, _lib.REC_E_CUR:_lib.REC_E_CUR + na].view(torch.float64)

    @property
    def initial_ess_energy(self):
        na = self.n_agents
        return self.rec[:, _lib.REC_E_INIT:_lib.REC_E_INIT + na].view(torch.float64)

    @property
    def cumulative_reward(self):
        return self.rec[:, _lib.REC_CUM].view(torch.float64)

    @property
    def steps(self):
        return (self.rec[:, _lib.REC_TIME] >> 32).to(torch.int32)

    @property
    def start_index(self):
        return (self.rec[:, _lib.REC_TIME] & 0xFFFFFFFF).to(torch.int32)

    @property
    def violation_mask(self):
        """uint64-as-int64 bit mask, bit b = bus position b outside [v_min, v_max]."""
        return self.rec[:, _lib.REC_VMASK]

    @property
    def violation_count(self):
        return (self.rec[:, _lib.REC_COUNTS] & 0xFFFFFFFF).to(torch.int32)

    @property
    def flags(self):
        return (self.rec[:, _lib.REC_COUNTS] >> 32).to(torch.int32)

    @property
    def line_limit_mask(self):
        return (self.rec[:, _lib.REC_LINES] & 0xFFFFFFFF).to(torch.int64)

    @property
    def pf_iterations(self):
        return (self.rec[:, _lib.REC_LINES] >> 32).to(torch.int32)

    # ------------------------------------------------------------------ episode control
    def _dev(self, x, dtype):
        if x is None:
            return None
        if isinstance(x, torch.Tensor):
            return x.to(device=self.device, dtype=dtype).contiguous()
        return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).to(self.device)

    RESET_RETRIES = 3        # redraws of an env whose initial power flow fails (the reference loops until solvable, :82-153)

    def reset(self, start_index=None, e0=None, a0=None, mask=None, return_obs=True, check=False, retries=None):
        """Replaces reset()/manual_reset() (:74-155, :157-239).

        With no draws given, each env draws (start row, E0, a0) from its own Philox stream
        keyed by (seed, env_offset + e, episode counter).  Envs whose initial power flow fails
        are re-drawn up to RESET_RETRIES times like the reference's `while not solvable` loop (:82-153) -- on the
        device, without a host round trip.  An env that still fails keeps FP_FLAG_RESET_FAILED in `flags`
        (`reset_failed_count()` reads the count); check=True synchronises and raises FlexGpuError instead;
        `retries` overrides RESET_RETRIES (0: a single launch, for per-step auto-resets).
        A reset restarts the observation history of the envs it resets: a window returned earlier by
        get_obs() / step(return_obs=...) no longer holds their previous episode -- copy `next_obs` before resetting."""
        m = self._dev(mask, torch.uint8)
        if start_index is None:
            if self._reset_failed is None:
                self._reset_failed = torch.zeros(1, dtype=torch.int32, device=self.device)
            n_retry = self.RESET_RETRIES if retries is None else int(retries)
            if n_retry == 0 and not check:         # per-step auto-reset: one launch, no failure count
                self._check(self._lib.fp_reset_random(self._h, self.seed, self.env_offset, _ptr(m), _lib.stream(self.device)), "fp_reset_random")
            else:
                self._check(self._lib.fp_reset_random_retry(self._h, self.seed, self.env_offset, _ptr(m), n_retry,
                                                            _ptr(self._reset_failed), _lib.stream(self.device)), "fp_reset_random_retry")
            if check and int(self._reset_failed.item()):
                raise _lib.FlexGpuError(f"{int(self._reset_failed.item())} envs found no solvable initial state in "
                                        f"{self.RESET_RETRIES + 1} draws")
        else:
            N, na = self.n_envs, self.n_agents
            s = self._dev(start_index, torch.int32).view(N)
            e = self._dev(e0, torch.float64).view(N, na)
            a = self._dev(a0, torch.float64).view(N, na * 4)
            lo, hi = int(s.min()), int(s.max())
            if lo < 0 or hi >= self.max_start():
                raise ValueError("start_index out of range for the loaded profiles")
            self._check(self._lib.fp_reset(self._h, _ptr(s), _ptr(e), _ptr(a), _ptr(m), _lib.stream(self.device)), "fp_reset")
        if return_obs == "ring":                                        # reset()'s get_obs (:155) for the reset envs, ring form
            self._check(self._lib.fp_obs_ring_reset_push(self._h, _ptr(m), _lib.stream(self.device)), "fp_obs_ring_reset_push")
            return self.obs_ring()
        if return_obs:
            return self.get_obs(), self.get_state()                     # :155
        return None

    def reset_failed_count(self):
        """Envs whose last random reset found no solvable initial state (synchronises)."""
        return 0 if self._reset_failed is None else int(self._reset_failed.item())

    def step(self, actions, mask=None, want_info=True, translate=False, return_obs=False):
        """Replaces step() (:241-356).  actions: [N, na, 4] (or [N, na*4]) fp32 or fp64 tensor.
        return_obs=True appends the next observation (one pushing get_obs, as model.py:223 does right
        after the step) to the returned tuple: (reward, done, info, obs).  return_obs="ring" does the same in ONE
        launch and returns the history in its native device layout (ObsRing) -- what the device policy consumes.
        translate=True: `actions` are the policy's raw fp32 outputs and translate_action
        (utils/util.py:121-129: clamp to [action_low, action_high], then 0.5 (x + 1)(high - low) + low,
        all in fp32 -- quirk Q5) is applied inside the step kernel, as model.py:218-220 does on the host."""
        if not isinstance(actions, torch.Tensor):
            actions = torch.as_tensor(np.ascontiguousarray(actions))
        if translate:
            actions = actions.to(torch.float32)
        elif actions.dtype not in (torch.float32, torch.float64):
            actions = actions.to(torch.float64)
        actions = actions.to(self.device).contiguous()
        if actions.numel() != self.n_envs * self.n_agents * self.n_actions:
            raise ValueError("actions must have n_envs * n_agents * 4 elements")         # :260
        m = self._dev(mask, torch.uint8)
        dt = _lib.FP_F32_POLICY if translate else (_lib.FP_F64 if actions.dtype == torch.float64 else _lib.FP_F32)
        if return_obs == "ring":                     # step + pushing get_obs in ONE launch, native env-minor ring
            p, sl, npad = C.c_void_p(), C.c_int32(), C.c_int64()
            self._check(self._lib.fp_step_ring(self._h, _ptr(actions), dt, _ptr(self._reward), _ptr(self._done),
                                               _ptr(self._info) if want_info else None, _ptr(m), C.byref(p), C.byref(sl),
                                               C.byref(npad), _lib.stream(self.device)), "fp_step_ring")
            obs = self._ring(p.value, sl.value, npad.value)
        elif return_obs:                             # step + pushing get_obs, dense strided view (fp_step_obs)
            p, ep, ap = C.c_void_p(), C.c_int64(), C.c_int64()
            self._check(self._lib.fp_step_obs(self._h, _ptr(actions), dt, _ptr(self._reward), _ptr(self._done),
                                              _ptr(self._info) if want_info else None, _ptr(m), C.byref(p), C.byref(ep),
                                              C.byref(ap), _lib.stream(self.device)), "fp_step_obs")
            obs = self._obs_view(p.value, ep.value, ap.value)
        else:
            self._check(self._lib.fp_step(self._h, _ptr(actions), dt, _ptr(self._reward), _ptr(self._done),
                                          _ptr(self._info) if want_info else None, _ptr(m), _lib.stream(self.device)), "fp_step")
        info = {k: self._info[:, i] for i, k in enumerate(_lib.INFO_KEYS)} if want_info else {}
        if return_obs:
            return self._reward, self._done, info, obs
        return self._reward, self._done, info

    def preview_step(self, actions, translate=False, want_info=True, want_voltage=False, want_mask=False):
        """What step(actions) would return and leave behind, without committing anything (fp_step_preview): no record,
        voltage, setpoint, line-flow, observation-history or statistics write, so it may be called any number of times
        between two steps.  actions: [N, na, 4] for one candidate per env, or [K, N, na, 4] for K candidates per env
        (one launch); dtypes and translate as step().  Returns (reward, done, info) -- plus voltages [.., N, n_bus] f64
        (what env.voltages would hold: after a failed solve the rolled-back ones) with want_voltage, plus the violation
        mask [.., N] (what env.violation_mask would read) with want_mask -- with a leading K dimension for [K, N, na, 4]
        actions.  info has step()'s keys.  Every returned tensor is freshly allocated."""
        if not isinstance(actions, torch.Tensor):
            actions = torch.as_tensor(np.ascontiguousarray(actions))
        if translate:
            actions = actions.to(torch.float32)
        elif actions.dtype not in (torch.float32, torch.float64):
            actions = actions.to(torch.float64)
        actions = actions.to(self.device).contiguous()
        N, na, nb = self.n_envs, self.n_agents, self.n_bus
        tail = (N, na, self.n_actions)
        if actions.dim() == 3 and tuple(actions.shape) == tail:
            k, lead = 1, ()
        elif actions.dim() == 4 and tuple(actions.shape[1:]) == tail and actions.shape[0] >= 1:
            k = int(actions.shape[0]); lead = (k,)
        else:
            raise ValueError(f"actions must be [n_envs, n_agents, 4] or [K, n_envs, n_agents, 4], got {tuple(actions.shape)}")
        dev = self.device
        reward = torch.empty(*lead, N, dtype=torch.float64, device=dev)
        done = torch.empty(*lead, N, dtype=torch.bool, device=dev)          # one byte per env, written as uint8
        info = torch.empty(*lead, N, _lib.FP_INFO_STRIDE, dtype=torch.float64, device=dev) if want_info else None
        volt = torch.empty(*lead, N, nb, dtype=torch.float64, device=dev) if want_voltage else None
        vmask = torch.empty(*lead, N, dtype=torch.int64, device=dev) if want_mask else None
        dt = _lib.FP_F32_POLICY if translate else (_lib.FP_F64 if actions.dtype == torch.float64 else _lib.FP_F32)
        self._check(self._lib.fp_step_preview(self._h, k, _ptr(actions), dt, _ptr(reward), _ptr(done), _ptr(info), _ptr(volt),
                                              _ptr(vmask), _lib.stream(dev)), "fp_step_preview")
        out = (reward, done, {k_: info[..., i] for i, k_ in enumerate(_lib.INFO_KEYS)} if want_info else {})
        if want_voltage:
            out += (volt,)
        if want_mask:
            out += (vmask,)
        return out

    def step_host(self, actions, want_info=False, translate=False):
        """End-to-end variant: host (numpy, ideally pinned) in, host out, through fp_step_host.
        Pinned fp32 actions (thread variant) are read by the step kernel straight from host memory, and the
        results are written straight into the pinned output buffers (zero-copy).  Pageable or fp64 actions
        are copied through device staging buffers.  The outputs are the same either way.
        translate: see step()."""
        a = np.ascontiguousarray(actions)
        if translate:
            a = np.ascontiguousarray(a, dtype=np.float32)
        elif a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        if a.size != self.n_envs * self.n_agents * self.n_actions:
            raise ValueError("actions must have n_envs * n_agents * 4 elements")
        if self._host is None:
            N = self.n_envs
            self._host = dict(
                reward=torch.empty(N, dtype=torch.float64).pin_memory(),
                done=torch.empty(N, dtype=torch.uint8).pin_memory(),
                info=torch.empty(N, _lib.FP_INFO_STRIDE, dtype=torch.float64).pin_memory())
        hb = self._host
        dt = _lib.FP_F32_POLICY if translate else (_lib.FP_F64 if a.dtype == np.float64 else _lib.FP_F32)
        self._check(self._lib.fp_step_host(
            self._h, a.ctypes.data_as(C.c_void_p), dt, C.c_void_p(hb["reward"].data_ptr()),
            C.c_void_p(hb["done"].data_ptr()), C.c_void_p(hb["info"].data_ptr()) if want_info else None,
            _lib.stream(self.device)), "fp_step_host")
        info = {k: hb["info"].numpy()[:, i] for i, k in enumerate(_lib.INFO_KEYS)} if want_info else {}
        return hb["reward"].numpy(), hb["done"].numpy().astype(bool), info

    # ------------------------------------------------------------------ observations
    def get_obs(self, push=True, dtype=torch.float32, contiguous=False):
        """Replaces get_obs() (:370-403).  push=True reproduces its history side effect (Q7).

        The default call (pushing, fp32 -- what the rollout loop does once per step, model.py:223) returns a
        strided VIEW [N, na, 6*history] of the handle's window ring (fp_get_obs_view): the push writes 48
        bytes per agent and nothing is re-materialised.  The view is read-only, valid until the next pushing
        call OR RESET (a reset zeroes the window ring of the envs it resets: copy `next_obs` before an
        auto-reset if it is to be stored), contiguous along the last dimension and mergeable over the first two (`.view(N * na, -1)`
        works; use `.contiguous()` or contiguous=True for a packed copy).  push=False, fp64 and
        contiguous=True go through their own buffers."""
        if push and dtype == torch.float32 and not contiguous:
            p, ep, ap = C.c_void_p(), C.c_int64(), C.c_int64()
            self._check(self._lib.fp_get_obs_view(self._h, 1, C.byref(p), C.byref(ep), C.byref(ap), _lib.stream(self.device)),
                        "fp_get_obs_view")
            return self._obs_view(p.value, ep.value, ap.value)
        buf = self._obs.get(dtype)
        if buf is None:
            buf = torch.empty(self.n_envs, self.n_agents, self.obs_size, dtype=dtype, device=self.device)
            self._obs[dtype] = buf
        dt = _lib.FP_F64 if dtype == torch.float64 else _lib.FP_F32
        self._check(self._lib.fp_get_obs(self._h, _ptr(buf), dt, 1 if push else 0, _lib.stream(self.device)), "fp_get_obs")
        return buf

    def obs_ring(self):
        """The observation history in its native device layout (fp_obs_ring): ObsRing, no push."""
        p, sl, npad = C.c_void_p(), C.c_int32(), C.c_int64()
        self._check(self._lib.fp_obs_ring(self._h, C.byref(p), C.byref(sl), C.byref(npad), _lib.stream(self.device)), "fp_obs_ring")
        return self._ring(p.value, sl.value, npad.value)

    def _ring(self, ptr, slot, n_pad):
        t = self._obs_views.get(("ring", ptr))
        if t is None:
            holder = _ExternalCudaBuffer(ptr, self.history * self.n_agents * 6 * n_pad * 4, self.device.index or 0)
            t = torch.as_tensor(holder, device=self.device).view(torch.float32).view(self.history, self.n_agents, 6, n_pad)
            self._obs_views[("ring", ptr)] = t
        return ObsRing(self, t, slot)

    def _obs_view(self, ptr, env_pitch, agent_pitch):
        view = self._obs_views.get(ptr)                              # one cached tensor per ring position
        if view is None:
            span = (self.n_envs - 1) * env_pitch + (self.n_agents - 1) * agent_pitch + self.obs_size
            holder = _ExternalCudaBuffer(ptr, span * 4, self.device.index or 0)
            flat = torch.as_tensor(holder, device=self.device).view(torch.float32)
            view = torch.as_strided(flat, (self.n_envs, self.n_agents, self.obs_size), (env_pitch, agent_pitch, 1))
            self._obs_views[ptr] = view
        return view

    def get_state(self, dtype=torch.float32):
        """Replaces get_state() (:358-368)."""
        buf = self._state.get(dtype)
        if buf is None:
            buf = torch.empty(self.n_envs, self.state_size, dtype=dtype, device=self.device)
            self._state[dtype] = buf
        dt = _lib.FP_F64 if dtype == torch.float64 else _lib.FP_F32
        self._check(self._lib.fp_get_state(self._h, _ptr(buf), dt, _lib.stream(self.device)), "fp_get_state")
        return buf

    def get_avail_actions(self):                 # :721-726
        return self._avail

    def get_obs_size(self):
        return self.obs_size

    def get_state_size(self):
        return self.state_size

    def get_total_actions(self):
        return self.n_actions

    def get_num_of_agents(self):
        return self.n_agents

    def get_env_info(self):                      # multiagentenv.py:61-67
        return {"state_shape": self.get_state_size(), "obs_shape": self.get_obs_size(),
                "n_actions": self.get_total_actions(), "n_agents": self.n_agents,
                "episode_limit": self.episode_limit}

    # ------------------------------------------------------------------ power flow only
    def power_flow(self, p, q, want_flows=True):
        """Batched power_flow_solver_simplified (utils/pf.py:115-192): p, q [n, nl] -> dict."""
        p = self._dev(p, torch.float64)
        q = self._dev(q, torch.float64)
        n = p.shape[0]
        if p.shape != (n, self.n_lines) or q.shape != p.shape:
            raise ValueError("p and q must be [n, n_bus - 1]")
        V = torch.empty(n, self.n_bus, dtype=torch.float64, device=self.device)
        Pl = Ql = Isq = None
        if want_flows:
            Pl, Ql, Isq = (torch.empty(n, self.n_lines, dtype=torch.float64, device=self.device) for _ in range(3))
        iters = torch.empty(n, dtype=torch.int32, device=self.device)
        failed = torch.empty(n, dtype=torch.uint8, device=self.device)
        self._check(self._lib.fp_power_flow(self._h, n, _ptr(p), _ptr(q), _ptr(V), _ptr(Pl), _ptr(Ql),
                                            _ptr(Isq), _ptr(iters), _ptr(failed), _lib.stream(self.device)), "fp_power_flow")
        return dict(V=V, P=Pl, Q=Ql, Isq=Isq, iters=iters, failed=failed.bool())

    def set_obs_history(self, keep=True):
        """keep=False: ring-only stepping for device rollouts -- step(..., return_obs='ring') pushes the env-minor fp32
        ring alone (91 -> 79 us per 131 072 envs); the fp64 history behind get_obs() is restored from the ring when a
        call needs it, with its entries at fp32 precision (fp32 reads are unchanged)."""
        self._check(self._lib.fp_set_obs_history(self._h, 1 if keep else 0), "fp_set_obs_history")

    # ------------------------------------------------------------------ checkpointing the device state (SURVEY 5)
    def _history(self, write):
        p, per = C.c_void_p(), C.c_int64()
        self._check(self._lib.fp_history_ptr(self._h, C.byref(p), C.byref(per), 1 if write else 0), "fp_history_ptr")
        holder = _ExternalCudaBuffer(p.value, self.n_envs * per.value * 8, self.device.index or 0)
        return torch.as_tensor(holder, device=self.device).view(torch.float64).view(self.n_envs, per.value)

    def state_dict(self):
        """The complete per-env device state as CPU tensors: records (energies, counters, masks), voltages, applied
        setpoints, observation history.  The reference checkpoints no env state (train_agent.py:144-147 saves the model
        only); this is for debugging and for resuming a rollout."""
        torch.cuda.synchronize(self.device)
        return {"rec": self.rec.cpu().clone(), "voltage": self.voltages.cpu().clone(), "setpoint": self.setpoints.cpu().clone(),
                "history": self._history(False).cpu().clone(), "n_envs": self.n_envs, "seed": self.seed, "env_offset": self.env_offset}

    def load_state_dict(self, sd):
        if int(sd["n_envs"]) != self.n_envs:
            raise ValueError("state_dict holds a different number of envs")
        self.rec.copy_(sd["rec"].to(self.device)); self.voltages.copy_(sd["voltage"].to(self.device))
        self.setpoints.copy_(sd["setpoint"].to(self.device)); self._history(True).copy_(sd["history"].to(self.device))
        self.seed, self.env_offset = int(sd["seed"]), int(sd["env_offset"])

    # ------------------------------------------------------------------ safety layer (SAFEMADDPG)
    def load_safety_model(self, coef, intercept, slack_weight=1000.0):
        """The fitted voltage regressor as safemaddpg.py:182-184 reads it: coef [n_bus, 2 n_bus], intercept [n_bus]."""
        coef = np.ascontiguousarray(coef, dtype=np.float64); icpt = np.ascontiguousarray(intercept, dtype=np.float64)
        if coef.shape != (self.n_bus, 2 * self.n_bus) or icpt.shape != (self.n_bus,):
            raise ValueError("coef must be [n_bus, 2 n_bus] and intercept [n_bus]")
        self._check(self._lib.fp_safety_load(self._h, coef.ctypes.data_as(C.c_void_p), icpt.ctypes.data_as(C.c_void_p),
                                             float(self.args_dict["v_min"]), float(self.args_dict["v_max"]), float(slack_weight)),
                    "fp_safety_load")

    def safety_project(self, actions, layout="reference", want_info=False):
        """safety_layer_optimization (safemaddpg.py:176-299) for every env: raw policy actions [N, na, 4] -> adjusted
        setpoints (fp32).  layout="reference": [N, 4 na] as the reference returns them ([x | c | d | g], :290-296);
        layout="agent": [N, na, 4].  want_info adds (slack [N, na] f64, intervened [N, na] bool)."""
        a = actions.to(self.device).contiguous()
        if a.dtype not in (torch.float32, torch.float64):
            a = a.to(torch.float64)
        if a.numel() != self.n_envs * self.n_agents * 4:
            raise ValueError("actions must have n_envs * n_agents * 4 elements")
        tm = layout == "reference"
        out = torch.empty((self.n_envs, 4 * self.n_agents) if tm else (self.n_envs, self.n_agents, 4), dtype=torch.float32, device=self.device)
        slack = torch.empty(self.n_envs, self.n_agents, dtype=torch.float64, device=self.device) if want_info else None
        moved = torch.empty(self.n_envs, self.n_agents, dtype=torch.uint8, device=self.device) if want_info else None
        self._check(self._lib.fp_safety_project(self._h, _ptr(a), _lib.FP_F64 if a.dtype == torch.float64 else _lib.FP_F32, _ptr(out),
                                                1 if tm else 0, _ptr(slack), _ptr(moved), _lib.stream(self.device)), "fp_safety_project")
        return (out, slack, moved.bool()) if want_info else out

    def load_safety_map(self, A, c, slack_weight=1000.0, v_min=None, v_max=None):
        """The full affine voltage map V = A [P_1, Q_1, ..., P_nb, Q_nb] + c (A [n_bus, 2 n_bus], c [n_bus], fp64 --
        e.g. pred.A, pred.c of a VoltagePredictor) for safety_project_affine.  The limits default to the env's."""
        A = np.ascontiguousarray(A, dtype=np.float64); c = np.ascontiguousarray(c, dtype=np.float64)
        if A.ndim != 2 or c.ndim != 1 or A.shape[0] != c.shape[0]:
            raise ValueError("A must be [n_bus, 2 n_bus] and c [n_bus]")
        v_min = float(self.args_dict["v_min"] if v_min is None else v_min)
        v_max = float(self.args_dict["v_max"] if v_max is None else v_max)
        self._check(self._lib.fp_safety_load_affine(self._h, A.shape[1], A.shape[0], A.ctypes.data_as(C.c_void_p),
                                                    c.ctypes.data_as(C.c_void_p), v_min, v_max, float(slack_weight)),
                    "fp_safety_load_affine")

    def safety_project_affine(self, actions, layout="reference", want_info=False):
        """The safety layer against the map of load_safety_map (every bus coupled to every building), for every env:
        raw policy actions [N, na, 4] -> adjusted setpoints (fp32), layouts as safety_project.  want_info adds
        (slack [N, n_bus] f64, intervened [N, na] bool, status [N] i32: iterations, 0 = already inside, -1 = cap hit)."""
        a = actions.to(self.device).contiguous()
        if a.dtype not in (torch.float32, torch.float64):
            a = a.to(torch.float64)
        if a.numel() != self.n_envs * self.n_agents * 4:
            raise ValueError("actions must have n_envs * n_agents * 4 elements")
        tm = layout == "reference"
        out = torch.empty((self.n_envs, 4 * self.n_agents) if tm else (self.n_envs, self.n_agents, 4), dtype=torch.float32, device=self.device)
        slack = torch.empty(self.n_envs, self.n_bus, dtype=torch.float64, device=self.device) if want_info else None
        moved = torch.empty(self.n_envs, self.n_agents, dtype=torch.uint8, device=self.device) if want_info else None
        status = torch.empty(self.n_envs, dtype=torch.int32, device=self.device) if want_info else None
        self._check(self._lib.fp_safety_project_affine(self._h, _ptr(a), _lib.FP_F64 if a.dtype == torch.float64 else _lib.FP_F32,
                                                       _ptr(out), 1 if tm else 0, _ptr(slack), _ptr(moved), _ptr(status), _lib.stream(self.device)),
                    "fp_safety_project_affine")
        return (out, slack, moved.bool(), status) if want_info else out

    # ------------------------------------------------------------------ statistics
    def episode_stats(self, reduce=True, reset=False):
        """Sums accumulated by every step since the last reset of the statistics (the batched
        form of madrl/models/model.py:247-265).  With torch.distributed initialised and
        reduce=True the vector is all-reduced (NCCL) -- the only collective on this path."""
        self._check(self._lib.fp_stats_read(self._h, _ptr(self._stats), _lib.stream(self.device)), "fp_stats_read")
        out = self._stats.clone()
        if reduce:
            sharding.reduce_stats(out)
        if reset:
            self._check(self._lib.fp_stats_reset(self._h, _lib.stream(self.device)), "fp_stats_reset")
        return sharding.stats_dict(out)

    # ------------------------------------------------------------------ test hooks
    def inject_failure(self, mask):
        """Fault injection: envs with a non-zero byte fail their next power flows."""
        self._inject = self._dev(mask, torch.uint8)
        self._check(self._lib.fp_inject_failure(self._h, _ptr(self._inject)), "fp_inject_failure")

    def launch_count(self):
        return int(self._lib.fp_launch_count(self._h))


class ObsRing:
    """The observation history where the device policy reads it: `ring` [history, n_agents, 6, n_pad] fp32 (env-minor:
    one push writes whole 128-byte lines), `slot` = ring slot of the newest push.  The window of env e / agent a is
    ring[(slot - history + 1 + s) % history, a, :, e] for s = 0 .. history-1 (oldest first); dense() materialises the
    reference's [N, n_agents, 6 * history] layout (get_obs, :387-401)."""

    def __init__(self, env, ring, slot):
        self.env, self.ring, self.slot = env, ring, int(slot)

    def dense(self, out=None):
        env = self.env
        if out is None:
            out = torch.empty(env.n_envs, env.n_agents, env.obs_size, dtype=torch.float32, device=env.device)
        env._check(env._lib.fp_obs_ring_gather(env._h, _ptr(out), _lib.stream(env.device)), "fp_obs_ring_gather")
        return out


class _ExternalCudaBuffer:
    """Exposes library-owned device memory through __cuda_array_interface__ (no copy)."""

    def __init__(self, ptr, nbytes, device_index):
        self.__cuda_array_interface__ = {
            "shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2, "strides": None,
        }
