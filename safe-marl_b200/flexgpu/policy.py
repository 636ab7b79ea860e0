"""The rollout loop on the device (SURVEY 8f ranks 1-2): acting policy, Transition writes, learner feed.

DevicePolicy    the shared-parameter RNNAgent (madrl/agents/rnn_agent.py:8-32) + select_action
                (utils/util.py:50-64) for N envs x n_agents (1 .. 5) per call, through fp_policy_act (tcgen05), reading
                the env's observation ring directly.
DeviceRollout   the body of train_process (madrl/models/model.py:213-254) with nothing crossing PCIe:
                policy -> fused translate_action + step + get_obs -> Transition fields into a DeviceReplayBuffer.
learner_batch   unpack_data (model.py:308-323) on a sampled window: the 12 batch tensors + the MADDPG critic input.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .predictor import DeviceReplayBuffer

N_AGENTS, OBS, HID, ACT = 5, 144, 64, 4          # N_AGENTS: the default agent count (IEEE-33 with five buildings)
MAX_AGENTS = 5                                    # fp_policy_create_agents accepts 1 .. 5
HISTORY, FEATURES = 24, 6                         # the observation ring [HISTORY, n_agents, FEATURES, n_pad] (OBS = 6 x 24)


def transition_fields(n_agents):
    """Transition (model.py:19) as fp32 replay fields, widths per transition (one env-step), for n_agents agents."""
    na = int(n_agents)
    return {"state": na * OBS, "action": na * ACT, "log_prob_a": na * ACT, "value": na, "next_value": na, "reward": na,
            "next_state": na * OBS, "done": 1, "last_step": 1, "action_avail": na * ACT, "last_hid": na * HID, "hid": na * HID}


def weight_shapes(n_agents):
    """RNNAgent.state_dict() shapes, in _WEIGHT_KEYS order: fc1 takes 144 observations + n_agents agent-id columns."""
    return ((HID, OBS + n_agents), (HID,), (HID,), (HID,), (3 * HID, HID), (3 * HID, HID), (3 * HID,), (3 * HID,), (ACT, HID), (ACT,))


def critic_shapes(n_agents):
    """MLPCritic.state_dict() shapes, in _CRITIC_KEYS order: fc1 takes n_agents x (144 + 4) + n_agents inputs."""
    return ((HID, n_agents * (OBS + ACT) + n_agents), (HID,), (HID,), (HID,), (HID, HID), (HID,), (1, HID), (1,))


TRANSITION_FIELDS = transition_fields(N_AGENTS)
_WEIGHT_KEYS = ("fc1.weight", "fc1.bias", "layernorm.weight", "layernorm.bias", "rnn.weight_ih", "rnn.weight_hh",
                "rnn.bias_ih", "rnn.bias_hh", "fc2.weight", "fc2.bias")
_WEIGHT_SHAPES = weight_shapes(N_AGENTS)
_CRITIC_KEYS = ("fc1.weight", "fc1.bias", "layernorm.weight", "layernorm.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias")
_CRITIC_SHAPES = critic_shapes(N_AGENTS)


def _ptr(t):
    if t is None or isinstance(t, C.c_void_p):
        return t
    return C.c_void_p(t.data_ptr())


def round_tf32(w):
    """Round-to-nearest-even to TF32 (10-bit mantissa): how fp_policy_load holds the weights."""
    u = np.ascontiguousarray(w, dtype=np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x0FFF + ((u >> 13) & 1)) & 0xFFFFE000
    return u.astype(np.uint32).view(np.float32).reshape(np.shape(w))


class DevicePolicy:
    """n_agents: the agent count the handle serves (1 .. 5, fixed).  With a state dict it is read from fc1.weight's width
    (144 + n_agents), and a different n_agents raises; without one it defaults to 5."""

    def __init__(self, state_dict=None, device="cuda:0", std=1.0, seed=0, n_agents=None):
        if state_dict is not None:
            shape = tuple(np.shape(state_dict["fc1.weight"]))
            inferred = shape[1] - OBS if len(shape) == 2 else None
            if inferred is None or not 1 <= inferred <= MAX_AGENTS:
                raise ValueError(f"fc1.weight: expected (64, 144 + n_agents) with n_agents in [1, 5], got {shape}")
            if n_agents is not None and int(n_agents) != inferred:
                raise ValueError(f"n_agents={n_agents} conflicts with fc1.weight {shape} (144 + {inferred} inputs: {inferred} agents)")
            n_agents = inferred
        n_agents = N_AGENTS if n_agents is None else int(n_agents)
        if not 1 <= n_agents <= MAX_AGENTS:
            raise ValueError(f"n_agents must be in [1, 5], got {n_agents}")
        self.n_agents = n_agents
        self._ring_dims = (HISTORY, n_agents, FEATURES)
        self.device = torch.device(device)
        if self.device.type != "cuda" or not torch.cuda.is_available():
            raise _lib.FlexGpuError("DevicePolicy needs a CUDA device; there is no CPU fallback")
        self._lib = _lib.lib()
        self._p = C.c_void_p()
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", idx)
        _lib.check(self._lib.fp_policy_create_agents(idx, self.n_agents, C.byref(self._p)), None, "fp_policy_create_agents",
                   self._lib.fp_policy_last_error)
        self.std = float(std)                       # fixed_policy_std (default.yaml: 1.0; gaussian_policy False)
        self.seed = int(seed)
        self._bufs = {}
        self.has_critic = False
        if state_dict is not None:
            self.load_state_dict(state_dict)

    def _check(self, rc, what):
        _lib.check(rc, self._p, what, self._lib.fp_policy_last_error)

    def close(self):
        if getattr(self, "_p", None) is not None and self._p.value:
            self._lib.fp_policy_destroy(self._p)
            self._p = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_state_dict(self, sd):
        """sd: RNNAgent.state_dict() (torch tensors) or a dict of arrays with the same keys."""
        arrs, na = [], self.n_agents
        for k, shape in zip(_WEIGHT_KEYS, weight_shapes(na)):
            v = sd[k]
            a = np.ascontiguousarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v, dtype=np.float32)
            if a.shape != shape:
                raise ValueError(f"{k}: expected {shape}, got {a.shape} (hid_size 64, obs 144 + {na} agent ids, 4 actions)")
            arrs.append(a)
        self._check(self._lib.fp_policy_load(self._p, *[a.ctypes.data_as(C.c_void_p) for a in arrs]), "fp_policy_load")

    def launch_count(self):
        return int(self._lib.fp_policy_launch_count(self._p))

    def load_critic(self, sd):
        """sd: MLPCritic.state_dict() (madrl/critics/mlp_critic.py, as MADDPG.construct_value_net builds it: input
        n_agents x 149, 745 for five agents)."""
        arrs, na = [], self.n_agents
        for k, shape in zip(_CRITIC_KEYS, critic_shapes(na)):
            v = sd[k]
            a = np.ascontiguousarray(v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else v, dtype=np.float32)
            if a.shape != shape:
                raise ValueError(f"critic {k}: expected {shape}, got {a.shape} (hid_size 64, {na} x (144 + 4) + {na} inputs)")
            arrs.append(a)
        self._check(self._lib.fp_critic_load(self._p, *[a.ctypes.data_as(C.c_void_p) for a in arrs]), "fp_critic_load")
        self.has_critic = True

    def _ring(self, ring, slot, n_envs):
        """(ring tensor, slot, n_envs) of an ObsRing or a raw ring, whose shape must be [24, n_agents, 6, n_pad]."""
        if hasattr(ring, "ring"):
            slot, n_envs, ring = ring.slot, ring.env.n_envs, ring.ring
        if tuple(ring.shape)[:-1] != self._ring_dims:
            raise ValueError(f"the observation ring must be [24, {self.n_agents}, 6, n_pad] for this {self.n_agents}-agent policy, "
                             f"got {tuple(ring.shape)}")
        return ring, slot, n_envs

    def value(self, ring, action, slot=None, n_envs=None, out=None):
        """MADDPG.value (maddpg.py:29-76) on the observation ring and `action` [N, n_agents, 4]: [N, n_agents, 1]
        (k_critic, tcgen05)."""
        ring, slot, n_envs = self._ring(ring, slot, n_envs)
        N, na = int(n_envs), self.n_agents
        act = action.to(device=self.device, dtype=torch.float32).contiguous()
        if tuple(act.shape) != (N, na, ACT):
            raise ValueError(f"action must be [n_envs, {na}, 4], got {tuple(act.shape)}")
        if out is not None and tuple(out.shape) != (N, na, 1):
            raise ValueError(f"out must be [n_envs, {na}, 1], got {tuple(out.shape)}")
        out = self._buf("value", (N, na, 1)) if out is None else out
        self._check(self._lib.fp_critic_value(self._p, _ptr(ring), int(slot), int(ring.shape[-1]), N, _ptr(act), _ptr(out), _lib.stream(self.device)),
                    "fp_critic_value")
        return out

    def _buf(self, name, shape):
        b = self._bufs.get(name)
        if b is None or b.shape != shape:
            b = torch.empty(shape, dtype=torch.float32, device=self.device)
            self._bufs[name] = b
        return b

    def act(self, ring, slot=None, n_envs=None, hid_in=None, reset=None, explore=True, eps=None, step=0, hid_out=None,
            want_mean=False, want_logp=True, hid_layout="rows", out="action", mean_out=None):
        """ring: an ObsRing (env.obs_ring() / step(..., return_obs='ring')) or a raw [24, n_agents, 6, n_pad] fp32 tensor
        with `slot` / `n_envs`.  Returns (action [N, na, 4], log_prob [N, na, 4] or None, hid, mean or None), na =
        n_agents; the output tensors are reused by the next call unless hid_out is given (out: name of the reused action
        buffer).  hid_layout: "rows" = [N, na, 64] (the reference's (b, n, hid)), "env_minor" = [na, 64, n_pad] (the
        kernel's native layout: coalesced accesses; hid_out required)."""
        ring, slot, n_envs = self._ring(ring, slot, n_envs)
        n_pad = ring.shape[-1]
        N, na = int(n_envs), self.n_agents
        rows = (N, na, ACT)
        if mean_out is not None and tuple(mean_out.shape) != rows:
            raise ValueError(f"mean_out must be [n_envs, {na}, 4], got {tuple(mean_out.shape)}")
        action = self._buf(out, rows)
        logp = self._buf("logp", rows) if want_logp else None
        mean = mean_out if mean_out is not None else (self._buf("mean", rows) if want_mean else None)
        em = hid_layout == "env_minor"
        hshape = (na, HID, n_pad) if em else (N, na, HID)
        if em and hid_out is None:
            raise ValueError(f"env-minor hidden states are [{na}, 64, n_pad] tensors (hid_out required)")
        if (hid_out is not None and tuple(hid_out.shape) != hshape) or (hid_in is not None and tuple(hid_in.shape) != hshape):
            raise ValueError(f"hidden states of this {na}-agent policy ({hid_layout}) are {list(hshape)} tensors")
        if hid_out is None:
            hid_out = self._buf("hid", hshape)
        if hid_in is not None and hid_in.data_ptr() == hid_out.data_ptr():
            raise ValueError("hid_in and hid_out must be different buffers")
        r = None if reset is None else reset.to(device=self.device, dtype=torch.uint8).contiguous()
        e = None if eps is None else eps.to(device=self.device, dtype=torch.float32).contiguous()
        if e is not None and e.numel() != N * na * ACT:
            raise ValueError(f"eps must hold n_envs x {na} x 4 draws, got {tuple(e.shape)}")
        self._check(self._lib.fp_policy_act(self._p, _ptr(ring), int(slot), int(n_pad), N, _ptr(hid_in), _ptr(r), _ptr(hid_out),
                                            1 if em else 0, _ptr(mean), _ptr(action), _ptr(logp), _ptr(e), self.seed, int(step),
                                            self.std, 1 if explore else 0, _lib.stream(self.device)), "fp_policy_act")
        return action, logp, hid_out, mean

    def sample(self, mean, explore=True, eps=None, step=0, want_logp=True, out="action"):
        """select_action alone on stored fc2 outputs `mean` [N, n_agents, 4] (act(..., want_mean=True)): another exploration
        draw of the same policy evaluation -- bit-identical to calling act() again on the same inputs with these draws."""
        N, na = int(mean.shape[0]), self.n_agents
        if tuple(mean.shape) != (N, na, ACT) or not mean.is_contiguous():
            raise ValueError(f"mean must be a contiguous [n_envs, {na}, 4] tensor, got {tuple(mean.shape)}")
        action = self._buf(out, (N, na, ACT))
        logp = self._buf("logp", (N, na, ACT)) if want_logp else None
        e = None if eps is None else eps.to(device=self.device, dtype=torch.float32).contiguous()
        if e is not None and e.numel() != N * na * ACT:
            raise ValueError(f"eps must hold n_envs x {na} x 4 draws, got {tuple(e.shape)}")
        self._check(self._lib.fp_policy_sample(self._p, _ptr(mean), N, _ptr(action), _ptr(logp), _ptr(e), self.seed, int(step),
                                               self.std, 1 if explore else 0, _lib.stream(self.device)), "fp_policy_sample")
        return action, logp

    def gather_windows(self, ring, n, out, pitch, row0=0, cap=None, slot=None):
        """Dense observation windows [n, n_agents, 144] of envs [0, n) into rows (row0 + e) mod cap of `pitch` floats of
        `out` (a tensor or a device pointer)."""
        ringt, slot, _ = self._ring(ring, slot, n)
        self._check(self._lib.fp_policy_gather_windows(self._p, _ptr(ringt), int(slot), int(ringt.shape[-1]), int(n), _ptr(out),
                                                       int(pitch), int(row0), int(cap if cap is not None else n), _lib.stream(self.device)),
                    "fp_policy_gather_windows")


class DeviceRollout:
    """train_process (model.py:198-267) for N envs at once.  Per step: k_policy (act on the ring + last_hid) ->
    fp_step_ring with FP_F32_POLICY actions (translate_action + step + pushing get_obs, one launch) -> Transition
    fields of the first `record_envs` envs into `replay` (a DeviceReplayBuffer with transition_fields(n_agents)).
    The env's n_agents must be the policy's, and its history 24 (the kernels' K = 6 x 24).  value /
    next_value are stored as zeros: MADDPG's losses recompute both from the critic (maddpg.py:104-107) and never read
    them.  Episodes end together (95 steps, quirk Q1): the finished envs are reset from their Philox streams and their
    hidden state restarts at zero (init_hidden, model.py:211).  An env can also terminate EARLY (solver failure,
    :314-337): with reset_done_each_step=True every step is followed by a masked reset of the envs it finished -- three
    small launches (~55 us at 131 072 envs), no host round trip -- exactly as the reference ends that env's episode and
    starts a new one; without it (the default: failures do not occur on feasible profiles) such an env pays its -200,
    is flagged done / last_step in its Transition, and keeps stepping until the batch's common reset."""

    def __init__(self, env, policy, replay=None, record_envs=None, max_steps=240, reset_done_each_step=False, value_fn=None,
                 fp64_history=False):
        if env.n_agents != policy.n_agents:
            raise ValueError(f"the env has {env.n_agents} agents, the policy {policy.n_agents}: "
                             f"build the policy with DevicePolicy(..., n_agents={env.n_agents})")
        if env.history != HISTORY:
            raise ValueError(f"the device rollout needs an observation history of {HISTORY} steps, the env has {env.history}")
        na = self.na = policy.n_agents
        self.fields = transition_fields(na)
        self.env, self.policy, self.replay = env, policy, replay
        # the loop consumes the fp32 ring only: by default the step stops pushing the fp64 history ring as well
        # (env.set_obs_history); a later env.get_obs() restores it from the ring at fp32 precision
        env.set_obs_history(bool(fp64_history))
        self.N = env.n_envs
        self.R = 0 if replay is None else int(self.N if record_envs is None else min(record_envs, self.N))
        if replay is not None and (dict(replay.fields) != self.fields or self.R > replay.size):
            raise ValueError(f"replay must be a DeviceReplayBuffer(transition_fields({na})) holding at least record_envs rows")
        self.max_steps = int(max_steps)
        self.reset_done_each_step = bool(reset_done_each_step)
        # value_fn: the critic behind the Transition's value / next_value, filled as train_process does (model.py:217, :225-226:
        # the critic on (state, action) and on (next_state, a SECOND sampled action from the policy with the new hidden state;
        # the second policy evaluation doubles k_policy's cost).  "native" = k_critic (tcgen05; policy.load_critic(...) holds the
        # reference's MLPCritic), straight from the observation ring; or a callable (obs [R, na, 144], action [R, na, 4]) ->
        # [R, na, 1], e.g. behaviour_net.value (maddpg.py:29-76) as a torch module.
        self.value_fn = value_fn
        if value_fn == "native" and not policy.has_critic:
            raise ValueError('value_fn="native" needs the critic weights: policy.load_critic(MLPCritic.state_dict())')
        dev = env.device
        self._n_pad = (self.N + 31) // 32 * 32                      # the observation ring's padding (fp_obs_ring)
        # hidden states in the policy kernel's env-minor layout [na, 64, n_pad]; hidden() gives the reference's [N, na, 64]
        self._hid = [torch.zeros(na, HID, self._n_pad, device=dev), torch.zeros(na, HID, self._n_pad, device=dev)]
        self._cur = 0
        self._reset_mask = None
        self._done_mask = None
        # with a critic, the policy evaluation behind the next-value action (model.py:225: policy(next_state, hid)) IS the
        # evaluation the next step starts with (:215-216: same observations, same hidden state) -- only the exploration draw
        # differs.  Its fc2 outputs and new hidden state are kept, and the next step re-draws (fp_policy_sample) instead of
        # running k_policy again, unless a reset intervened.  Same bits as evaluating twice.
        self._mean2 = torch.empty(self.N, na, ACT, device=dev) if value_fn is not None else None
        self._cache_valid = False
        self.t = 0                                  # step within the episode
        self.total_steps = 0
        self.ring = None
        self._fptr = {}
        if replay is not None:
            for i, k in enumerate(replay.names):
                p = C.c_void_p()
                replay._check(replay._lib.fp_replay_field_ptr(replay._r, i, C.byref(p)), "fp_replay_field_ptr")
                self._fptr[k] = p
            if value_fn is not None:
                if value_fn != "native":
                    self._dense = torch.empty(self.R, na * OBS, device=dev)
                self._hid_scratch = torch.empty(na, HID, self._n_pad, device=dev)

    def reset(self):
        self.ring = self.env.reset(return_obs="ring")              # state, _ = env.reset() (model.py:208)
        self._hid[self._cur].zero_()                                # init_hidden (model.py:211)
        self._reset_mask = None
        self._cache_valid = False
        self.t = 0
        return self.ring

    def _rows(self, name, src, pos):
        pol = self.policy
        w = self.fields[name]
        pol._check(pol._lib.fp_policy_rows_to_ring(pol._p, _ptr(src), self.R, w, self._fptr[name], pos, self.replay.size,
                                                   _lib.stream(pol.device)), "fp_policy_rows_to_ring")

    def _hidden_rows(self, name, hid_em, pos, zero_mask=None):
        pol = self.policy
        pol._check(pol._lib.fp_policy_hidden_to_ring(pol._p, _ptr(hid_em), self._n_pad, self.R, self._fptr[name], pos, self.replay.size,
                                                     _ptr(zero_mask), _lib.stream(pol.device)), "fp_policy_hidden_to_ring")

    def hidden(self):
        """The current hidden state in the reference's layout [N, n_agents, 64] (a copy)."""
        return self._hid[self._cur][:, :, :self.N].permute(2, 0, 1).contiguous()

    def _dense_obs(self):
        self.policy.gather_windows(self.ring, self.R, self._dense, self.na * OBS, 0, self.R)
        return self._dense.view(self.R, self.na, OBS)

    def _value(self, action, name):
        """The critic on (the ring as it stands, action) for the recorded envs: [R, na] fp32, contiguous."""
        if self.value_fn == "native":
            out = self.policy._buf(name, (self.R, self.na, 1))              # the recorded envs only
            return self.policy.value(self.ring.ring, action[:self.R], slot=self.ring.slot, n_envs=self.R, out=out).view(self.R, self.na)
        with torch.no_grad():
            return self.value_fn(self._dense_obs(), action[:self.R]).reshape(self.R, self.na).float().contiguous()

    def step(self, explore=True, eps=None, eps_next=None):
        if self.ring is None:
            self.reset()
        env, pol = self.env, self.policy
        last_hid, hid = self._hid[self._cur], self._hid[1 - self._cur]
        if self._cache_valid and self._reset_mask is None:          # evaluated already for the previous step's next-value action: re-draw
            action, logp = pol.sample(self._mean2, explore=explore, eps=eps, step=self.total_steps)
            self._hid[1 - self._cur], self._hid_scratch = self._hid_scratch, self._hid[1 - self._cur]
            hid = self._hid[1 - self._cur]
            pos, state_written = (self.replay.reserve(self.R) if self.R else None), False
        else:
            pos, state_written = (self.replay.reserve(self.R) if self.R else None), False
            if self.R and self.ring.ring.shape[-1] >= 128:          # `state` rows written by k_policy's writer warps from the blocks it stages
                pol._check(pol._lib.fp_policy_state_sink(pol._p, self._fptr["state"], self.fields["state"], pos, self.replay.size, self.R),
                           "fp_policy_state_sink")
                state_written = True
            action, logp, hid, _ = pol.act(self.ring, hid_in=last_hid, reset=self._reset_mask, explore=explore, eps=eps,
                                           step=self.total_steps, hid_out=hid, hid_layout="env_minor")  # model.py:215-216
        self._cache_valid = False
        if self.R:
            if not state_written:
                pol.gather_windows(self.ring, self.R, self._fptr["state"], self.fields["state"], pos, self.replay.size)
            self._hidden_rows("last_hid", last_hid, pos, self._reset_mask)     # a restarted env's last_hid is the zero state it acted from
            if self.value_fn is not None:                                      # value = critic(state, action) (model.py:217)
                self._rows("value", self._value(action, "value"), pos)
        # translate_action (:218) + env.step (:220) + get_obs (:223) in one launch
        reward, done, info, self.ring = env.step(action, translate=True, want_info=False, return_obs="ring")
        self.t += 1
        self.total_steps += 1
        if self.R:
            pol.gather_windows(self.ring, self.R, self._fptr["next_state"], self.fields["next_state"], pos, self.replay.size)
            self._hidden_rows("hid", hid, pos)
            if self.value_fn is not None:   # next_value = critic(next_state, a second sampled action from the new hidden state) (model.py:225-226)
                a2, _, _, _ = pol.act(self.ring, hid_in=hid, explore=explore, eps=eps_next, step=(1 << 40) + self.total_steps,
                                      hid_out=self._hid_scratch, hid_layout="env_minor", want_logp=False, out="action2",
                                      mean_out=self._mean2)
                self._cache_valid = True
                self._rows("next_value", self._value(a2, "next_value"), pos)
            # action, log_prob_a, reward per agent, done, last_step, action_avail (and value / next_value = 0 without a critic): one launch
            f = self._fptr
            pol._check(pol._lib.fp_policy_transition_tail(
                pol._p, _ptr(action), _ptr(logp), _ptr(reward), _ptr(done), self.R, 1 if self.t == self.max_steps else 0,
                1 if self.value_fn is None else 0, f["action"], f["log_prob_a"], f["value"], f["next_value"], f["reward"], f["done"],
                f["last_step"], f["action_avail"], pos, self.replay.size, _lib.stream(pol.device)), "fp_policy_transition_tail")
        self._cur = 1 - self._cur
        self._reset_mask = None
        if self.t >= env.episode_limit - 1 or self.t >= self.max_steps:        # every env of the batch has terminated (Q1)
            mask = done.to(torch.uint8) if self.t < self.max_steps else torch.ones_like(done, dtype=torch.uint8)
            self.ring = env.reset(mask=mask, return_obs="ring")
            self._reset_mask = mask.clone()
            self.t = 0
        elif self.reset_done_each_step:                                         # early terminations (solver failure): their own new episode
            if self._done_mask is None:
                self._done_mask = torch.empty(self.N, dtype=torch.uint8, device=done.device)
            self._done_mask.copy_(done)
            self.ring = env.reset(mask=self._done_mask, return_obs="ring", retries=0)
            self._reset_mask = self._done_mask
        return reward, done


def learner_batch(policy, replay, batch_size, start=None, reward_normalisation=True, critic_input=True):
    """unpack_data (model.py:308-323) on `batch_size` consecutive transitions (get_batch, replay_buffer.py:14-21):
    the reference's 12 tensors in its shapes -- including its quirk log_prob_a = action (:313) -- plus, for MADDPG,
    `critic_in` [batch * na, na x 149] (maddpg.py:29-66; [batch * 5, 745] for five agents), na = policy.n_agents.
    Everything stays on the device."""
    na = policy.n_agents
    if dict(replay.fields) != transition_fields(na):
        raise ValueError(f"replay must be a DeviceReplayBuffer(transition_fields({na})) for this {na}-agent policy")
    b = replay.get_batch(batch_size, start=start)
    B = batch_size
    out = {
        "state": b["state"].view(B, na, OBS), "action": b["action"].view(B, na, ACT),
        "log_prob_a": b["action"].view(B, na, ACT),                           # sic: model.py:313 concatenates batch.action
        "value": b["value"].view(B, na, 1), "next_value": b["next_value"].view(B, na, 1),
        "reward": b["reward"], "next_state": b["next_state"].view(B, na, OBS), "done": b["done"].view(B, 1),
        "last_step": b["last_step"].view(B, 1), "action_avail": b["action_avail"].view(B, na, ACT),
        "last_hid": b["last_hid"].view(B, na, HID), "hid": b["hid"].view(B, na, HID),
    }
    crit = torch.empty(B * na, na * (OBS + 1 + ACT), device=replay.device) if critic_input else None
    rn = torch.empty(B, na, device=replay.device) if reward_normalisation else None
    policy._check(policy._lib.fp_learner_feed(policy._p, _ptr(b["state"]), _ptr(b["action"]), _ptr(b["reward"]), B, _ptr(crit),
                                              _ptr(rn), _lib.stream(policy.device)), "fp_learner_feed")
    if reward_normalisation:
        out["reward"] = rn
    if critic_input:
        out["critic_in"] = crit
    return out


def smoke(env, device):
    """Tiny policy + rollout invocation for __graft_entry__.smoke(): k_policy on the env's own observation ring against
    a plain torch fp32 evaluation of RNNAgent.forward (rnn_agent.py:24-32) with the same (TF32-rounded) matrices, for the
    env's own agent count."""
    na = env.n_agents
    g = torch.Generator().manual_seed(0)
    sd = {k: (torch.randn(s, generator=g) * 0.1) for k, s in zip(_WEIGHT_KEYS, weight_shapes(na))}
    sd["layernorm.weight"] = 1.0 + sd["layernorm.weight"]
    pol = DevicePolicy(sd, device=device)
    ring = env.obs_ring()
    n = env.n_envs
    h_in = (torch.rand(n, na, HID, generator=g) - 0.5).to(device)
    act, _, hid, mean = pol.act(ring, hid_in=h_in, explore=False, want_mean=True, hid_out=torch.empty(n, na, HID, device=device))
    w = {k: v.to(device) for k, v in sd.items()}
    for k in ("rnn.weight_ih", "rnn.weight_hh"):
        w[k] = torch.from_numpy(round_tf32(sd[k].numpy())).to(device)
    w1 = sd["fc1.weight"].numpy().copy(); w1[:, :OBS] = round_tf32(w1[:, :OBS]); w["fc1.weight"] = torch.from_numpy(w1).to(device)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        obs = ring.dense().view(n * na, OBS)
        x = torch.cat([obs, torch.eye(na, device=device).repeat(n, 1)], dim=1) @ w["fc1.weight"].T + w["fc1.bias"]
        x = torch.relu(torch.nn.functional.layer_norm(x, (HID,), w["layernorm.weight"], w["layernorm.bias"], 1e-5))
        h0 = h_in.view(-1, HID)
        gi = x @ w["rnn.weight_ih"].T + w["rnn.bias_ih"]; gh = h0 @ w["rnn.weight_hh"].T + w["rnn.bias_hh"]
        r = torch.sigmoid(gi[:, :HID] + gh[:, :HID]); z = torch.sigmoid(gi[:, HID:2 * HID] + gh[:, HID:2 * HID])
        nn_ = torch.tanh(gi[:, 2 * HID:] + r * gh[:, 2 * HID:])
        h1 = (1 - z) * nn_ + z * h0
        m = h1 @ w["fc2.weight"].T + w["fc2.bias"]
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    err = max(float((mean.view(-1, ACT) - m).abs().max()), float((hid.view(-1, HID) - h1).abs().max()),
              float((act.view(-1, ACT) - torch.tanh(m)).abs().max()))
    assert err < 5e-5, f"policy mismatch {err}"
    ro = DeviceRollout(env, pol)
    ro.ring = ring
    ro.step()
    pol.close()
    return err


def critic_input(policy, state, action):
    """The MADDPG critic's input rows (maddpg.py:29-66) for dense observations [B, na, 144] and actions [B, na, 4], na =
    policy.n_agents: [B * na, na x 149] = all agents' observations | one-hot agent id | all agents' actions."""
    B, na = state.shape[0], policy.n_agents
    st = state.reshape(B, na * OBS).contiguous(); ac = action.reshape(B, na * ACT).float().contiguous()
    out = torch.empty(B * na, na * (OBS + 1 + ACT), device=st.device)
    policy._check(policy._lib.fp_learner_feed(policy._p, _ptr(st), _ptr(ac), None, B, _ptr(out), None, _lib.stream(policy.device)), "fp_learner_feed")
    return out
