"""fp64 references of the device rollout's kernels for any agent count na in 1 .. 5, shared by the GPU tests.

The error model is the one stated in tests/test_gpu_rollout_scale.py's docstring; only the shapes follow na: the policy's
fc1 has 144 + na inputs (its kappa does not depend on na: K = 144 either way), the critic's fc1 na x 144 observation and
na x 4 action columns, K padded to 24 for the actions: m = 2 (18 na + 3) MMA instructions, kappa = 1 + m / 4."""
import numpy as np
import torch

CHUNK = 65536
U = 2.0 ** -24
KAPPA_FC1, KAPPA_RZ, KAPPA_N, KAPPA_CFC2 = 19.0, 9.0, 5.0, 5.0
C_SIG = C_TANH = 6e-7
C_TANH_FAST = 8 * 2.0 ** -23
SENT = 7.25e6                                       # sentinel: no output of these kernels comes near it
KEYS = ("fc1.weight", "fc1.bias", "layernorm.weight", "layernorm.bias", "rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih",
        "rnn.bias_hh", "fc2.weight", "fc2.bias")
CKEYS = ("fc1.weight", "fc1.bias", "layernorm.weight", "layernorm.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias")


def kappa_critic_fc1(na):
    return 1 + 2 * (18 * na + 3) / 4


def tf32(w):
    from flexgpu.policy import round_tf32
    return round_tf32(np.asarray(w, dtype=np.float32)).astype(np.float64)


def f32(x):
    return np.asarray(x, dtype=np.float32).astype(np.float64)


def realistic_policy(seed, na):
    """An RNNAgent of na agents with torch's default initialisation spread and a trained-looking LayerNorm."""
    rng = np.random.default_rng(seed)
    k1, kg = 1 / np.sqrt(144 + na), 1 / 8
    sd = {"fc1.weight": rng.uniform(-k1, k1, (64, 144 + na)), "fc1.bias": rng.uniform(-k1, k1, 64),
          "layernorm.weight": 1 + rng.normal(0, 0.2, 64), "layernorm.bias": rng.normal(0, 0.2, 64),
          "rnn.weight_ih": rng.uniform(-kg, kg, (192, 64)), "rnn.weight_hh": rng.uniform(-kg, kg, (192, 64)),
          "rnn.bias_ih": rng.uniform(-kg, kg, 192), "rnn.bias_hh": rng.uniform(-kg, kg, 192),
          "fc2.weight": rng.uniform(-kg, kg, (4, 64)), "fc2.bias": rng.uniform(-kg, kg, 4)}
    return {k: v.astype(np.float32) for k, v in sd.items()}


def realistic_critic(seed, na):
    rng = np.random.default_rng(seed)
    k1, k2 = 1 / np.sqrt(149 * na), 1 / 8
    sd = {"fc1.weight": rng.uniform(-k1, k1, (64, 149 * na)), "fc1.bias": rng.uniform(-k1, k1, 64),
          "layernorm.weight": 1 + rng.normal(0, 0.2, 64), "layernorm.bias": rng.normal(0, 0.2, 64),
          "fc2.weight": rng.uniform(-k2, k2, (64, 64)), "fc2.bias": rng.uniform(-k2, k2, 64),
          "fc3.weight": rng.uniform(-k2, k2, (1, 64)), "fc3.bias": rng.uniform(-k2, k2, 1)}
    return {k: v.astype(np.float32) for k, v in sd.items()}


def random_ring(n, na, seed, cuda):
    """A [24, na, 6, n_pad] ring of observation-like values (per-feature scales, rows differ) inside a larger allocation
    filled with NaN: the env columns [n, n_pad) and everything past the ring's last element are NaN, so a read past the
    last agent or env poisons an output row.  Returns (ring view, the whole allocation)."""
    n_pad = (n + 31) // 32 * 32
    g = torch.Generator(device=cuda).manual_seed(seed)
    scale = torch.tensor([0.3, 1.0, 0.05, 0.8, 0.02, 1.5], device=cuda).view(1, 1, 6, 1)
    size = 24 * na * 6 * n_pad
    whole = torch.full((64 + size + 24 * 6 * n_pad + 4096,), float("nan"), device=cuda)
    ring = whole[64:64 + size].view(24, na, 6, n_pad)                   # 256-byte aligned: the TMA path stays available
    ring[:, :, :, :n] = scale * (0.5 + torch.randn(24, na, 6, n, device=cuda, generator=g))
    return ring, whole


def windows(ring, slot, e0, e1):
    """Dense windows [c, na, 144] (oldest entry first) of envs [e0, e1) by plain indexing of the ring."""
    na = ring.shape[1]
    idx = torch.tensor([(slot + 1 + r) % 24 for r in range(24)], device=ring.device)
    return ring[:, :, :, e0:e1][idx].permute(3, 1, 0, 2).reshape(e1 - e0, na, 144)


def policy_mats(sd, dev):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
    w1 = np.asarray(sd["fc1.weight"], dtype=np.float32)
    na = w1.shape[1] - 144
    b1a = np.stack([f32(np.float32(sd["fc1.bias"]) + w1[:, 144 + a]) for a in range(na)])          # one fp32 addition
    return {"W1": t(tf32(w1[:, :144])), "b1a": t(b1a), "g": t(f32(sd["layernorm.weight"])), "b": t(f32(sd["layernorm.bias"])),
            "Wih": t(tf32(sd["rnn.weight_ih"])), "Whh": t(tf32(sd["rnn.weight_hh"])), "bih": t(f32(sd["rnn.bias_ih"])),
            "bhh": t(f32(sd["rnn.bias_hh"])), "W2": t(f32(sd["fc2.weight"])), "b2": t(f32(sd["fc2.bias"]))}


def critic_mats(sd, dev):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
    w1 = np.asarray(sd["fc1.weight"], dtype=np.float32)
    na = w1.shape[1] // 149
    b1a = np.stack([f32(np.float32(sd["fc1.bias"]) + w1[:, 144 * na + a]) for a in range(na)])
    return {"na": na, "Wo": t(tf32(w1[:, :144 * na])), "Wa": t(tf32(w1[:, 145 * na:])), "b1a": t(b1a),
            "g": t(f32(sd["layernorm.weight"])), "b": t(f32(sd["layernorm.bias"])), "W2": t(tf32(sd["fc2.weight"])),
            "b2": t(f32(sd["fc2.bias"])), "w3": t(f32(sd["fc3.weight"])[0]), "b3": float(np.float32(sd["fc3.bias"][0]))}


def critic_reference(M, obs_all, act):
    """fp64 critic of obs_all [c, na x 144], act [c, na x 4]: value [c, na] and its bound."""
    x, ac = obs_all.double(), act.double()
    acc = x @ M["Wo"].T + ac @ M["Wa"].T                                            # [c, 64]
    e_acc = kappa_critic_fc1(M["na"]) * 2.0 ** -20 * (x.abs() @ M["Wo"].abs().T + ac.abs() @ M["Wa"].abs().T)
    v = acc[:, None, :] + M["b1a"][None]                                          # [c, na, 64]
    e1 = e_acc[:, None, :] + ulp(v)
    y, e_y = layernorm_bound(v, e1, M["g"], M["b"])
    q0 = torch.relu(y)
    u = q0 @ M["W2"].T + M["b2"]
    e_u = e_y @ M["W2"].abs().T + KAPPA_CFC2 * 2.0 ** -20 * (q0 @ M["W2"].abs().T) + ulp(u)
    q = torch.relu(u)
    val = q @ M["w3"] + M["b3"]
    e_val = e_u @ M["w3"].abs() + 2.0 ** -18 * (q @ M["w3"].abs() + abs(M["b3"]))
    return val, e_val


def ulp(x):
    """fp32 spacing of |x| (x float64): 2^(exponent - 23), at least the smallest normal's."""
    m, e = torch.frexp(x.abs().float().double())
    return torch.where(m == 0, torch.full_like(x, 2.0 ** -149), torch.ldexp(torch.ones_like(x), (e - 24).clamp(min=-149)))


def layernorm_bound(v, e1, g, b):
    """Centred LayerNorm of v [.., 64] (fp64) with input error e1: (y, e_y) as in the module docstring."""
    mu = v.mean(-1, keepdim=True)
    vq = v.view(*v.shape[:-1], 4, 16)
    dq = U * vq.cumsum(-1)[..., 1:].abs().sum(-1) / 16                                # rounding of the four 16-term means
    mq = vq.mean(-1)
    merge = U * ((mq[..., 0] + mq[..., 1]).abs() + (mq[..., 2] + mq[..., 3]).abs() + mq.sum(-1).abs())[..., None] / 4
    e_mu = e1.mean(-1, keepdim=True) + dq.mean(-1, keepdim=True) + merge
    d = v - mu
    var = (d * d).mean(-1, keepdim=True)
    # input error; the centres' rounding: first order through the between-quarter term of the merge, second order in M2
    e_var = 2 * (d.abs() * e1).mean(-1, keepdim=True) + e1.mean(-1, keepdim=True) ** 2 + 2.0 ** -19 * var + \
        ((mq - mu).abs() * (dq + merge)).mean(-1, keepdim=True) + (dq.amax(-1, keepdim=True) + e_mu) ** 2
    rstd = 1 / torch.sqrt(var + 1e-5)
    e_r = e_var / (2 * (var + 1e-5 - e_var).clamp(min=1e-12)) + 2.0 ** -21
    y = d * rstd * g + b
    e_y = g.abs() * rstd * (1 + e_r) * (e1 + e_mu) + g.abs() * d.abs() * rstd * (e_r + 2.0 ** -23) + ulp(y)
    return y, e_y


def action_bound(m, e_m, z, e_z, std, explore):
    """(a, e_a, x, e_x) of select_action at the reference mean m with draws z (fp64) of error e_z."""
    if not explore:
        x, e_x = m, e_m
    else:
        x = m + std * z
        e_x = e_m + std * e_z + ulp(x)
    a = torch.tanh(x)
    e_a = (1 - a * a + 2 * e_x).clamp(max=1) * e_x + C_TANH_FAST
    return a, e_a, x, e_x


def logp_bound(a, e_a, z, e_z, x, std):
    """Reference log-probability and its per-element bound (module docstring)."""
    lp = -0.5 * z * z - np.log(std) - 0.5 * np.log(2 * np.pi) - torch.log(1 - a * a + 1e-6)
    d = std * z
    e_gauss = (z.abs() / std) * (ulp(x) + ulp(d) + std * e_z) + e_z * e_z / 2 + 4 * U * z * z / 2 + 2 * U
    w = 1 - a * a + 1e-6
    dw = 2 * a.abs() * e_a + e_a * e_a + 2.0 ** -23
    e_log = dw / torch.clamp(w - dw, min=0.99e-6)
    logf = torch.where((w >= 0.5) & (w <= 2), torch.full_like(w, 2.0 ** -21.41), 3 * ulp(torch.log(w)))
    return lp, e_gauss + e_log + logf + ulp(lp)


def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on uint32 arrays (counter words c0..c3, key k0, k1), as flex_common.cuh philox4x32_10."""
    c = [np.asarray(v, dtype=np.uint32) for v in (c0, c1, c2, c3)]
    k0, k1 = np.uint32(k0), np.uint32(k1)
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    for _ in range(10):
        p0 = M0 * c[0].astype(np.uint64)
        p1 = M1 * c[2].astype(np.uint64)
        c = [(p1 >> np.uint64(32)).astype(np.uint32) ^ c[1] ^ k0, (p1 & np.uint64(0xFFFFFFFF)).astype(np.uint32),
             (p0 >> np.uint64(32)).astype(np.uint32) ^ c[3] ^ k1, (p0 & np.uint64(0xFFFFFFFF)).astype(np.uint32)]
        k0 = np.uint32((int(k0) + 0x9E3779B9) & 0xFFFFFFFF)
        k1 = np.uint32((int(k1) + 0xBB67AE85) & 0xFFFFFFFF)
    return c


def u53(a, b):
    return ((a >> np.uint32(5)).astype(np.uint64) << np.uint64(26) | (b >> np.uint32(6)).astype(np.uint64)).astype(np.float64) / 2.0 ** 53


def philox_normals(rows, seed, step):
    """The four exploration normals of rows [rows] (fp64 Box-Muller on the exact fp32 uniforms) and their fp32 error bound."""
    rows = np.asarray(rows, dtype=np.uint64)
    s = np.uint64(step)
    x, y, z_, w = philox((rows & np.uint64(0xFFFFFFFF)).astype(np.uint32), (rows >> np.uint64(32)).astype(np.uint32),
                         np.full(rows.shape, int(step) & 0xFFFFFFFF, np.uint32), np.full(rows.shape, int(s >> np.uint64(32)), np.uint32),
                         seed & 0xFFFFFFFF, seed >> 32)
    u0 = ((x >> np.uint32(8)).astype(np.float64) + 1) / 2.0 ** 24
    u1 = (y >> np.uint32(8)).astype(np.float64) / 2.0 ** 24
    u2 = ((z_ >> np.uint32(8)).astype(np.float64) + 1) / 2.0 ** 24
    u3 = (w >> np.uint32(8)).astype(np.float64) / 2.0 ** 24
    out, err = [], []
    for ua, ub in ((u0, u1), (u2, u3)):
        L = np.log(ua)
        ra = np.sqrt(-2 * L)
        e_L = np.where(ua >= 0.5, 2.0 ** -21.41, 3 * np.spacing(np.abs(L).astype(np.float32)).astype(np.float64))
        e_ra = 2 * e_L / (np.sqrt(2 * np.abs(L) + 2 * e_L) + ra) + U * ra
        ang = 2 * np.pi * ub
        e_trig = 2.0 ** -20.5 + 2 * U * 2 * np.pi
        for f in (np.cos, np.sin):
            zz = ra * f(ang)
            out.append(zz)
            err.append(e_ra * np.abs(f(ang)) + ra * e_trig + np.spacing(np.abs(zz).astype(np.float32)).astype(np.float64))
    return np.stack(out, -1), np.stack(err, -1)


class Worst:
    def __init__(self, tag):
        self.tag, self.w = tag, {}

    def check(self, name, got, want, bound, key="", rms=False):
        err = (got.double() - want).abs()
        r = err / bound
        ratio = float(r.max())
        k = f"{name}{key}"
        self.w[k] = max(self.w.get(k, 0.0), ratio)
        bad = ~(err <= bound)
        assert not bool(bad.any()), (self.tag, k, int(bad.sum()), ratio)
        if rms:
            # The bound adds |W| e over 64 or more terms with worst-case signs; independent roundings add in quadrature and
            # are a fraction of their worst case, so over a whole launch the RMS of err / bound stays far below 1 / 64.  An
            # error that is not rounding -- a dropped or truncated product, a wrong weight -- does not average out.
            q = float(torch.sqrt((r * r).mean()))
            self.w[k + " rms"] = max(self.w.get(k + " rms", 0.0), q)
            assert q < 1 / 64, (self.tag, k, "rms", q)

    def report(self):
        print(f"max(err/bound) {self.tag}: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(self.w.items())))

def policy_reference(M, obs, h):
    """fp64 RNNAgent forward of obs [c, na, 144] (fp32 values) and h [c, na, 64]: mean, h', and their bounds."""
    x = obs.double()
    v = x @ M["W1"].T + M["b1a"][None]                                                 # [c, na, 64]
    e1 = KAPPA_FC1 * 2.0 ** -20 * (x.abs() @ M["W1"].abs().T) + ulp(v)
    y, e_y = layernorm_bound(v, e1, M["g"], M["b"])
    xr, e_x = torch.relu(y), e_y
    Wih, Whh = M["Wih"], M["Whh"]
    gi, gh = xr @ Wih.T, h @ Whh.T
    Ai, Ah = Wih.abs(), Whh.abs()
    sx, sh = xr @ Ai.T, h.abs() @ Ah.T
    bsum = M["bih"] + M["bhh"]
    arg_rz = gi[..., :128] + gh[..., :128] + bsum[:128]
    e_rz = e_x @ Ai[:128].T + KAPPA_RZ * 2.0 ** -20 * (sx[..., :128] + sh[..., :128]) + \
        2.0 ** -23 * ((gi[..., :128] + gh[..., :128]).abs() + bsum[:128].abs())
    rz = torch.sigmoid(arg_rz)
    e_g = 0.25 * e_rz + C_SIG
    r, z, e_r, e_z = rz[..., :64], rz[..., 64:], e_g[..., :64], e_g[..., 64:]
    gin, ghn = gi[..., 128:] + M["bih"][128:], gh[..., 128:] + M["bhh"][128:]
    e_gin = e_x @ Ai[128:].T + KAPPA_N * 2.0 ** -20 * sx[..., 128:]
    e_ghn = KAPPA_N * 2.0 ** -20 * sh[..., 128:]
    e_an = e_gin + r * e_ghn + ghn.abs() * e_r + 2.0 ** -22 * (gi[..., 128:].abs() + M["bih"][128:].abs() +
                                                              r * (gh[..., 128:].abs() + M["bhh"][128:].abs()))
    n = torch.tanh(gin + r * ghn)
    e_n = (1 - n * n + e_an).clamp(max=1) * e_an + C_TANH
    h1 = n + z * (h - n)
    e_h = (h - n).abs() * e_z + (1 - z + e_z) * e_n + U * (h - n).abs() + ulp(h1)
    m = h1 @ M["W2"].T + M["b2"]
    e_m = e_h @ M["W2"].abs().T + 2.0 ** -18 * (h1.abs() @ M["W2"].abs().T + M["b2"].abs())
    return m, e_m, h1, e_h


def torch_mats(sd, dev, critic=False):
    """The loaders' matrices as fp32 torch tensors: fc1's observation / action columns and the GRU / critic fc2 matrices
    TF32-rounded, everything else as given (what policy.smoke() compares against)."""
    w = {k: torch.from_numpy(np.asarray(v, dtype=np.float32).copy()) for k, v in sd.items()}
    if critic:
        na = w["fc1.weight"].shape[1] // 149
        w1 = w["fc1.weight"].numpy().copy()
        w1[:, :144 * na] = tf32(w1[:, :144 * na]); w1[:, 145 * na:] = tf32(w1[:, 145 * na:])
        w["fc1.weight"] = torch.from_numpy(w1.astype(np.float32)); w["fc2.weight"] = torch.from_numpy(tf32(sd["fc2.weight"]).astype(np.float32))
    else:
        w1 = w["fc1.weight"].numpy().copy(); w1[:, :144] = tf32(w1[:, :144])
        w["fc1.weight"] = torch.from_numpy(w1.astype(np.float32))
        for k in ("rnn.weight_ih", "rnn.weight_hh"):
            w[k] = torch.from_numpy(tf32(sd[k]).astype(np.float32))
    return {k: v.to(dev) for k, v in w.items()}


def rnn_agent_torch(w, obs, h):
    """RNNAgent.forward (rnn_agent.py:24-32) in torch fp32 on obs [N, na, 144] with the one-hot agent id, h [N, na, 64]:
    (mean [N, na, 4], h' [N, na, 64])."""
    N, na = obs.shape[0], obs.shape[1]
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        x = torch.cat([obs.reshape(N * na, 144), torch.eye(na, device=obs.device).repeat(N, 1)], 1) @ w["fc1.weight"].T + w["fc1.bias"]
        x = torch.relu(torch.nn.functional.layer_norm(x, (64,), w["layernorm.weight"], w["layernorm.bias"], 1e-5))
        h0 = h.reshape(N * na, 64)
        gi = x @ w["rnn.weight_ih"].T + w["rnn.bias_ih"]; gh = h0 @ w["rnn.weight_hh"].T + w["rnn.bias_hh"]
        r = torch.sigmoid(gi[:, :64] + gh[:, :64]); z = torch.sigmoid(gi[:, 64:128] + gh[:, 64:128])
        n_ = torch.tanh(gi[:, 128:] + r * gh[:, 128:])
        h1 = (1 - z) * n_ + z * h0
        m = h1 @ w["fc2.weight"].T + w["fc2.bias"]
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return m.view(N, na, 4), h1.view(N, na, 64)


def critic_input_torch(obs, act):
    """MADDPG.value's input rows (maddpg.py:29-66) by torch.cat: [N * na, na x 149]."""
    N, na = obs.shape[0], obs.shape[1]
    o = obs.reshape(N, 1, na * 144).expand(N, na, na * 144)
    a = act.reshape(N, 1, na * 4).expand(N, na, na * 4)
    eye = torch.eye(na, device=obs.device).expand(N, na, na)
    return torch.cat([o, eye, a], 2).reshape(N * na, na * 149)


def mlp_critic_torch(w, obs, act):
    """MLPCritic (mlp_critic.py:5-36) in torch fp32: [N, na, 1]."""
    N, na = obs.shape[0], obs.shape[1]
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        x = critic_input_torch(obs.float(), act.float()) @ w["fc1.weight"].T + w["fc1.bias"]
        x = torch.relu(torch.nn.functional.layer_norm(x, (64,), w["layernorm.weight"], w["layernorm.bias"], 1e-5))
        x = torch.relu(x @ w["fc2.weight"].T + w["fc2.bias"])
        v = x @ w["fc3.weight"].T + w["fc3.bias"]
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return v.view(N, na, 1)
