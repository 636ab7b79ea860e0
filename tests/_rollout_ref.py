"""fp64 references of the device rollout's kernels (k_policy, k_sample, k_critic) for any agent count na in 1 .. 5, their
per-element error model, and the drivers that run the kernels into sentinel-filled outputs and check every row.

Reference.  torch float64 on the device, in chunks of 65 536 envs, from the raw observation ring by plain indexing
(window entry r of env e, agent a, feature f = ring[(slot + 1 + r) % 24, a, f, e]), with exactly the matrices the loaders
hold: fc1's observation (and, for the critic, action) columns, the GRU matrices and the critic's fc2 rounded to TF32
(flexgpu.policy.round_tf32); biases, LayerNorm parameters, the policy's fc2 and the critic's fc3 unrounded fp32; the
one-hot column folded into the bias by one fp32 addition.

Error model, per element, propagated in float64 next to the reference (u = 2^-24, ulp = fp32 spacing of the value):
  * tcgen05 GEMM, A = activations split x = hi + lo (hi TF32-exact), B = TF32 weights, fp32 accumulator, m MMA instructions
    of K = 8 into one accumulator:  e <= kappa 2^-20 |W||x|,  kappa = 1 + m / 4.  The 1 is lo's own truncation to TF32
    (|lo| < 2^-10 |x|, truncated to 11 bits: < 2^-20 |x|); hi x W is exact (11 x 11 bits).  Each instruction adds its
    products to the accumulator with at most 2 ulp (truncating alignment) of a magnitude <= sum |W||x|: 2 m 2^-23 =
    (m / 4) 2^-20.  fc1: m = 2 x 18 (policy, K = 144 whatever na: kappa = 19), 2 x (18 na + 3) (critic, na x 144
    observation columns and na x 4 action columns padded to K = 24: kappa_critic_fc1(na), 47.5 at na = 5); GRU: m = 32
    for r | z (x and h sides in one accumulator: kappa = 9), 16 for gi_n and gh_n (kappa = 5); critic fc2: m = 16
    (kappa = 5).  A bias is added in fp32 after the MMA: + ulp(v).
  * LayerNorm, centred (mean_q, M2_q per 16-column quarter, Chan merge): e_mu = mean(e1) + the rounding of the sums in
    the kernel's order (u times every partial sum, from the reference values); e_var = 2 mean(|v - mu| e1) + mean(e1)^2
    + e_mu^2 + 2^-19 var (the 16-term fma chains and the merge, 32 roundings); rstd: e_r = e_var / (2 (var + 1e-5 -
    e_var)) + 2^-21 (rsqrtf 2 ulp, the + 1e-5);  e_y = |g| rstd (e1 + e_mu) + |g| |v - mu| rstd (e_r + 2^-23) + ulp(y).
    ReLU: Lipschitz 1.  A common offset C of v enters only through ulp(v) and the sums' rounding: linear in C.
  * GRU: gate arguments e = |W| e_x + kappa 2^-20 (|W_ih||x| + |W_hh||h|) + 2^-23 (|acc| + |b|) (the biases stored
    pre-scaled by log2 e, one fma in the exponential's unit).  sigmoid8 / tanh8_scaled: ex2.approx (2 ulp), the + 1,
    rcp4's four roundings (<= 2.4e-7 relative, policy.cu rcp4): c_sig = c_tanh = 6e-7 absolute.  r, z: 1/4 e + c_sig;
    n: argument e_n = e_gin + r e_ghn + |gh_n + b_hn| e_r + 2^-22 (|gi_n| + |b_in| + r (|gh_n| + |b_hn|)), then
    (1 - n^2 + e) e + c_tanh.  h' = n + z (h - n): |h - n| e_z + (1 - z + e_z) e_n + u |h - n| + ulp(h').
  * fc2 (fp32 fma chains of 16, four partial sums, + bias): e_m = |W2| e_h + 2^-18 (|W2||h| + |b2|).
  * action a = tanh_fast(x) (__expf, __fdividef: absolute error < 8 2^-23 on [0, 15]): e_a = min(1, 1 - a^2 + 2 e_x) e_x
    + 8 2^-23, x = m (test mode) or fma(std, z, m) (e_x = e_m + std e_z + ulp(x)).
  * log-probability: -(x - m)^2 / (2 std^2) - log std - log sqrt(2 pi) - log(1 - a^2 + 1e-6).  The Gaussian term from
    d = x - m in fp32: (|z| / std)(ulp(x) + ulp(d) + std e_z) + 4 u z^2 / 2.  The tanh correction, conditioned on the row's
    own a: w = 1 - a^2 + 1e-6 moves by dw = 2 |a| e_a + e_a^2 + 3 2^-25 (a^2, 1 - a^2, + 1e-6 in fp32), so the log by
    dw / max(w - dw, 0.99e-6) (the kernel's a <= 1: w >= 1e-6), plus __logf (2^-21.41 absolute on [0.5, 2], else 3 ulp).
    Near |a| = 1 one ulp of a moves logp by ~0.1: a flat tolerance cannot hold on millions of draws.  The formula alone is
    checked separately: logp against the fp64 formula at the kernel's own fp32 a and x (caller eps, std = 1).
  * Philox + Box-Muller: z_ref in fp64 from the exact uniforms of the numpy port.  ra = sqrt(-2 __logf(u0)): e_L =
    2^-21.41 (u0 in [0.5, 1]) or 3 ulp(L) and e_ra = 2 e_L / (sqrt(2 |L| + 2 e_L) + sqrt(2 |L|)) + u ra; the angle
    fp32(2 pi) u1 (up to 2 pi: __sincosf outside [-pi, pi], whose sin.approx / cos.approx absolute error is 2^-20.5 over
    +-100 pi) + 2 u 2 pi; e_z = e_ra + ra e_trig + ulp(z).
Worst.report prints max(err / bound) per quantity."""
import contextlib

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


def ring_from_windows(obs, slot):
    """The inverse of windows(): windows [n, na, 144] (oldest entry first; numpy or torch) -> the env-minor ring
    [24, na, 6, n_pad] on obs's device with its newest entry in `slot`, zeros past env n."""
    obs = torch.as_tensor(obs)
    n, na = obs.shape[0], obs.shape[1]
    n_pad = (n + 31) // 32 * 32
    w = obs.reshape(n, na, 24, 6)
    ring = torch.zeros(24, na, 6, n_pad, device=obs.device)
    for r in range(24):
        ring[(slot + 1 + r) % 24, :, :, :n] = w[:, :, r, :].permute(1, 2, 0)
    return ring


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


# ------------------------------------------------------------------------------------------------ drivers
@contextlib.contextmanager
def hbm_traffic():
    """1 GB of HBM traffic on a side stream racing what the block launches; synchronises the device on exit."""
    side = torch.cuda.Stream()
    junk = torch.empty(1 << 28, device=torch.cuda.current_device())
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(4):
            junk.mul_(0.5)
    yield
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()


def hidden_input(n, na, n_pad, kind, layout, cuda, seed):
    """act()'s hidden-state input of `kind` none / given / reset (every third env) in `layout` rows / env_minor:
    (hid_in, reset, h_ref), h_ref [n, na, 64] the rows the kernel must start from."""
    g = torch.Generator(device=cuda).manual_seed(seed)
    h = 0.9 * (2 * torch.rand(n, na, 64, device=cuda, generator=g) - 1)
    reset = None
    if kind == "reset":
        reset = torch.zeros(n, dtype=torch.uint8, device=cuda); reset[::3] = 1
    h_ref = torch.zeros_like(h) if kind == "none" else h.clone()
    if reset is not None:
        h_ref[reset.bool()] = 0
    if kind == "none":
        return None, None, h_ref
    if layout == "rows":
        return h, reset, h_ref
    em = torch.zeros(na, 64, n_pad, device=cuda); em[:, :, :n] = h.permute(1, 2, 0)
    return em, reset, h_ref


def run_policy(pol, ring, slot, n, hid_in, reset, layout, mode, eps, step):
    """act() in `mode` eps / philox / test, under side-stream HBM traffic, into sentinel-filled outputs with a guard band
    past row n (and, env-minor, past column n and agent na): (action, logp, hid rows, mean)."""
    na, n_pad, dev = pol.n_agents, ring.shape[-1], ring.device
    full = {k: torch.full((n + 64, na, 4), SENT, device=dev) for k in ("action", "logp", "mean")}
    for k in ("action", "logp"):
        pol._bufs[k] = full[k][:n]
    if layout == "rows":
        hfull = torch.full((n + 8, na, 64), SENT, device=dev); hid_out = hfull[:n]
    else:
        hfull = torch.full((na + 1, 64, n_pad), SENT, device=dev); hid_out = hfull[:na]
    with hbm_traffic():
        pol.act(ring, slot=slot, n_envs=n, hid_in=hid_in, reset=reset, explore=mode != "test",
                eps=eps if mode == "eps" else None, step=step, hid_out=hid_out, hid_layout=layout, want_mean=True,
                mean_out=full["mean"][:n])
    for k in ("action", "logp", "mean"):
        assert bool((full[k][n:] == SENT).all()), ("written past row n", k)
    if layout == "rows":
        assert bool((hfull[n:] == SENT).all()), "hidden rows written past n"
        h_rows = hid_out
    else:
        assert bool((hfull[na:] == SENT).all()) and bool((hfull[:na, :, n:] == SENT).all()), "env-minor hidden written past n / na"
        h_rows = hfull[:na, :, :n].permute(2, 0, 1)
    return full["action"][:n].clone(), full["logp"][:n].clone(), h_rows.clone(), full["mean"][:n].clone()


def check_policy(wst, pol, M, ring, slot, n, h_ref, eps, step, outs, *, rms):
    """run_policy's outputs `outs` by mode, every row in chunks against policy_reference: mean and hid (the same in every
    mode), then action and log-probability with the caller's eps, with the Philox port's draws and in test mode."""
    na, dev = pol.n_agents, ring.device
    for mode in ("philox", "test"):                                          # the network's outputs do not depend on the draw
        assert torch.equal(outs[mode][3], outs["eps"][3]) and torch.equal(outs[mode][2], outs["eps"][2])
    for e0 in range(0, n, CHUNK):
        e1 = min(n, e0 + CHUNK)
        m, e_m, h1, e_h = policy_reference(M, windows(ring, slot, e0, e1), h_ref[e0:e1].double())
        wst.check("mean", outs["eps"][3][e0:e1], m, e_m, rms=rms)
        wst.check("hid", outs["eps"][2][e0:e1], h1, e_h, rms=rms)
        rows = (np.arange(e0, e1, dtype=np.uint64)[:, None] * np.uint64(na) + np.arange(na, dtype=np.uint64)[None]).reshape(-1)
        zp, ezp = philox_normals(rows, pol.seed, step)
        z_ph = torch.from_numpy(zp).to(dev).view(e1 - e0, na, 4); e_ph = torch.from_numpy(ezp).to(dev).view(e1 - e0, na, 4)
        z_eps = eps[e0:e1].double()
        for mode, z, ez in (("eps", z_eps, torch.zeros_like(z_eps)), ("philox", z_ph, e_ph), ("test", None, None)):
            act, logp = outs[mode][0][e0:e1], outs[mode][1][e0:e1]
            a, e_a, x, e_x = action_bound(m, e_m, z, ez, pol.std, mode != "test")
            wst.check("action", act, a, e_a, f"[{mode}]")
            if mode == "test":
                assert bool((logp == 0).all())
                continue
            lp, e_lp = logp_bound(a, e_a, z, ez, x, pol.std)
            wst.check("logp", logp, lp, e_lp, f"[{mode}]")


def critic_rows(wst, pol, M, ring, slot, n, act, key="", *, rms):
    """value() of the first n envs under side-stream HBM traffic into a sentinel-filled output (the rows past n_envs keep
    their sentinels), every row in chunks against critic_reference."""
    na = ring.shape[1]
    out_full = torch.full((ring.shape[-1] + 16, na, 1), SENT, device=ring.device)
    with hbm_traffic():
        pol.value(ring, act[:n], slot=slot, n_envs=n, out=out_full[:n])
    assert bool((out_full[n:] == SENT).all()), "value written past n_envs"
    for e0 in range(0, n, CHUNK):
        e1 = min(n, e0 + CHUNK)
        val, e_val = critic_reference(M, windows(ring, slot, e0, e1).reshape(e1 - e0, na * 144), act[e0:e1].reshape(e1 - e0, na * 4))
        wst.check("value", out_full[e0:e1, :, 0], val, e_val, key, rms=rms)
