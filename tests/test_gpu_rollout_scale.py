"""The device rollout's kernels at rollout scale, every row: k_policy, k_sample and k_critic against a float64 reference
with a per-element error bound, the Philox exploration draws against a numpy port, the Transition writers bit for bit,
and the LayerNorm's invariance to a common offset of its input.

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
    (m / 4) 2^-20.  fc1: m = 2 x 18 (policy, K = 144: kappa = 19), 2 x (90 + 3) (critic, 720 observation + 24 action
    columns: kappa = 47.5); GRU: m = 32 for r | z (x and h sides in one accumulator: kappa = 9), 16 for gi_n and gh_n
    (kappa = 5); critic fc2: m = 16 (kappa = 5).  A bias is added in fp32 after the MMA: + ulp(v).
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
Each test prints max(err / bound) per quantity and size."""
import numpy as np
import pytest
import torch
from _golden import load_ref_policy

pytestmark = pytest.mark.gpu
KEYS = ("fc1.weight", "fc1.bias", "layernorm.weight", "layernorm.bias", "rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih",
        "rnn.bias_hh", "fc2.weight", "fc2.bias")
CKEYS = ("fc1.weight", "fc1.bias", "layernorm.weight", "layernorm.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias")
CHUNK = 65536
U = 2.0 ** -24
KAPPA_FC1, KAPPA_RZ, KAPPA_N, KAPPA_CFC1, KAPPA_CFC2 = 19.0, 9.0, 5.0, 47.5, 5.0
C_SIG = C_TANH = 6e-7
C_TANH_FAST = 8 * 2.0 ** -23
SENT = 7.25e6                                       # sentinel: no output of these kernels comes near it
BIG = 131072


def ulp(x):
    """fp32 spacing of |x| (x float64): 2^(exponent - 23), at least the smallest normal's."""
    m, e = torch.frexp(x.abs().float().double())
    return torch.where(m == 0, torch.full_like(x, 2.0 ** -149), torch.ldexp(torch.ones_like(x), (e - 24).clamp(min=-149)))


def tf32(w):
    from flexgpu.policy import round_tf32
    return round_tf32(np.asarray(w, dtype=np.float32)).astype(np.float64)


def f32(x):
    return np.asarray(x, dtype=np.float32).astype(np.float64)


# ------------------------------------------------------------------------------------------------ inputs and weights
def realistic_policy(seed):
    """An RNNAgent with torch's default initialisation spread and a trained-looking LayerNorm."""
    rng = np.random.default_rng(seed)
    k1, kg = 1 / np.sqrt(149), 1 / 8
    sd = {"fc1.weight": rng.uniform(-k1, k1, (64, 149)), "fc1.bias": rng.uniform(-k1, k1, 64),
          "layernorm.weight": 1 + rng.normal(0, 0.2, 64), "layernorm.bias": rng.normal(0, 0.2, 64),
          "rnn.weight_ih": rng.uniform(-kg, kg, (192, 64)), "rnn.weight_hh": rng.uniform(-kg, kg, (192, 64)),
          "rnn.bias_ih": rng.uniform(-kg, kg, 192), "rnn.bias_hh": rng.uniform(-kg, kg, 192),
          "fc2.weight": rng.uniform(-kg, kg, (4, 64)), "fc2.bias": rng.uniform(-kg, kg, 4)}
    return {k: v.astype(np.float32) for k, v in sd.items()}


def realistic_critic(seed):
    rng = np.random.default_rng(seed)
    k1, k2 = 1 / np.sqrt(745), 1 / 8
    sd = {"fc1.weight": rng.uniform(-k1, k1, (64, 745)), "fc1.bias": rng.uniform(-k1, k1, 64),
          "layernorm.weight": 1 + rng.normal(0, 0.2, 64), "layernorm.bias": rng.normal(0, 0.2, 64),
          "fc2.weight": rng.uniform(-k2, k2, (64, 64)), "fc2.bias": rng.uniform(-k2, k2, 64),
          "fc3.weight": rng.uniform(-k2, k2, (1, 64)), "fc3.bias": rng.uniform(-k2, k2, 1)}
    return {k: v.astype(np.float32) for k, v in sd.items()}


def make_ring(n, slot_seed, cuda, obs_src):
    """[24, 5, 6, n_pad] ring from the golden observation windows: env e carries window e % n_src times (1 + 0.05 N(0, 1)),
    so rows differ; columns past n are zeros, as the env leaves them."""
    n_pad = (n + 31) // 32 * 32
    src = torch.from_numpy(np.ascontiguousarray(obs_src, dtype=np.float32)).to(cuda)           # [n_src, 5, 144]
    g = torch.Generator(device=cuda).manual_seed(slot_seed)
    ring = torch.zeros(24, 5, 6, n_pad, device=cuda)
    for e0 in range(0, n, CHUNK):
        e1 = min(n, e0 + CHUNK)
        idx = torch.arange(e0, e1, device=cuda) % src.shape[0]
        w = src[idx] * (1 + 0.05 * torch.randn(e1 - e0, 5, 144, device=cuda, generator=g))
        ring[:, :, :, e0:e1] = w.view(e1 - e0, 5, 24, 6).permute(2, 1, 3, 0)      # slot order = window order; rotated below
    return ring


def windows(ring, slot, e0, e1):
    """Dense windows [c, 5, 144] (oldest entry first) of envs [e0, e1) by plain indexing of the ring."""
    idx = torch.tensor([(slot + 1 + r) % 24 for r in range(24)], device=ring.device)
    return ring[:, :, :, e0:e1][idx].permute(3, 1, 0, 2).reshape(e1 - e0, 5, 144)


def rotate(ring, slot):
    """A ring whose window order is its slot order, re-laid so that its newest entry sits in `slot`."""
    idx = torch.tensor([(r - slot - 1) % 24 for r in range(24)], device=ring.device)
    return ring[idx].contiguous()


# ------------------------------------------------------------------------------------------------ fp64 policy reference
def policy_mats(sd, dev):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
    w1 = np.asarray(sd["fc1.weight"], dtype=np.float32)
    b1a = np.stack([f32(np.float32(sd["fc1.bias"]) + w1[:, 144 + a]) for a in range(5)])          # one fp32 addition
    return {"W1": t(tf32(w1[:, :144])), "b1a": t(b1a), "g": t(f32(sd["layernorm.weight"])), "b": t(f32(sd["layernorm.bias"])),
            "Wih": t(tf32(sd["rnn.weight_ih"])), "Whh": t(tf32(sd["rnn.weight_hh"])), "bih": t(f32(sd["rnn.bias_ih"])),
            "bhh": t(f32(sd["rnn.bias_hh"])), "W2": t(f32(sd["fc2.weight"])), "b2": t(f32(sd["fc2.bias"]))}


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


def policy_reference(M, obs, h):
    """fp64 RNNAgent forward of obs [c, 5, 144] (fp32 values) and h [c, 5, 64]: mean, h', and their bounds."""
    x = obs.double()
    v = x @ M["W1"].T + M["b1a"][None]                                                 # [c, 5, 64]
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


# ------------------------------------------------------------------------------------------------ Philox4x32-10 in numpy
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


def test_philox_port_matches_the_reset_draws(fonet):
    """The numpy port against oracle.c_mirror.draw_random, whose philox4x32_10 draws are bit-matched to the GPU's resets:
    seeds and env ids past 2^32 included (all four counter words and both key words are live)."""
    from oracle import c_mirror
    for seed in (0, 1234, (7 << 32) + 5, 2 ** 64 - 1):
        for gid in (0, 3, 1000, (1 << 32) + 17):
            for episode in (0, 9):
                _, _, a0 = c_mirror.draw_random(fonet, seed, gid, episode, 1000)
                b = np.arange(10, dtype=np.uint32)
                c = philox(np.full(10, gid & 0xFFFFFFFF, np.uint32), np.full(10, gid >> 32, np.uint32),
                           np.full(10, episode, np.uint32), b, seed & 0xFFFFFFFF, seed >> 32)
                v0, v1 = u53(c[0], c[1]), u53(c[2], c[3])
                want = np.empty((5, 4)); want[:, 0] = v0[0::2]; want[:, 1] = v1[0::2]; want[:, 2] = v0[1::2]; want[:, 3] = v1[1::2]
                assert np.array_equal(a0.reshape(5, 4), want), (seed, gid, episode)


# ------------------------------------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def gold():
    return load_ref_policy()


@pytest.fixture(scope="module")
def policies(gold, cuda):
    from flexgpu.policy import DevicePolicy
    sds = {"real": realistic_policy(21), "gold": {k: np.asarray(gold["wt_" + k], dtype=np.float32) for k in KEYS}}
    pols = {k: (DevicePolicy(sd, device=cuda, std=1.0, seed=(5 << 32) + 77), policy_mats(sd, cuda)) for k, sd in sds.items()}
    yield pols
    for p, _ in pols.values():
        p.close()


def sentinel_views(pol, n):
    """Output buffers of the handle replaced by the first n rows of sentinel-filled tensors 64 rows longer."""
    dev = pol.device
    full = {k: torch.full((n + 64, 5, 4), SENT, device=dev) for k in ("action", "logp", "mean")}
    for k in ("action", "logp"):
        pol._bufs[k] = full[k][:n]
    return full


def hidden_input(n, n_pad, kind, layout, cuda, seed):
    g = torch.Generator(device=cuda).manual_seed(seed)
    h = 0.9 * (2 * torch.rand(n, 5, 64, device=cuda, generator=g, dtype=torch.float32) - 1)
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
    em = torch.zeros(5, 64, n_pad, device=cuda); em[:, :, :n] = h.permute(1, 2, 0)
    return em, reset, h_ref


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


# ------------------------------------------------------------------------------------------------ k_policy, every row
# per size, configurations that together cover both hidden layouts, the three hidden inputs, slots 0 / 11 / 23 and both
# weight sets; each runs explore with caller eps, explore with Philox and test mode
CONFIGS = [("rows", "none", 0, "real"), ("env_minor", "given", 11, "gold"), ("rows", "reset", 23, "gold"),
           ("env_minor", "reset", 0, "real"), ("rows", "given", 11, "real")]
SIZES = [129, 3840, BIG, BIG + 77, 1 << 20]


def run_policy(pol, ring, slot, n, hid_in, reset, layout, mode, eps, step, n_pad):
    full = sentinel_views(pol, n)
    if layout == "rows":
        hfull = torch.full((n + 8, 5, 64), SENT, device=ring.device)
        hid_out = hfull[:n]
    else:
        hfull = torch.full((5, 64, n_pad), SENT, device=ring.device)
        hid_out = hfull
    side = torch.cuda.Stream()
    junk = torch.empty(1 << 28, device=ring.device)                   # 1 GB of HBM traffic racing the kernel
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(4):
            junk.mul_(0.5)
    act, logp, hid, mean = pol.act(ring, slot=slot, n_envs=n, hid_in=hid_in, reset=reset, explore=mode != "test",
                                   eps=eps if mode == "eps" else None, step=step, hid_out=hid_out, hid_layout=layout,
                                   want_mean=True, mean_out=full["mean"][:n])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for k in ("action", "logp", "mean"):
        assert bool((full[k][n:] == SENT).all()), ("written past row n", k)
    if layout == "rows":
        assert bool((hfull[n:] == SENT).all()), "hidden rows written past n"
        h_rows = hid_out
    else:
        assert bool((hfull[:, :, n:] == SENT).all()), "env-minor hidden columns [n, n_pad) written"
        h_rows = hfull[:, :, :n].permute(2, 0, 1)
    return full["action"][:n].clone(), full["logp"][:n].clone(), h_rows.clone(), full["mean"][:n].clone()


@pytest.mark.parametrize("n", SIZES)
def test_policy_every_row_against_fp64(policies, gold, cuda, n):
    step = (1 << 40) + 3
    n_pad = (n + 31) // 32 * 32
    base = make_ring(n, n, cuda, gold["obs0"])
    wst = Worst(f"k_policy n={n}")
    configs = CONFIGS if n < (1 << 20) else CONFIGS[:3]
    for ci, (layout, hkind, slot, wname) in enumerate(configs):
        pol, M = policies[wname]
        ring = rotate(base, slot)
        hid_in, reset, h_ref = hidden_input(n, n_pad, hkind, layout, cuda, ci + n)
        eps = torch.randn(n, 5, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(ci))
        outs = {mode: run_policy(pol, ring, slot, n, hid_in, reset, layout, mode, eps, step, n_pad) for mode in ("eps", "philox", "test")}
        for mode in ("philox", "test"):                                      # the network's outputs do not depend on the draw
            assert torch.equal(outs[mode][3], outs["eps"][3]) and torch.equal(outs[mode][2], outs["eps"][2])
        for e0 in range(0, n, CHUNK):
            e1 = min(n, e0 + CHUNK)
            m, e_m, h1, e_h = policy_reference(M, windows(ring, slot, e0, e1), h_ref[e0:e1].double())
            wst.check("mean", outs["eps"][3][e0:e1], m, e_m, rms=True)
            wst.check("hid", outs["eps"][2][e0:e1], h1, e_h, rms=True)
            z_eps = eps[e0:e1].double()
            rows = (np.arange(e0, e1, dtype=np.uint64)[:, None] * np.uint64(5) + np.arange(5, dtype=np.uint64)[None]).reshape(-1)
            zp, ezp = philox_normals(rows, pol.seed, step)
            z_ph = torch.from_numpy(zp).to(cuda).view(e1 - e0, 5, 4); e_ph = torch.from_numpy(ezp).to(cuda).view(e1 - e0, 5, 4)
            for mode, z, ez in (("eps", z_eps, torch.zeros_like(z_eps)), ("philox", z_ph, e_ph), ("test", None, None)):
                act, logp = outs[mode][0][e0:e1], outs[mode][1][e0:e1]
                a, e_a, x, e_x = action_bound(m, e_m, z, ez, pol.std, mode != "test")
                wst.check("action", act, a, e_a, f"[{mode}]")
                if mode == "test":
                    assert bool((logp == 0).all())
                    continue
                lp, e_lp = logp_bound(a, e_a, z, ez, x, pol.std)
                wst.check("logp", logp, lp, e_lp, f"[{mode}]")
            if e0 == 0:                                    # the formula alone, at the kernel's own fp32 a and x (caller eps)
                mk = outs["eps"][3][e0:e1].double()
                xk = (mk + z_eps).float().double()                   # fma(1, z, m): exact sum, one rounding
                ak = outs["eps"][0][e0:e1].double()
                wk = 1 - ak * ak + 1e-6
                dw = 2.0 ** -23                                       # a^2, 1 - a^2, + 1e-6 in fp32
                gauss = 0.5 * (xk - mk) ** 2
                lp_self = -gauss - 0.5 * np.log(2 * np.pi) - torch.log(wk)
                logf = torch.where(wk >= 0.5, torch.full_like(wk, 2.0 ** -21.41), 3 * ulp(torch.log(wk)))
                bound = dw / (wk - dw).clamp(min=0.99e-6) + logf + (xk - mk).abs() * ulp(xk - mk) + 4 * U * (xk - mk) ** 2 + \
                    ulp(lp_self) + ulp(gauss + 0.92) + 2 * U
                wst.check("logp_formula", outs["eps"][1][e0:e1], lp_self, bound)
    wst.report()


# ------------------------------------------------------------------------------------------------ Philox and k_sample
def test_sample_philox_against_port_and_bit_identical_to_act(policies, gold, cuda):
    """k_sample's Philox draws at 131 072 envs against the numpy port (seed >= 2^32; step 2^40 + t differs from step t: the
    counter's high step word is live), the 5.77-sigma truncation of the design, and fp_policy_sample on act's mean equal to
    act's action and logp bit for bit, with Philox and with eps, explore and test."""
    pol, M = policies["real"]
    n = BIG
    ring = rotate(make_ring(n, 3, cuda, gold["obs0"]), 5)
    eps = torch.randn(n, 5, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(4))
    wst = Worst("k_sample n=131072")
    rows = np.arange(n * 5, dtype=np.uint64)
    for t in (0, 6):
        step = (1 << 40) + t
        for explore, e in ((True, None), (True, eps), (False, None)):
            a1, lp1, _, m1 = pol.act(ring, slot=5, n_envs=n, explore=explore, eps=e, step=step, want_mean=True,
                                     hid_out=torch.empty(n, 5, 64, device=cuda))
            a1, lp1, m1 = a1.clone(), lp1.clone(), m1.clone()
            a2, lp2 = pol.sample(m1, explore=explore, eps=e, step=step)
            assert torch.equal(a1, a2) and torch.equal(lp1, lp2), (t, explore, e is None)
        m = m1.double()
        a_s, lp_s = [v.clone() for v in pol.sample(m1, explore=True, step=step)]
        zp, ezp = philox_normals(rows, pol.seed, step)
        z = torch.from_numpy(zp).to(cuda).view(n, 5, 4); ez = torch.from_numpy(ezp).to(cuda).view(n, 5, 4)
        a, e_a, x, _ = action_bound(m, torch.zeros_like(m), z, ez, pol.std, True)
        wst.check("action", a_s, a, e_a)
        lp, e_lp = logp_bound(a, e_a, z, ez, x, pol.std)
        wst.check("logp", lp_s, lp, e_lp)
        # the low-step draws are different numbers: dropping the counter's high word would make them equal
        z_low, _ = philox_normals(rows, pol.seed, t)
        assert np.mean(z_low == zp) < 1e-6
        a_low, _ = pol.sample(m1, explore=True, step=t)
        assert float((a_low != a_s).float().mean()) > 0.99
        # u0 in (0, 1]: |z| <= sqrt(-2 ln 2^-24) = 5.768 by construction (a 5.77-sigma truncation of the normals)
        zmax = np.sqrt(-2 * np.log(2.0 ** -24))
        assert np.abs(zp).max() <= zmax and np.abs(zp).max() > 4.5
        # from the kernel's own action: |x - m| = |atanh(a) - m| never exceeds the truncation (where a is not saturated)
        ok = a_s.abs() < 0.999
        zk = (torch.atanh(a_s.double()) - m)[ok]
        assert float(zk.abs().max()) <= zmax + 1e-3
    wst.report()


# ------------------------------------------------------------------------------------------------ k_critic, every row
def critic_mats(sd, dev):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
    w1 = np.asarray(sd["fc1.weight"], dtype=np.float32)
    b1a = np.stack([f32(np.float32(sd["fc1.bias"]) + w1[:, 720 + a]) for a in range(5)])
    return {"Wo": t(tf32(w1[:, :720])), "Wa": t(tf32(w1[:, 725:])), "b1a": t(b1a), "g": t(f32(sd["layernorm.weight"])),
            "b": t(f32(sd["layernorm.bias"])), "W2": t(tf32(sd["fc2.weight"])), "b2": t(f32(sd["fc2.bias"])),
            "w3": t(f32(sd["fc3.weight"])[0]), "b3": float(np.float32(sd["fc3.bias"][0]))}


def critic_reference(M, obs_all, act):
    """fp64 critic of obs_all [c, 720], act [c, 20]: value [c, 5] and its bound; also the LayerNorm input and output."""
    x, ac = obs_all.double(), act.double()
    acc = x @ M["Wo"].T + ac @ M["Wa"].T                                            # [c, 64]
    e_acc = KAPPA_CFC1 * 2.0 ** -20 * (x.abs() @ M["Wo"].abs().T + ac.abs() @ M["Wa"].abs().T)
    v = acc[:, None, :] + M["b1a"][None]                                          # [c, 5, 64]
    e1 = e_acc[:, None, :] + ulp(v)
    y, e_y = layernorm_bound(v, e1, M["g"], M["b"])
    q0 = torch.relu(y)
    u = q0 @ M["W2"].T + M["b2"]
    e_u = e_y @ M["W2"].abs().T + KAPPA_CFC2 * 2.0 ** -20 * (q0 @ M["W2"].abs().T) + ulp(u)
    q = torch.relu(u)
    val = q @ M["w3"] + M["b3"]
    e_val = e_u @ M["w3"].abs() + 2.0 ** -18 * (q @ M["w3"].abs() + abs(M["b3"]))
    return val, e_val


@pytest.fixture(scope="module")
def critic(cuda):
    from flexgpu.policy import DevicePolicy
    sd = realistic_critic(5)
    pol = DevicePolicy(None, device=cuda)
    pol.load_critic(sd)
    yield pol, critic_mats(sd, cuda)
    pol.close()


def critic_rows(pol, M, ring, slot, n, act, wst, key=""):
    out_full = torch.full((ring.shape[-1] + 16, 5, 1), SENT, device=ring.device)
    side = torch.cuda.Stream()
    junk = torch.empty(1 << 28, device=ring.device)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(4):
            junk.mul_(0.5)
    pol.value(ring, act[:n], slot=slot, n_envs=n, out=out_full[:n])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    assert bool((out_full[n:] == SENT).all()), "value written past n_envs"
    for e0 in range(0, n, CHUNK):
        e1 = min(n, e0 + CHUNK)
        val, e_val = critic_reference(M, windows(ring, slot, e0, e1).reshape(e1 - e0, 720), act[e0:e1].reshape(e1 - e0, 20))
        wst.check("value", out_full[e0:e1, :, 0], val, e_val, key, rms=True)


@pytest.mark.parametrize("n", [BIG, BIG + 77, 1 << 20])
def test_critic_every_row_against_fp64(critic, gold, cuda, n):
    pol, M = critic
    base = make_ring(n, 7 + n, cuda, gold["obs1"])
    act = torch.tanh(torch.randn(n, 5, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(n)))
    wst = Worst(f"k_critic n={n}")
    for slot in (0, 11, 23):
        critic_rows(pol, M, rotate(base, slot), slot, n, act, wst, f"[slot {slot}]")
    if n == BIG:                                        # DeviceRollout's native-value call: record_envs < n_pad, TMA path
        critic_rows(pol, M, rotate(base, 11), 11, 40000, act, wst, "[n_envs 40000]")
    wst.report()


# ------------------------------------------------------------------------------------------------ LayerNorm offset invariance
OFFSETS = (0.0, 1.0, 4.0, 16.0, 64.0)


def probe_policy(gold, C):
    """The golden fc1 / LayerNorm with fc1.bias + C, under a GRU that exposes the LayerNorm: W_ih's n block = I, every other
    gate weight 0, the z bias -40 (z = sigmoid(-20) after the kernel's clamp, 2e-9), so h' = tanh(relu(LN(v))) per unit."""
    sd = {k: np.asarray(gold["wt_" + k], dtype=np.float32).copy() for k in KEYS}
    sd["fc1.bias"] = (sd["fc1.bias"] + np.float32(C)).astype(np.float32)
    sd["rnn.weight_ih"] = np.zeros((192, 64), np.float32); sd["rnn.weight_ih"][128:] = np.eye(64, dtype=np.float32)
    sd["rnn.weight_hh"] = np.zeros((192, 64), np.float32)
    sd["rnn.bias_ih"] = np.zeros(192, np.float32); sd["rnn.bias_ih"][64:128] = -40.0
    sd["rnn.bias_hh"] = np.zeros(192, np.float32)
    return sd


def test_layernorm_offset_invariance_policy(gold, cuda):
    """fc1.bias + C leaves the network unchanged.  (a) mean and hid of the golden network against the C = 0 fp64 reference,
    inside the error model evaluated at the shifted pre-activation (the offset enters through ulp(v) and the sums' rounding:
    linear in C).  (b) The sharp check: the fc1 accumulator is bit-identical for every C (the bias is added after the MMA),
    so on the probe network the difference of the C and C = 0 runs is the LayerNorm's alone: per unit at most the sum of
    both runs' LayerNorm bounds with exact inputs (e1 = ulp(v)), times tanh', plus both runs' rounding after it."""
    from flexgpu.policy import DevicePolicy
    n = BIG
    slot = 11
    ring = rotate(make_ring(n, 19, cuda, gold["obs0"]), slot)
    h_in = 0.9 * (2 * torch.rand(n, 5, 64, device=cuda, generator=torch.Generator(device=cuda).manual_seed(2)) - 1)
    wst = Worst("LayerNorm offset, k_policy n=131072")
    ref0 = policy_mats({k: np.asarray(gold["wt_" + k], dtype=np.float32) for k in KEYS}, cuda)
    probe = {}
    for C in OFFSETS:
        sd = {k: np.asarray(gold["wt_" + k], dtype=np.float32).copy() for k in KEYS}
        sd["fc1.bias"] = (sd["fc1.bias"] + np.float32(C)).astype(np.float32)
        pol = DevicePolicy(sd, device=cuda)
        _, _, hid, mean = pol.act(ring, slot=slot, n_envs=n, hid_in=h_in, explore=False, want_mean=True, hid_out=torch.empty(n, 5, 64, device=cuda))
        MC = policy_mats(sd, cuda)
        for e0 in range(0, n, CHUNK):
            e1 = min(n, e0 + CHUNK)
            obs = windows(ring, slot, e0, e1)
            m0, _, h0, _ = policy_reference(ref0, obs, h_in[e0:e1].double())
            mc, e_m, hc, e_h = policy_reference(MC, obs, h_in[e0:e1].double())          # the model at the shifted v
            # + what the fp32 folding of fc1.bias + C + one-hot column changes exactly (the pre-activation's representation)
            wst.check("mean", mean[e0:e1], m0, e_m + (mc - m0).abs(), f"[C={C:g}]")
            wst.check("hid", hid[e0:e1], h0, e_h + (hc - h0).abs(), f"[C={C:g}]")
        pol.load_state_dict(probe_policy(gold, C))
        _, _, hp, _ = pol.act(ring, slot=slot, n_envs=n, hid_in=None, explore=False, hid_out=torch.empty(n, 5, 64, device=cuda))
        probe[C] = (hp.clone(), MC["b1a"])
        pol.close()

    def probe_ref(acc, b1a, e_acc=0.0):               # tanh(relu(LN(acc + b1a))) with input error e_acc + ulp(v), and its bound
        v = acc + b1a[None]
        y, e_y = layernorm_bound(v, e_acc + ulp(v), ref0["g"], ref0["b"])
        n_ = torch.tanh(torch.relu(y))
        return n_, (1 - n_ * n_ + e_y).clamp(max=1) * (e_y + 2.0 ** -20 * y.abs()) + C_TANH + 2.0 ** -22 * y.abs() + 3e-9 + ulp(n_)
    for C in OFFSETS[1:]:
        for e0 in range(0, n, CHUNK):
            e1 = min(n, e0 + CHUNK)
            x = windows(ring, slot, e0, e1).double()
            acc = x @ ref0["W1"].T
            (r0, b0), (rc, bc) = probe_ref(acc, probe[0.0][1]), probe_ref(acc, probe[C][1])
            wst.check("probe_hid_diff", probe[C][0][e0:e1].double() - probe[0.0][0][e0:e1].double(), rc - r0, b0 + bc, f"[C={C:g}]")
            if C == OFFSETS[1]:                         # the probe itself against fp64, fc1's error included
                r0f, b0f = probe_ref(acc, probe[0.0][1], KAPPA_FC1 * 2.0 ** -20 * (x.abs() @ ref0["W1"].abs().T))
                wst.check("probe_hid", probe[0.0][0][e0:e1], r0f, b0f, "[C=0]")
    wst.report()


def test_layernorm_offset_invariance_critic(gold, cuda):
    """As for the policy: the critic's fc1.bias + C against the C = 0 fp64 reference within the model, and on a probe
    critic (fc2 = I, fc2.bias = 0, fc3 = unit j) whose value is relu(LN(v))_j, the C run against the C = 0 run."""
    from flexgpu.policy import DevicePolicy
    n = BIG
    slot = 23
    ring = rotate(make_ring(n, 23, cuda, gold["obs1"]), slot)
    act = torch.tanh(torch.randn(n, 5, 4, device=cuda, generator=torch.Generator(device=cuda).manual_seed(8)))
    sd0 = realistic_critic(9)
    M0 = critic_mats(sd0, cuda)
    j = int(np.argmax(np.abs(sd0["layernorm.weight"])))
    wst = Worst("LayerNorm offset, k_critic n=131072")
    probe = {}
    pol = DevicePolicy(None, device=cuda)
    for C in OFFSETS:
        sd = {k: v.copy() for k, v in sd0.items()}
        sd["fc1.bias"] = (sd["fc1.bias"] + np.float32(C)).astype(np.float32)
        pol.load_critic(sd)
        val = pol.value(ring, act, slot=slot, n_envs=n).clone()
        MC = critic_mats(sd, cuda)
        for e0 in range(0, n, CHUNK):
            e1 = min(n, e0 + CHUNK)
            obs, ac = windows(ring, slot, e0, e1).reshape(e1 - e0, 720), act[e0:e1].reshape(e1 - e0, 20)
            v0, _ = critic_reference(M0, obs, ac)
            vc, e_v = critic_reference(MC, obs, ac)
            wst.check("value", val[e0:e1, :, 0], v0, e_v + (vc - v0).abs(), f"[C={C:g}]")
        sd["fc2.weight"] = np.eye(64, dtype=np.float32); sd["fc2.bias"] = np.zeros(64, np.float32)
        sd["fc3.weight"] = np.zeros((1, 64), np.float32); sd["fc3.weight"][0, j] = 1.0; sd["fc3.bias"] = np.zeros(1, np.float32)
        pol.load_critic(sd)
        probe[C] = (pol.value(ring, act, slot=slot, n_envs=n).clone()[:, :, 0], MC["b1a"])
    pol.close()

    def probe_ref(acc, b1a):                           # relu(LN(acc + b1a))_j with exact input and its bound
        v = acc + b1a[None]
        y, e_y = layernorm_bound(v, ulp(v), M0["g"], M0["b"])
        return torch.relu(y[..., j]), e_y[..., j] + 2.0 ** -20 * y[..., j].abs() + ulp(y[..., j])
    for C in OFFSETS[1:]:
        for e0 in range(0, n, CHUNK):
            e1 = min(n, e0 + CHUNK)
            obs, ac = windows(ring, slot, e0, e1).reshape(e1 - e0, 720).double(), act[e0:e1].reshape(e1 - e0, 20).double()
            acc = (obs @ M0["Wo"].T + ac @ M0["Wa"].T)[:, None, :]
            (r0, b0), (rc, bc) = probe_ref(acc, probe[0.0][1]), probe_ref(acc, probe[C][1])
            wst.check("probe_value_diff", probe[C][0][e0:e1].double() - probe[0.0][0][e0:e1].double(), rc - r0, b0 + bc, f"[C={C:g}]")
    wst.report()


# ------------------------------------------------------------------------------------------------ Transition writers
@pytest.fixture(scope="module")
def big_env(cuda, profiles):
    from flexgpu import BatchedFlexProvisionEnv
    e = BatchedFlexProvisionEnv(None, n_envs=BIG, device=cuda, profiles=profiles, seed=12)
    yield e
    e.close()


def dense_rows(ring, slot, n):
    return torch.cat([windows(ring, slot, e0, min(n, e0 + CHUNK)) for e0 in range(0, n, CHUNK)]).reshape(n, 720)


@pytest.mark.parametrize("record,variant", [(BIG, "plain"), (50000, "plain"), (50000, "native"), (BIG, "failures")])
def test_rollout_transition_writers_at_scale(big_env, gold, cuda, record, variant):
    """DeviceRollout on 131 072 envs: every field of every recorded row against plain torch indexing of the ring before and
    after the step, the hidden states and the step's outputs (bit for bit); the reserved window wraps in the middle of a
    128-env tile, and the replay rows outside it keep their sentinels."""
    from flexgpu.policy import DevicePolicy, DeviceRollout, TRANSITION_FIELDS
    from flexgpu.predictor import DeviceReplayBuffer
    env = big_env
    N = env.n_envs
    pol = DevicePolicy({k: gold["wt_" + k] for k in KEYS}, device=cuda, seed=(3 << 32) + 1)
    if variant == "native":
        pol.load_critic(realistic_critic(13))
    cap = record + 500 if record == N else 60000
    pos0 = cap - ((record // 2) // 128 * 128 + 64)                       # the first step's window wraps 64 envs into a tile
    buf = DeviceReplayBuffer(cap, TRANSITION_FIELDS, device=cuda)
    buf.reserve(cap)
    for k, w in TRANSITION_FIELDS.items():
        buf.write(k, 0, torch.full((cap, w), SENT, device=cuda))
    buf.reserve(pos0)
    head = pos0
    ro = DeviceRollout(env, pol, replay=buf, record_envs=record, reset_done_each_step=variant == "failures",
                       value_fn="native" if variant == "native" else None)
    ro.reset()
    R = ro.R
    captured = {}
    orig_step = env.step

    def spy(*a, **kw):
        out = orig_step(*a, **kw)
        captured["ring"], captured["slot"] = out[3].ring.clone(), out[3].slot
        return out
    env.step = spy
    try:
        for t in range(2):
            if variant == "failures":
                fail = torch.zeros(N, dtype=torch.uint8, device=cuda)
                if t == 0:
                    fail[5::997] = 1
                env.inject_failure(fail)
            pre_ring, pre_slot = ro.ring.ring.clone(), ro.ring.slot
            last_hid = ro._hid[ro._cur][:, :, :N].permute(2, 0, 1).clone()
            reset = None if ro._reset_mask is None else ro._reset_mask.bool().clone()
            reward, done = ro.step()
            torch.cuda.synchronize()
            pos = head
            head = (head + R) % cap
            got = buf.get_batch(cap, start=0)                             # logical order: physical row p = (p - head) mod cap
            phys = {k: torch.roll(v, shifts=head, dims=0) for k, v in got.items()}
            rows = (pos + torch.arange(R, device=cuda)) % cap
            want = {"state": dense_rows(pre_ring, pre_slot, R), "next_state": dense_rows(captured["ring"], captured["slot"], R),
                    "hid": ro._hid[ro._cur][:, :, :R].permute(2, 0, 1).reshape(R, 320),
                    "action": pol._bufs["action"][:R].reshape(R, 20), "log_prob_a": pol._bufs["logp"][:R].reshape(R, 20),
                    "reward": reward[:R, None].float().repeat(1, 5), "done": done[:R, None].float(),
                    "last_step": done[:R, None].float(), "action_avail": torch.ones(R, 20, device=cuda)}
            lh = last_hid[:R].reshape(R, 320).clone()
            if reset is not None:
                lh[reset[:R]] = 0
                assert int(reset[:R].sum()) > 0
            want["last_hid"] = lh
            if variant == "native":
                want["value"] = pol._bufs["value"].view(R, 5); want["next_value"] = pol._bufs["next_value"].view(R, 5)
            else:
                want["value"] = want["next_value"] = torch.zeros(R, 5, device=cuda)
            for k, w in want.items():
                assert torch.equal(phys[k][rows], w), (t, k)
            outside = torch.ones(cap, dtype=torch.bool, device=cuda)
            outside[rows] = False
            if t == 0 and bool(outside.any()):
                for k in TRANSITION_FIELDS:
                    assert bool((phys[k][outside] == SENT).all()), ("row outside the window written", k)
            if variant == "failures":
                if t == 0:
                    assert int(done.sum()) == len(range(5, N, 997))
                else:                                              # the restarted envs acted from a zero hidden state
                    h_zero = pol.act(pre_ring, slot=pre_slot, n_envs=N, hid_in=None, explore=False,
                                     hid_out=torch.empty(N, 5, 64, device=cuda))[2]
                    assert torch.equal(want["hid"][reset[:R]], h_zero[:R][reset[:R]].reshape(-1, 320))
                env.inject_failure(None)
    finally:
        env.step = orig_step
        pol.close(); buf.close()

