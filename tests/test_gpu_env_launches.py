"""Kernel launches of every env verb, on both kernel variants: env.launch_count() advances by a fixed number per call.

One env walks through the verbs in a fixed order, so the state that decides the extra launches is fixed too: whether
the window ring and the env-minor ring exist and are valid (rebuilds, ring restarts after a reset), the variant
(translate_action fused into the thread step kernel, an elementwise pre-pass before the warp one; the one-launch ring
step of the thread variant) and the retry launches of the random reset.  A host-layer change that drops or adds a
launch anywhere on these paths changes a delta.
"""
import numpy as np
import pytest
import torch

from _env_check import make_env, reset_draws

N = 300                  # not a multiple of the 32-env tile

# (verb, launches on the thread variant, launches on the warp variant), in the order they run
EXPECTED = [
    ("reset", 1, 1),
    ("reset masked", 1, 1),
    ("reset random, 0 retries", 1, 1),
    ("reset random, 3 retries", 8, 8),                  # 4 resets + 4 retry-mask builds
    ("step f32", 1, 1),
    ("step f64", 1, 1),
    ("step f32 masked", 1, 1),
    ("step translate", 1, 2),                           # warp: translation pre-pass
    ("preview K=1 f32", 1, 1),
    ("preview K=1 translate", 1, 2),
    ("preview K=3 translate", 1, 2),
    ("preview K=3 f64", 1, 1),
    ("get_obs view, first", 2, 2),                      # window ring built + push
    ("get_obs view", 1, 1),
    ("obs_ring, first", 1, 1),                          # env-minor ring built
    ("reset, rings live", 3, 3),                        # + both rings restarted
    ("reset masked, rings live", 3, 3),
    ("reset random, 0 retries, rings live", 3, 3),
    ("reset random, 3 retries, rings live", 16, 16),
    ("step return_obs=True", 2, 2),                     # step + window push
    ("step return_obs=ring", 2, 3),                     # thread: ring rebuilt + fused step; warp: step + push + rebuild
    ("step return_obs=ring again", 1, 3),
    ("step return_obs=ring masked", 4, 3),              # not fused: thread rebuilds the window ring first
    ("step return_obs=ring translate", 1, 4),
    ("step return_obs=True translate", 3, 3),
    ("get_obs dense", 1, 1),
    ("get_obs dense, no push", 1, 1),
    ("get_obs view after dense", 2, 2),
    ("get_state", 1, 1),
    ("power_flow", 1, 1),
    ("safety_project", 1, 1),
    ("safety_project_affine", 1, 1),
]


@pytest.mark.gpu
def test_launches_per_verb(cuda, profiles, variant):
    env = make_env(cuda, profiles, N, variant, seed=3)
    na, nl, nb = env.n_agents, env.n_lines, env.n_bus
    rng = np.random.default_rng(0)
    start, e0, a0 = reset_draws(rng, N, na, env.max_start())
    mask = torch.from_numpy((np.arange(N) % 3 == 0).astype(np.uint8))

    def acts(*lead, dtype=torch.float32):
        return torch.from_numpy(rng.uniform(-1, 1, (*lead, N, na, 4))).to(dtype=dtype, device=cuda)

    p = env.network.base_p[None, 1:] * rng.uniform(0.7, 1.3, (64, nl))
    q = env.network.base_q[None, 1:] * rng.uniform(0.7, 1.3, (64, nl))
    env.load_safety_model(rng.normal(0, 0.02, (nb, 2 * nb)), np.full(nb, 1.0))
    env.load_safety_map(rng.normal(0, 0.02, (nb, 2 * nb)), np.full(nb, 1.0))
    verbs = {
        "reset": lambda: env.reset(start, e0, a0, return_obs=False),
        "reset masked": lambda: env.reset(start, e0, a0, mask=mask, return_obs=False),
        "reset random, 0 retries": lambda: env.reset(return_obs=False, retries=0),
        "reset random, 3 retries": lambda: env.reset(return_obs=False, retries=3),
        "step f32": lambda: env.step(acts()),
        "step f64": lambda: env.step(acts(dtype=torch.float64)),
        "step f32 masked": lambda: env.step(acts(), mask=mask),
        "step translate": lambda: env.step(acts(), translate=True),
        "preview K=1 f32": lambda: env.preview_step(acts()),
        "preview K=1 translate": lambda: env.preview_step(acts(), translate=True),
        "preview K=3 translate": lambda: env.preview_step(acts(3), translate=True),
        "preview K=3 f64": lambda: env.preview_step(acts(3, dtype=torch.float64)),
        "get_obs view, first": lambda: env.get_obs(),
        "get_obs view": lambda: env.get_obs(),
        "obs_ring, first": lambda: env.obs_ring(),
        "step return_obs=True": lambda: env.step(acts(), return_obs=True),
        "step return_obs=ring": lambda: env.step(acts(), return_obs="ring"),
        "step return_obs=ring again": lambda: env.step(acts(), return_obs="ring"),
        "step return_obs=ring masked": lambda: env.step(acts(), mask=mask, return_obs="ring"),
        "step return_obs=ring translate": lambda: env.step(acts(), translate=True, return_obs="ring"),
        "step return_obs=True translate": lambda: env.step(acts(), translate=True, return_obs=True),
        "get_obs dense": lambda: env.get_obs(contiguous=True),
        "get_obs dense, no push": lambda: env.get_obs(push=False, contiguous=True),
        "get_obs view after dense": lambda: env.get_obs(),
        "get_state": lambda: env.get_state(),
        "power_flow": lambda: env.power_flow(p, q),
        "safety_project": lambda: env.safety_project(acts()),
        "safety_project_affine": lambda: env.safety_project_affine(acts()),
    }
    col = 1 if variant == "thread" else 2
    seen, want = [], []
    for row in EXPECTED:
        verb = row[0].replace(", rings live", "")
        before = env.launch_count()
        verbs[verb]()
        seen.append((row[0], env.launch_count() - before))
        want.append((row[0], row[col]))
    torch.cuda.synchronize(cuda)
    env.close()
    assert seen == want, "\n".join(f"{v:40s} {d:3d}  expected {w:3d}" for (v, d), (_, w) in zip(seen, want))
