"""TEST INFRASTRUCTURE — CPU restatement of the rollout policy's critic-guided plan search (tacorl_b200/rollout.py
PlanSearch / plan_search, csrc/plan_search.cu, DESIGN.md section 16.2): the search's Philox uniforms, its candidates,
the twin-critic score in fp64, the elite refit and best-so-far tracking as the device states them in fp32 (so that
they can be recomputed bit for bit from the device's own candidates and scores), and a whole search in fp64."""
import numpy as np
import torch

from oracle import replay_oracle as RO

SEARCH_DRAW0 = 256                 # the search's first draw (decoder: 0..16, policy sampler: 32 + d)


def _u24(w):
    return (np.asarray(w) >> 8).astype(np.float32) * np.float32(2.0 ** -24)


def search_uniforms(seed, t, env_id, k, K, P):
    """(u_a, u_b), each (K, P) float32, of round k of one environment: candidate c, dimension d takes words 0 and 1 of
    the Philox4x32-10 draw j = 256 + (k K + c) P + d, key (lo32(seed), hi32(seed)), counter (lo32(t), hi32(t), env_id,
    j), as (w >> 8) 2^-24."""
    seed, t = int(seed) & 0xFFFFFFFFFFFFFFFF, int(t) & 0xFFFFFFFFFFFFFFFF
    j = SEARCH_DRAW0 + (k * K + np.arange(K, dtype=np.uint64)[:, None]) * P + np.arange(P, dtype=np.uint64)[None, :]
    w0, w1, _, _ = RO.philox4x32_10(t & 0xFFFFFFFF, t >> 32, int(env_id), j, seed & 0xFFFFFFFF, seed >> 32)
    return _u24(w0), _u24(w1)


def candidates(mu, sigma, ua, ub, k):
    """Round k's pre-tanh candidates (K, P) in fp64: mu + sigma sqrt(-2 ln(1 - u_a)) cos(2 pi u_b); candidate 0 of
    round 0 is mu itself."""
    ua, ub = torch.as_tensor(ua).double(), torch.as_tensor(ub).double()
    eps = torch.sqrt(-2.0 * torch.log1p(-ua)) * torch.cos(2.0 * np.pi * ub)
    z = torch.as_tensor(mu).double() + torch.as_tensor(sigma).double() * eps
    if k == 0:
        z[0] = torch.as_tensor(mu).double()
    return z


def q_mlp(layers, x):
    """MLPQNetwork on x: SiLU after every layer but the last.  layers: [(W, b)], fp64."""
    for i, (W, b) in enumerate(layers):
        x = x @ W.double().t() + b.double()
        if i < len(layers) - 1:
            x = x * torch.sigmoid(x)
    return x[..., 0]


def score(critics, e, z):
    """min(Q1(e_1, tanh z), Q2(e_2, tanh z)) in fp64, NaN -> -inf.  critics: two layer lists; e: the two (D,) inputs
    (embedding | goal embedding); z (K, P)."""
    a = torch.tanh(z.double())
    q = [q_mlp(critics[j], torch.cat([e[j].double().expand(a.shape[0], -1), a], -1)) for j in range(2)]
    s = torch.minimum(q[0], q[1])
    return torch.where(torch.isnan(q[0]) | torch.isnan(q[1]), torch.full_like(s, -np.inf), s)


def elites(scores, E):
    """Indices (ascending) of the E best scores, ties to the lower index."""
    s = np.asarray(scores, dtype=np.float64)
    order = sorted(range(len(s)), key=lambda c: (-s[c], c))
    return sorted(order[:E])


def refit_f32(z, scores, E, min_std):
    """The refit as the device computes it, in fp32: the elites' mean (sum in ascending c, / E), then the population std
    (squared deviations summed in ascending c, / E, sqrt) floored at min_std.  z (K, P) float32 -> (mu, sigma) (P,)."""
    z = np.asarray(z, dtype=np.float32)
    idx = elites(scores, E)
    s = np.zeros(z.shape[1], dtype=np.float32)
    for c in idx:
        s = s + z[c]
    m = s / np.float32(E)
    q = np.zeros_like(m)
    for c in idx:
        d = z[c] - m
        q = q + d * d
    sd = np.sqrt(q / np.float32(E))
    return m, np.maximum(sd, np.float32(min_std))


def best_update(best, k, z, scores):
    """Best-so-far after round k: best = None or (z (P,), score); a round's best (ties: lower c) replaces it only when
    strictly better, so ties keep the earliest (k, c)."""
    s = np.asarray(scores, dtype=np.float64)
    c = elites(s, 1)[0]
    if best is None or k == 0 or s[c] > best[1]:
        return np.asarray(z[c]).copy(), float(s[c])
    return best


def search(critics, e, mu, sigma, samples, elites_n, iterations, min_std, seed, t, env_id):
    """The whole search of one environment in fp64 (the refit in fp64 too).  Returns (plan (P,), value, trace), trace
    a list of per-round dicts {z, scores, mu, sigma}."""
    mu, sigma = torch.as_tensor(mu).double(), torch.as_tensor(sigma).double()
    P = mu.shape[0]
    best, trace = None, []
    for k in range(iterations):
        ua, ub = search_uniforms(seed, t, env_id, k, samples, P)
        z = candidates(mu, sigma, ua, ub, k)
        s = score(critics, e, z)
        trace.append({"z": z, "scores": s, "mu": mu, "sigma": sigma})
        best = best_update(best, k, z.numpy(), s.numpy())
        zi = z[elites(s.numpy(), elites_n)]
        mu = zi.mean(0)
        sigma = torch.clamp(((zi - mu) ** 2).mean(0).sqrt(), min=min_std)
    return torch.tanh(torch.as_tensor(best[0])), best[1], trace
