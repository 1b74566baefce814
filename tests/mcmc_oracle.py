"""CPU restatement of splatfacto's MCMC strategy (nerfstudio 1.1.5 `strategy="mcmc"` -> gsplat 1.4.0 MCMCStrategy), in numpy
float64, for the tests of qed_splatter_b200/mcmc.py and csrc/mcmc.cu.

Restated from memory of the upstream code (gsplat/strategy/mcmc.py, gsplat/strategy/ops.py relocate / sample_add /
inject_noise_to_position, gsplat/relocation.py + csrc relocation kernel, nerfstudio splatfacto get_loss_dict); neither is
installed here.  `compute_relocation` keeps gsplat's literal double loop over the binomial table.

Also restated: Philox4x32-10 as curand_philox4x32_x.h defines it, and this library's sampler on top of it (quantised
inverse CDF, see csrc/mcmc.cu) and Box-Muller normals.
"""
from math import comb

import numpy as np

N_MAX = 51
FLT_EPS = float(np.finfo(np.float32).eps)
_M = 0xFFFFFFFF


def sigmoid32(x):
    x = np.asarray(x, np.float32)
    return (np.float32(1.0) / (np.float32(1.0) + np.exp(-x))).astype(np.float32)


# ---- gsplat compute_relocation (literal) --------------------------------------------------------------------------------
def binoms(n_max=N_MAX):
    b = np.zeros((n_max, n_max), np.float64)
    for n in range(n_max):
        for k in range(n + 1):
            b[n, k] = comb(n, k)
    return b


def compute_relocation(o, scales, ratios, n_max=N_MAX):
    """o [n], scales [n,3] (exp of the log-scales), ratios [n] -> (o', scale') unclamped, float64, gsplat's double loop."""
    B = binoms(n_max)
    o = np.asarray(o, np.float64)
    scales = np.asarray(scales, np.float64)
    ratios = np.clip(np.asarray(ratios), 1, n_max)
    o_new = np.empty_like(o)
    s_new = np.empty_like(scales)
    for t in range(o.size):
        n = int(ratios[t])
        x = 1.0 - (1.0 - o[t]) ** (1.0 / n)
        d = 0.0
        for i in range(1, n + 1):
            for k in range(i):
                d += B[i - 1, k] * ((-1.0) ** k / np.sqrt(k + 1.0)) * x ** (k + 1)
        o_new[t] = x
        s_new[t] = o[t] / d * scales[t]
    return o_new, s_new


def denominator_identity(x, n):
    """The same denominator by the hockey-stick identity: sum_{j=1..n} C(n, j) (-1)^(j-1) x^j / sqrt(j)."""
    return sum(comb(n, j) * (-1.0) ** (j - 1) * x ** j / np.sqrt(j) for j in range(1, n + 1))


def _relocation_update(p, rows, counts, min_opacity):
    """compute_relocation on the unique drawn rows (ratio = bincount + 1) and the writes of logit(o'), log(scale')."""
    o = sigmoid32(p["opacities"][rows]).astype(np.float64)
    sc = np.exp(p["scales"][rows].astype(np.float32)).astype(np.float64)
    o_new, s_new = compute_relocation(o, sc, counts[rows] + 1)
    o_new = np.clip(o_new.astype(np.float32), np.float32(min_opacity), np.float32(1.0 - FLT_EPS)).astype(np.float64)
    p["opacities"][rows] = np.log(o_new / (1.0 - o_new))
    p["scales"][rows] = np.log(s_new.astype(np.float32).astype(np.float64))


def relocate(p, m, v, draws, dead, min_opacity):
    """gsplat ops.relocate given the draws (alive rows, one per dead row): params / moments are dicts of float64 arrays
    (means [N,3], quats [N,4], scales [N,3] log, opacities [N] logit, sh [N,16,3]); updated in place."""
    draws = np.asarray(draws, np.int64)
    dead = np.asarray(dead, np.int64)
    N = p["means"].shape[0]
    counts = np.bincount(draws, minlength=N)
    rows = np.unique(draws)
    _relocation_update(p, rows, counts, min_opacity)
    for g in p:
        p[g][dead] = p[g][draws]
        m[g][rows] = 0.0  # drawn rows only (gsplat's optimizer_fn: v[sampled_idxs] = 0)
        v[g][rows] = 0.0


def sample_add(p, m, v, draws, min_opacity):
    """gsplat ops.sample_add given the draws -> new (p, m, v) dicts with len(draws) rows appended."""
    draws = np.asarray(draws, np.int64)
    N = p["means"].shape[0]
    counts = np.bincount(draws, minlength=N)
    _relocation_update(p, np.unique(draws), counts, min_opacity)
    p2 = {g: np.concatenate([p[g], p[g][draws]]) for g in p}
    m2 = {g: np.concatenate([m[g], np.zeros_like(m[g][draws])]) for g in m}
    v2 = {g: np.concatenate([v[g], np.zeros_like(v[g][draws])]) for g in v}
    return p2, m2, v2


def quat_to_rotmat(q):
    q = q / np.maximum(np.linalg.norm(q, axis=-1, keepdims=True), 1e-12)
    w, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y),
                     2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x),
                     2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)], -1).reshape(-1, 3, 3)


def inject_noise(p, normals, scaler):
    """gsplat inject_noise_to_position given the normals [N,3] (randn_like(means) upstream): means += covar @ noise."""
    o = 1.0 / (1.0 + np.exp(-p["opacities"]))
    R = quat_to_rotmat(p["quats"])
    S = np.exp(p["scales"])
    covar = np.einsum("nij,nj,nkj->nik", R, S * S, R)
    noise = normals * (1.0 / (1.0 + np.exp(-100.0 * ((1.0 - o) - 0.995))))[:, None] * scaler
    p["means"] = p["means"] + np.einsum("nij,nj->ni", covar, noise)


def regularizers(logit_op, log_scales, opacity_reg, scale_reg):
    """splatfacto get_loss_dict with mcmc: -> (opacity term, scale term, d/d logit_op, d/d log_scales)."""
    o = 1.0 / (1.0 + np.exp(-np.asarray(logit_op, np.float64)))
    e = np.exp(np.asarray(log_scales, np.float64))
    N = o.size
    return opacity_reg * o.mean(), scale_reg * e.mean(), opacity_reg / N * o * (1 - o), scale_reg / e.size * e


# ---- Philox4x32-10 (curand_philox4x32_x.h) and the sampler / normals of csrc/mcmc.cu ---------------------------------------
def philox4x32_10(c0, c1, c2, c3, seed):
    c = [np.asarray(x, np.uint64) & np.uint64(_M) for x in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(seed & _M), np.uint64((seed >> 32) & _M)
    M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    for r in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & np.uint64(_M)
        hi1, lo1 = p1 >> np.uint64(32), p1 & np.uint64(_M)
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(0x9E3779B9)) & np.uint64(_M)
        k1 = (k1 + np.uint64(0xBB67AE85)) & np.uint64(_M)
    return c


def weights(logit_op, min_opacity, zero_dead):
    w = np.floor(16777216.0 / (1.0 + np.exp(-np.asarray(logit_op, np.float32).astype(np.float64)))).astype(np.int64)
    if zero_dead:
        w[sigmoid32(logit_op) <= np.float32(min_opacity)] = 0
    return w


def sample(logit_op, n_draws, seed, step, stream_id, min_opacity=0.005, zero_dead=False):
    """-> (draws int64 [n_draws], total weight)."""
    cum = np.cumsum(weights(logit_op, min_opacity, zero_dead))
    total = int(cum[-1])
    if total == 0 or n_draws == 0:
        return np.zeros(0, np.int64), total
    j = np.arange(n_draws, dtype=np.uint64)
    x, y, _, _ = philox4x32_10(j, step, stream_id, 0, seed)
    u64 = (x << np.uint64(32)) | y
    u = np.array([(int(a) * total) >> 64 for a in u64.tolist()], dtype=np.int64)
    return np.searchsorted(cum, u, side="right").astype(np.int64), total


def uniform(x):
    return np.asarray(x, np.float64) * 2.0 ** -32 + 2.0 ** -33


def normals(N, seed, step):
    """[N,3]: Box-Muller on the four words of Philox counter (i, step, 0, 0): (x, y) -> n0, n1 and (z, w) -> n2."""
    x, y, z, w = philox4x32_10(np.arange(N, dtype=np.uint64), step, 0, 0, seed)
    r1, r2 = np.sqrt(-2.0 * np.log(uniform(x))), np.sqrt(-2.0 * np.log(uniform(z)))
    return np.stack([r1 * np.cos(2 * np.pi * uniform(y)), r1 * np.sin(2 * np.pi * uniform(y)), r2 * np.cos(2 * np.pi * uniform(w))], -1)
