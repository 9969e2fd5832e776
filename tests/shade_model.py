"""One bounce of k_shade / k_scan restated per slot in numpy: the exact model that the shading tests hold the kernels to.

Plain functions over arrays (no pytest here), imported by tests/test_shade_model.py, which pins them to the C oracle, and by
tests/test_gpu_wavefront_exact.py, which holds ptap_shade and ptap_render to them.

What is exact and what is bounded:
  - the RNG (utility.h:43-62 + thrust::minstd_rand + uniform_real_distribution<float>) is restated in integers: bit for bit;
  - survival, stable compaction order, throughput (x albedo, x 0.01f on a miss), new origins pt + 0.1 n, reflections, unchanged rays of
    SPECULAR / REFRACTIVE and the film contribution sqrt(throughput) are binary32 arithmetic without a transcendental: bit for bit;
  - sampled directions go through sinf / cosf / powf: they are evaluated here in float64 from the exact float32 draws and the exact
    float32 frame vectors, and compared within DIR_TOL, plus, for METAL, the error that powf's few ulp in cos(theta) cause in
    sin(theta) = sqrt(1 - cos^2), bounded by its condition number (it grows as cos / sin when the lobe sample is near the axis).
"""
from __future__ import annotations

import numpy as np

f32 = np.float32
FLOAT_MAX = f32(9999999.0)
DIFFUSE, SPECULAR, REFLECTIVE, REFRACTIVE, EMISSIVE, COAT, METAL = range(7)
K_MAX_DEPTH = 16                     # ptap.h: rounds a frame may have
DIR_TOL = 2e-6                       # libdevice sinf / cosf against float64: a few ulp of a unit vector
POWF_ULP = 4                         # CUDA Math API: maximum ulp error of powf
M31 = 2147483647                     # minstd_rand's modulus 2^31 - 1
TWO_PI = f32(6.2831853071795864769252867665590057683943)           # utility.h:20
SQRT_ONE_THIRD = f32(0.5773502691896257645091487805019574556476)   # utility.h:21

# Edge seeds of the RNG as (iter, slot, remaining).  Found by a vectorised search: for each remaining in 2..16 and every iter < 2^22
# (2^16 for the second), h = utilHash(0x80000000 | remaining << 22 | iter) was matched against utilHash(slot) ^ target for the 256
# slots below 256 (a sorted table and searchsorted).  ZERO_SEED's hash is 2 * (2^31 - 1), so hash mod (2^31 - 1) = 0 and the seed rule
# makes the state 1.  ONE_DRAW's first draw leaves a state in [2^31 - 63, 2^31 - 2], where (float)(x - 1) rounds up to 2^31: u01 = 1.0f.
ZERO_SEED = (4025021, 144, 2)
ONE_DRAW = (55644, 75, 5)


# ---------------------------------------------------------------------------------------------------------------------------- RNG

def util_hash(a):
    """utility.h:43-53 in uint32."""
    a = np.asarray(a).astype(np.uint32)
    u = np.uint32
    with np.errstate(over="ignore"):
        a = (a + u(0x7ed55d16)) + (a << u(12))
        a = (a ^ u(0xc761c23c)) ^ (a >> u(19))
        a = (a + u(0x165667b1)) + (a << u(5))
        a = (a + u(0xd3a2646c)) ^ (a << u(9))
        a = (a + u(0xfd7046c5)) + (a << u(3))
        a = (a ^ u(0xb55a4f09)) ^ (a >> u(16))
    return a


def seed_hash(it, slot, remaining):
    """The 32-bit seed before thrust's reduction: bits of `it` at and above 2^22 overlap the remaining-bounce bits, as in the reference."""
    it = np.asarray(it).astype(np.int64).astype(np.uint32)
    rem = np.asarray(remaining).astype(np.int64).astype(np.uint32)
    with np.errstate(over="ignore"):
        key = np.uint32(0x80000000) | (rem << np.uint32(22)) | it
    return util_hash(key) ^ util_hash(np.asarray(slot).astype(np.int64).astype(np.uint32))


def rng_seed(it, slot, remaining):
    """minstd_rand state after seeding: hash mod (2^31 - 1), 0 -> 1 (int64)."""
    x = seed_hash(it, slot, remaining).astype(np.int64) % M31
    return np.where(x == 0, 1, x)


def rng_draws(state, k):
    """k draws of uniform_real_distribution<float>(0, 1) from each state: x <- 48271 x mod (2^31 - 1), u = (float)(x - 1) / 2^31.
    Returns a (..., k) float32 array; the conversion rounds to nearest, so u can be exactly 1.0f."""
    x = np.asarray(state, np.int64)
    out = []
    for _ in range(k):
        x = (x * 48271) % M31
        out.append((x - 1).astype(np.float32) / f32(2147483648.0))
    return np.stack(out, axis=-1)


# ------------------------------------------------------------------------------------------------------- binary32 vector helpers

def dot32(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def cross32(x, y):
    return np.stack([x[..., 1] * y[..., 2] - y[..., 1] * x[..., 2],
                     x[..., 2] * y[..., 0] - y[..., 2] * x[..., 0],
                     x[..., 0] * y[..., 1] - y[..., 0] * x[..., 1]], axis=-1)


def normalize32(v):
    """v * (1 / sqrt(dot(v, v))), every operation rounded to binary32 (glm::normalize as the kernels evaluate it)."""
    return v * (f32(1.0) / np.sqrt(dot32(v, v)))[..., None]


def reflect32(i, n):
    """utility.h:64-69: n - n * (2 (i.n))."""
    return n - n * (f32(2.0) * dot32(i, n))[..., None]


def _pick(mask, a, b):
    return np.where(mask[..., None], np.asarray(a, np.float32), np.asarray(b, np.float32))


# ---------------------------------------------------------------------------------------------------------------------- scatter

def hemisphere(n, u_up, u_around):
    """utility.h:91-123 in float64 from the float32 draws and the float32 frame (up, over, around, p1, p2 are exact binary32)."""
    up = np.sqrt(u_up)
    over = np.sqrt(f32(1.0) - up * up)
    around = u_around * TWO_PI
    nn = _pick(np.abs(n[..., 0]) < SQRT_ONE_THIRD, (1, 0, 0), _pick(np.abs(n[..., 1]) < SQRT_ONE_THIRD, (0, 1, 0), (0, 0, 1)))
    p1 = normalize32(cross32(n, nn))
    p2 = normalize32(cross32(n, p1))
    a = around.astype(np.float64)[..., None]
    ov = over.astype(np.float64)[..., None]
    return n.astype(np.float64) * up.astype(np.float64)[..., None] + p1 * (np.cos(a) * ov) + p2 * (np.sin(a) * ov)


def metal(n, d, u_phi, u_r2):
    """utility.h:145-170 (after its two unused draws): (direction in float64, extra tolerance).  cos(theta) = powf(1 - r2, 1/31) carries
    POWF_ULP ulp; sin(theta) = sqrt(1 - cos^2) amplifies that by cos / sin.  The extra tolerance is the worst change of sin(theta)
    over that interval of cos(theta) (and the rounding of cos^2), evaluated exactly rather than linearised, so it stays finite at sin = 0."""
    phi = TWO_PI * u_phi
    base = (f32(1.0) - u_r2).astype(np.float64)
    expo = np.float64(f32(1.0) / (f32(30.0) + f32(1.0)))
    c = base ** expo
    s = np.sqrt(np.maximum(0.0, 1.0 - c * c))
    dc = POWF_ULP * np.spacing(c.astype(np.float32)).astype(np.float64)
    e = 2.0 * c * dc + 2.0 ** -24                                     # |error of 1 - c*c| in binary32: powf's error plus the product's rounding
    ds = np.maximum(s - np.sqrt(np.maximum(s * s - e, 0.0)), np.sqrt(s * s + e) - s) + 2.0 ** -24 * s
    w = normalize32(d - (n * f32(2.0)) * dot32(n, d)[..., None])
    a = _pick(np.abs(w[..., 0]).astype(np.float64) > 0.1, (0, 1, 0), (1, 0, 0))
    uu = normalize32(cross32(a, w))
    vv = cross32(w, uu)
    p = phi.astype(np.float64)[..., None]
    out = uu * (np.cos(p) * s[..., None]) + vv * (np.sin(p) * s[..., None]) + w * c[..., None]
    return out, ds + dc


def scatter(kind, n, d, it, slot, remaining):
    """New direction of a DIFFUSE (0) / METAL (1) / COAT (2) bounce, or a reflection (3), for arrays of float32 normals and normalised
    directions: (direction float64, tolerance, exact) where `exact` marks directions that are binary32 arithmetic only (reflections)."""
    n = np.asarray(n, np.float32); d = np.asarray(d, np.float32)
    kind = np.broadcast_to(np.asarray(kind), n.shape[:-1])
    u = rng_draws(np.broadcast_to(rng_seed(it, slot, remaining), n.shape[:-1]), 4)
    out = np.zeros(n.shape, np.float64)
    tol = np.full(n.shape[:-1], DIR_TOL)
    exact = np.zeros(n.shape[:-1], bool)
    k = kind == 0
    out[k] = hemisphere(n[k], u[k, 0], u[k, 1])
    k = kind == 1
    out[k], extra = metal(n[k], d[k], u[k, 2], u[k, 3])
    tol[k] += extra
    k = kind == 2
    refl = k & (u[..., 0] < f32(0.5))
    out[refl] = reflect32(d[refl], n[refl]); exact[refl] = True
    hem = k & ~refl
    out[hem] = hemisphere(n[hem], u[hem, 1], u[hem, 2])
    k = kind == 3
    out[k] = reflect32(d[k], n[k]); exact[k] = True
    return out, tol, exact


# ------------------------------------------------------------------------------------------------------------------- one bounce

def survives(hit, mat_type, remaining):
    """A path continues after this bounce: it hit something, has bounces left after this one, and did not hit an emitter."""
    return hit & (remaining > 1) & (mat_type != EMISSIVE)


def attenuate(color, hit, mat_type, albedo):
    """Throughput after the bounce: x albedo for DIFFUSE / METAL / COAT / EMISSIVE / REFLECTIVE hits, unchanged for SPECULAR /
    REFRACTIVE (and any other type), x 0.01f on a miss.  binary32, per channel."""
    mult = hit & np.isin(mat_type, (DIFFUSE, METAL, COAT, EMISSIVE, REFLECTIVE))
    out = np.array(color, np.float32, copy=True)
    out[mult] = out[mult] * np.asarray(albedo, np.float32)[mult]
    out[~hit] = out[~hit] * f32(0.01)
    return out


def shade(orig, dir, color, hit, dist, normal, mat_type, albedo, it, remaining, directions=True):
    """k_shade for every slot i of a round (slot = index, which seeds the RNG).  Inputs are per-slot arrays; `dist` is the world
    distance the shade kernel uses.  Returns a dict:
      alive (n,), order (survivor slots in stable order), color (n, 3) throughput after the bounce, contrib (n, 3) = sqrt(color),
      and for the survivors in order: orig (binary32, exact), dir (float64), dir_tol, dir_exact (directions=False: no directions)."""
    orig = np.asarray(orig, np.float32); dir = np.asarray(dir, np.float32); normal = np.asarray(normal, np.float32)
    n = len(orig)
    alive = survives(hit, mat_type, remaining)
    col = attenuate(color, hit, mat_type, albedo)
    order = np.nonzero(alive)[0]
    o, d, nrm, t = orig[order], dir[order], normal[order], mat_type[order]
    dn = normalize32(d)
    pt = o + dn * np.asarray(dist, np.float32)[order][:, None]
    moved = np.isin(t, (DIFFUSE, METAL, COAT, REFLECTIVE))
    new_o = np.where(moved[:, None], pt + nrm * f32(0.1), o)
    if not directions:
        return {"alive": alive, "order": order, "color": col, "contrib": np.sqrt(col), "orig": new_o, "n": n}
    kind = np.select([t == DIFFUSE, t == METAL, t == COAT, t == REFLECTIVE], [0, 1, 2, 3], -1)
    new_d, tol, exact = scatter(np.where(kind < 0, 3, kind), nrm, dn, it, order, remaining)
    keep = kind < 0                                                   # SPECULAR / REFRACTIVE: no branch, ray unchanged
    new_d[keep] = d[keep]; tol[keep] = 0.0; exact[keep] = True
    return {"alive": alive, "order": order, "color": col, "contrib": np.sqrt(col), "orig": new_o, "dir": new_d,
            "dir_tol": tol, "dir_exact": exact, "n": n}


def dir_errors(got, model):
    """(worst error / tolerance over the sampled directions, whether every exact direction is bit-equal)."""
    got = np.asarray(got, np.float32)
    ex = model["dir_exact"]
    err = np.abs(got.astype(np.float64) - model["dir"]).max(axis=-1) if len(got) else np.zeros(0)
    ratio = float((err[~ex] / model["dir_tol"][~ex]).max(initial=0.0))
    same = bool(np.array_equal(got[ex], model["dir"][ex].astype(np.float32)))
    return ratio, same


# ------------------------------------------------------------------------------------------------------------------------ film

def predict_film(probes, H, W, depth):
    """The film ptap_render must produce, bit for bit.  probes[iteration][round] = (pixels, hit, mat_type, albedo) of every round's
    wavefront in slot order (hit: bool, albedo: (n, 3) float32 of the hit model).  Paths are chained through the rounds by pixel,
    throughputs multiplied in round order in binary32, and each iteration's sqrt(throughput) contributions added to a zero film in
    iteration order (each pixel owns one path per iteration)."""
    film = np.zeros((H * W, 3), np.float32)
    for rounds in probes:
        col = np.ones((H * W, 3), np.float32)
        for r, (pix, hit, mat_type, albedo) in enumerate(rounds):
            c = attenuate(col[pix], hit, mat_type, albedo)
            col[pix] = c
            done = ~survives(hit, mat_type, depth - r)
            film[pix[done]] += np.sqrt(c[done])
    return film.reshape(H, W, 3)
