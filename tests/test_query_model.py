"""CPU model of the early exit of the any-hit traversal (k_trace_bvh<.., ANY>, ptap_query_occluded; DESIGN.md 4.8).

Occlusion of a segment of world length L is defined through the closest hit: R1.model >= 0 and R1.dist < L.  The any-hit kernel retires a
ray as occluded at an accepted triangle of model m with model-space t when

    M + (M * tie + cb) < min(L, FLOAT_MAX),    M = max(|t|, EPSILON) * ascale,

ascale = |d_w| / |W3 d_w| (world units per model-space t, computed at instance entry), tie and cb the slack of the kernel's exit step.
L is clamped to FLOAT_MAX because a hit at world distance FLOAT_MAX or more is a miss of the closest hit (the reference starts
min_dist there): with L = inf, "any hit" means any hit the closest-hit query reports.
Everywhere else it only tightens bounds that were already conservative, so the answer stays the closest hit's.  This file checks the
early-exit half without a GPU: wherever the rule would fire for some accepted hit of some model, the oracle's closest hit (tier R1) is
nearer than L.  The inputs are the oracle's probes: every accepted hit of a model, the exact world distance of a hit, and R1 itself."""
import numpy as np

from test_gpu_production import _sphere_scene

EPSILON = np.float32(0.005)         # Config.h:4
TIE = np.float32(1.5e-4)            # api.cu: sc.tie of a scene whose matrices are inverses
FLOAT_MAX = np.float32(9999999.0)   # Config.h:5
F32 = np.float32


def _slack(models):
    """c_pad as the upload computes it: 4e-5 * max(1, largest |translation|) + 1e-3, rounded once to binary32."""
    m2w = models["model_to_world"].astype(np.float64)
    max_trans = max(1.0, float(np.abs(m2w[:, 12:15]).max()))
    return F32(4e-5 * max_trans + 1e-3)


def _ascale(w2m, d):
    """|d_w| / |W3 d_w| in binary32 as the kernel's instance entry forms it (xmat4: row sums in order; rsqrt and a fast divide there, so
    the upper end of a few ulps is taken: the rule only gets easier to fire)."""
    w = w2m.astype(np.float32)
    dm = [F32(F32(F32(w[r] * d[0]) + F32(w[4 + r] * d[1])) + F32(w[8 + r] * d[2])) for r in range(3)]
    mlen = F32(np.sqrt(F32(F32(F32(dm[0] * dm[0]) + F32(dm[1] * dm[1])) + F32(dm[2] * dm[2]))))
    wil = F32(1.0) / F32(np.sqrt(F32(F32(F32(d[0] * d[0]) + F32(d[1] * d[1])) + F32(d[2] * d[2]))))
    return F32(F32(F32(1.0) / F32(mlen * wil)) * F32(1.0 + 1e-6))


def _threshold(m, cb):
    """The smallest L - as the binary32 expression M + (M * tie + cb) - below which the rule does not fire for hit scale M."""
    return F32(m + F32(F32(m * TIE) + cb))


def _check(oscene, rays, rs):
    a = oscene.arrays()
    models = a["models"]
    c_pad = _slack(models)
    want = oscene.trace(rays, 1)
    fired = checked = 0
    for i, ray in enumerate(rays):
        o, d = ray[:3], ray[3:]
        cb = F32(c_pad + F32(F32(1e-4) * F32(F32(F32(abs(o[0])) + F32(abs(o[1]))) + F32(abs(o[2])))))
        thr_min = np.inf
        Ls = []
        for im in range(len(models)):
            tri, t = oscene.model_hits(ray, im)
            if len(t) == 0:
                continue
            asc = _ascale(models[im]["world_to_model"], d)
            m = np.maximum(np.abs(t), EPSILON).astype(np.float32) * asc
            thr = np.array([_threshold(F32(x), cb) for x in m], np.float32)
            thr_min = min(thr_min, float(thr.min()))
            Ls += [np.nextafter(F32(EPSILON * asc), F32(np.inf)), np.nextafter(thr.min(), F32(np.inf)), thr.min()]
            k = rs.randint(len(t))
            Ls.append(oscene.hit_distance(ray, im, t[k]))                   # L equal to a hit's own world distance
        hit = want["model"][i] >= 0
        dist = want["dist"][i]
        Ls += [F32(rs.uniform(0, 2 * dist)) if hit else F32(rs.uniform(0, 2000)), F32(np.inf), F32(5e7), FLOAT_MAX]
        for L in Ls:
            if thr_min < min(L, FLOAT_MAX):                                 # the kernel would retire the ray as occluded
                fired += 1
                assert hit and dist < L, f"ray {i}: the early exit fires at L = {L!r}, but R1 = ({want['model'][i]}, {dist!r})"
            checked += 1
        if thr_min < FLOAT_MAX:                                             # and for every L: the rule fires iff min(L, FLOAT_MAX) > thr_min
            assert hit and dist <= thr_min, f"ray {i}: R1 dist {dist!r} beyond the rule's threshold {thr_min!r}"
    return fired, checked


def _rays(n, seed):
    rs = np.random.RandomState(seed)
    o = np.stack([rs.uniform(-450, 500, n), rs.uniform(-100, 850, n), rs.uniform(-450, 900, n)], 1)
    d = rs.randn(n, 3)
    d[: n // 25, rs.randint(0, 3)] = 0.0
    d *= rs.uniform(0.1, 30.0, (n, 1))
    return np.concatenate([o, d], 1).astype(np.float32)


def test_early_exit_rule_on_the_reference_scene(port, oracle_scene):
    """20,000 random rays through the room of the reference's coded scene (11 models, world scales from 0.25 to 100)."""
    rs = np.random.RandomState(3)
    fired, checked = _check(oracle_scene, _rays(20000, 47), rs)
    assert fired > 10000 and checked - fired > 10000, (fired, checked)


def test_early_exit_rule_at_large_instance_scale(port):
    """Instances scaled x500 ... x900: the t >= -EPSILON band is several world units wide, so the EPSILON term of M decides.  Rays start
    0.1 to 20 world units off (and inside) the surfaces at every angle, grazing included."""
    scales = [500.0, 650.0, 900.0, 520.0, 700.0]
    s, centres = _sphere_scene(scales, 11)
    a = s.arrays()
    oscene = port.OracleScene({k: a[k] for k in ("models", "meshes", "vertices", "triangles")})
    rs = np.random.RandomState(13)
    rays = []
    for c, sc in centres:
        n = 4000
        p = rs.randn(n, 3); p /= np.linalg.norm(p, axis=1, keepdims=True)
        o = c + p * sc + p * rs.choice([-20.0, -3.0, -0.1, 0.1, 1.0, 3.0, 20.0], n)[:, None]
        t = rs.randn(n, 3); t -= p * np.sum(t * p, axis=1, keepdims=True); t /= np.linalg.norm(t, axis=1, keepdims=True)
        ang = rs.choice([0.0, 1e-3, 1e-2, 0.1, 0.5, 1.5], n)[:, None] * rs.choice([-1.0, 1.0], n)[:, None]
        d = (t * np.cos(ang) + p * np.sin(ang)) * rs.uniform(0.2, 40.0, (n, 1))
        rays.append(np.concatenate([o, d], 1))
    rays = np.concatenate(rays).astype(np.float32)
    want = oscene.trace(rays, 1)
    assert ((want["model"] >= 0) & (want["t_model"] < 0)).sum() > 100, "the test must exercise winners behind the origin"
    fired, checked = _check(oscene, rays, rs)
    assert fired > 10000 and checked - fired > 10000, (fired, checked)
    # origins 0.9e7 to 3e7 world units away, aimed at the instances: their hits straddle FLOAT_MAX, beyond which the closest hit is a
    # miss however many triangles the predicate accepts, so L = inf or 5e7 must not retire those rays
    far = far_rays(centres, 2000, 14)
    wf = oscene.trace(far, 1)
    beyond = sum(len(oscene.model_hits(r, im)[1]) > 0 for r in far[wf["model"] < 0] for im in range(len(scales)))
    assert (wf["model"] >= 0).sum() > 100 and beyond > 100, ((wf["model"] >= 0).sum(), beyond)
    _check(oscene, far, rs)


def far_rays(centres, n_per, seed):
    """Rays from 0.9e7 ... 3e7 world units away towards the instance centres (slightly off-axis)."""
    rs = np.random.RandomState(seed)
    rays = []
    for c, sc in centres:
        p = rs.randn(n_per, 3); p /= np.linalg.norm(p, axis=1, keepdims=True)
        o = c + p * rs.uniform(0.9e7, 3e7, (n_per, 1))
        d = -p + rs.uniform(-0.3, 0.3, (n_per, 3)) * sc / np.linalg.norm(o - c, axis=1, keepdims=True)
        rays.append(np.concatenate([o, d * rs.uniform(0.5, 5.0, (n_per, 1))], 1))
    return np.concatenate(rays).astype(np.float32)
