"""Capsule-collision culls against the fp64 oracle on crowded, rotated, degenerate and near-contact scenes.

The LM assembly, the collision flags and the path metrics all find their colliding pairs the same way: a register cull
from bounding spheres (collision.cuh: self_cull_mask / env_cull_mask; k_metrics.cu: env_midpoint_bounds and the warp
threshold of the exact minima), then the exact closed form for the survivors.  A cull that is too tight drops a real
contact.  The tests here put contacts where that shows:

  * scenes of eight obstacles, so that the LM assembly's second survivor-mask group (obstacles OGRP = 64 / NCAP and up)
    and obstacle index 7 of the metrics' candidate encoding are used; rotated copies, so that the rotated-cuboid branch
    of every cull runs, mixed with identity ones in the same mask group; prefixes of 0, 1, OGRP, OGRP + 1 and 8 obstacles;
  * a degenerate scene: zero-thickness plates, and a box that swallows the base and the first links (capsule axes inside
    a box: d = -radius and no normal), evaluated on q = 0 and single-joint perturbations of it (axes parallel to faces);
  * near-contact configurations, found by fp64 bisection along joint-space segments, at signed distances of +-2e-5,
    +-2e-4 and +-2e-3 m on one chosen test - preferring geometry where the bounding-sphere bound is nearly tight, so that
    a cull a few millimetres too tight loses them.

Sign comparisons leave out every configuration with an oracle distance within SIGN_BAND of 0.  Gradient comparisons also
leave out configurations where the gradient of an active term is ill-defined: a capsule axis within AXIS_BAND of a box
surface (the kernels zero the normal below 1e-6 m, the oracle below 1e-12 m), or closest features so nearly parallel
that fp32 rounding of the same closed form alone moves the gradient by a quarter of its tolerance.  What is left out is
counted and bounded, so no check can become vacuous.
"""
import functools

import numpy as np
import pytest
import torch

from oracle import robots as R, kinematics as K, geometry as G, lm as L
from oracle.workloads import cuboid_tensors, random_configs, synthetic_problem

ROBOTS = ["fetch", "fetch_arm", "panda"]
DEV = "cuda:0"

SIGN_BAND = 5e-6          # |d| below this: the sign is not compared
AXIS_BAND = 1e-5          # capsule axis closer than this to a box surface: the normal is not compared
TOL_D = 1e-5              # fp32 capsule distance (test_gpu_parity.test_collision_distances_and_jacobians)
TOL_G_SELF, TOL_G_ENV = 2e-4, 2e-3  # fp32 distance gradients, same source
TARGETS = (-2e-3, -2e-4, -2e-5, 2e-5, 2e-4, 2e-3)
MAX_EXCLUDED = 0.05       # largest fraction of checked waypoints a band may leave out
MAX_INSENSITIVE = 0.10    # largest fraction of waypoints with active terms whose smallest term is within 10x the tolerance


def ogrp(r):
    """obstacles per 64-bit survivor mask of the LM assembly (k_lm_full.cu: OGRP = 64 / NCAP)"""
    return 64 // len(R.get_model(r).capsules)


def n_static(model):
    """leading capsules on links no joint moves (collision.cuh: n_static_capsules): the assembly does not test them"""
    first_moving = min(model.actuated) + 1
    return sum(1 for c in model.capsules if c.frame < first_moving)


def zero_config(model):
    lim = torch.tensor(model.actuated_joints_limits, dtype=torch.float64)
    return torch.zeros(model.ndof, dtype=torch.float64).clamp(lim[:, 0], lim[:, 1])


# ------------------------------------------------------------------------------------------------------------------
# scenes


class Scene:
    """Cuboids in the reference's convention (oracle.workloads.cuboid_tensors: [lo, hi] in the frame Tcuboid, Tcuboid[3,3]
    = 0), float32 - what the kernels receive; the oracle evaluates the same numbers in float64."""

    def __init__(self, name, cuboids, Tcuboids):
        self.name = name
        self.cuboids = [c.float() for c in cuboids]
        self.Tcuboids = [t.float() for t in Tcuboids]

    @property
    def n(self):
        return len(self.cuboids)

    def prefix(self, n):
        return Scene(f"{self.name}[:{n}]", self.cuboids[:n], self.Tcuboids[:n])

    def c64(self):
        return [c.double() for c in self.cuboids], [t.double() for t in self.Tcuboids]

    def ops_obstacles(self):
        from cppflow_b200 import ops

        return ops.Obstacles(self.cuboids, self.Tcuboids)


def _rotation(axis, ang):
    axis = np.asarray(axis, dtype=np.float64)
    axis = axis / np.linalg.norm(axis)
    Kx = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(ang) * Kx + (1 - np.cos(ang)) * (Kx @ Kx)


def _static_clear(model, cuboid, Tcuboid):
    """the capsules no joint moves stay 2 cm clear (else every configuration would collide with the obstacle)"""
    d = G.env_collision_distances(model, zero_config(model)[None], cuboid.double(), Tcuboid.double())[0]
    return float(d[: n_static(model)].min()) > 0.02


@functools.lru_cache(maxsize=None)
def crowded8(r):
    """8 axis-aligned cuboids of 5-30 cm, centred on points the arm's distal capsules reach, one per height band, spread in
    azimuth; each is hit by between 0.5 % and 35 % of random configurations, and mostly by the arm's distal links."""
    m = R.get_model(r)
    rng = np.random.default_rng({"fetch": 101, "fetch_arm": 102, "panda": 103}[r])
    x = random_configs(m, 3000, seed=104).double()
    P1, P2, _, _, _ = K.capsule_world_endpoints(m, x)
    pts = (0.5 * (P1 + P2))[:, -4:].reshape(-1, 3).numpy()  # the distal capsules' midpoints
    order = np.argsort(pts[:, 2])
    bands = np.array_split(order, 8)
    probe = random_configs(m, 1500, seed=105).double()
    boxes = []
    for k, band in enumerate(bands):
        az_goal = -2.6 + 5.2 * k / 7.0
        az = np.arctan2(pts[band, 1], pts[band, 0])
        cands = band[np.argsort(np.abs(np.angle(np.exp(1j * (az - az_goal)))))]
        for i in cands[:200]:
            size = rng.uniform(0.05, 0.30, 3)
            box = (*pts[i], *size)
            c, Tc = cuboid_tensors([box], torch.float64)
            d = G.env_collision_distances(m, probe, c[0], Tc[0])
            hit = (d.min(dim=1).values < 0).double().mean()
            # mostly hit by the arm: the links next to the shoulder have short lever arms (small distance gradients)
            near_shoulder = (d[:, : n_static(m) + 3].min(dim=1).values < 0).double().mean()
            if 0.005 < float(hit) < 0.35 and float(near_shoulder) < 0.02 and _static_clear(m, c[0], Tc[0]):
                boxes.append(box)
                break
        else:
            raise AssertionError(f"no obstacle placement for height band {k}")
    cuboids, Tcuboids = cuboid_tensors(boxes)
    return Scene("crowded8", cuboids, Tcuboids)


@functools.lru_cache(maxsize=None)
def rotated8(r):
    """crowded8's centres and sizes, rotated about random axes (clear of the capsules no joint moves); obstacles 2 and 6
    keep the identity, so that mask group 0 (and group 1 of the 10-capsule robots) mixes both branches of the culls"""
    base = crowded8(r)
    rng = np.random.default_rng({"fetch": 201, "fetch_arm": 202, "panda": 203}[r])
    Tcuboids = []
    m = R.get_model(r)
    for o, (c, Tc) in enumerate(zip(base.cuboids, base.Tcuboids)):
        Tc = Tc.clone()
        while o not in (2, 6):
            Tc[:3, :3] = torch.tensor(_rotation(rng.normal(size=3), rng.uniform(0.3, 2.8)), dtype=torch.float32)
            if _static_clear(m, c, Tc):
                break
        Tcuboids.append(Tc)
    return Scene("rotated8", base.cuboids, Tcuboids)


@functools.lru_cache(maxsize=None)
def degenerate(r):
    """a zero-thickness plate just beside a forearm capsule at q = 0 (the capsule's axis is parallel to it), a
    rotated zero-thickness plate across the forearm, and a box that encloses the base and the first links"""
    m = R.get_model(r)
    q0 = zero_config(m)[None]
    P1, P2, radii, _, _ = K.capsule_world_endpoints(m, q0)
    mid = (0.5 * (P1 + P2))[0]
    # the plate lies beside capsule len - 4 (Fetch's forearm, Panda's link5), normal to the world axis its q = 0 axis is
    # most nearly perpendicular to, half a radius from that axis
    c_mid = len(m.capsules) - 4
    k = int((P2 - P1)[0, c_mid].abs().argmin())
    centre = [float(v) for v in mid[c_mid]]
    centre[k] -= 0.5 * float(radii[c_mid])
    size = [0.4, 0.4, 0.4]
    size[k] = 0.0
    boxes = [
        (*centre, *size),
        (float(mid[-3, 0]), float(mid[-3, 1]), float(mid[-3, 2]), 0.0, 0.3, 0.3),
        # base + first links: Fetch's base and torso, Panda's link0 and link1
        (0.0, 0.0, 0.3, 0.7, 0.7, 0.6) if r.startswith("fetch") else (0.0, 0.0, 0.1, 0.3, 0.3, 0.2),
    ]
    cuboids, Tcuboids = cuboid_tensors(boxes)
    Tcuboids[1][:3, :3] = torch.tensor(_rotation([0.0, 0.3, 1.0], 0.6), dtype=torch.float32)
    return Scene("degenerate", cuboids, Tcuboids)


# ------------------------------------------------------------------------------------------------------------------
# fp64 oracle helpers


def _env_rows(model, x, lo, hi, Rb, tb):
    """[n, C] signed capsule-cuboid distances with one obstacle per row (the oracle's formula, G.env_collision_distances)"""
    P1, P2, radii, _, _ = K.capsule_world_endpoints(model, x)
    A = torch.einsum("ncj,njk->nck", P1 - tb[:, None], Rb)
    B = torch.einsum("ncj,njk->nck", P2 - tb[:, None], Rb)
    t = G.segment_box_closest(A, B, lo[:, None], hi[:, None])
    Cb = A + t[..., None] * (B - A)
    diff = Cb - torch.minimum(torch.maximum(Cb, lo[:, None]), hi[:, None])
    return diff.norm(dim=-1) - radii


def _bound_gap(model, x, scene, kind_env, pidx, oidx, cidx):
    """true distance minus the bounding-sphere lower bound the culls use (0 = the cull is tight), per row"""
    P1, P2, radii, _, _ = K.capsule_world_endpoints(model, x)
    hl = 0.5 * (P2 - P1).norm(dim=-1)
    mid = 0.5 * (P1 + P2)
    ar = torch.arange(x.shape[0])
    ia = torch.tensor([p[0] for p in model.pairs])[pidx]
    ib = torch.tensor([p[1] for p in model.pairs])[pidx]
    d_self = G.self_collision_distances(model, x)[ar, pidx]
    b_self = (mid[ar, ia] - mid[ar, ib]).norm(dim=-1) - hl[ar, ia] - hl[ar, ib] - radii[ia] - radii[ib]
    cu, Tc = scene.c64()
    lo = torch.stack([c[:3] for c in cu])[oidx]
    hi = torch.stack([c[3:] for c in cu])[oidx]
    Rb = torch.stack([t[:3, :3] for t in Tc])[oidx]
    tb = torch.stack([t[:3, 3] for t in Tc])[oidx]
    d_env = _env_rows(model, x, lo, hi, Rb, tb)[ar, cidx]
    mb = torch.einsum("nj,njk->nk", mid[ar, cidx] - tb, Rb)
    b_env = (mb - torch.minimum(torch.maximum(mb, lo), hi)).norm(dim=-1) - hl[ar, cidx] - radii[cidx]
    return torch.where(kind_env, d_env - b_env, d_self - b_self)


def _test_distance(model, x, scene, kind_env, pidx, oidx, cidx):
    ar = torch.arange(x.shape[0])
    cu, Tc = scene.c64()
    d_env = _env_rows(model, x, torch.stack([c[:3] for c in cu])[oidx], torch.stack([c[3:] for c in cu])[oidx],
                      torch.stack([t[:3, :3] for t in Tc])[oidx], torch.stack([t[:3, 3] for t in Tc])[oidx])[ar, cidx]
    d_self = G.self_collision_distances(model, x)[ar, pidx]
    return torch.where(kind_env, d_env, d_self)


def _bisect(model, scene, qa, qb, target, rows, iters=50):
    """fp64 bisection of d_test(qa + s (qb - qa)) = target for s in [0, 1] (d_test(qa) < target < d_test(qb)); the result is
    rounded to float32, the precision the kernels take"""
    lo = torch.zeros(qa.shape[0], dtype=torch.float64)
    hi = torch.ones_like(lo)
    for _ in range(iters):
        s = 0.5 * (lo + hi)
        below = _test_distance(model, qa + s[:, None] * (qb - qa), scene, *rows) < target
        lo, hi = torch.where(below, s, lo), torch.where(below, hi, s)
    return (qa + (0.5 * (lo + hi))[:, None] * (qb - qa)).float()


@functools.lru_cache(maxsize=None)
def near_contacts(r, scene_name):
    """Near-contact configurations of a scene: for every obstacle three capsule tests and for six self pairs one each,
    bisected to each of TARGETS.  Of 32 random candidate tests per obstacle (48 for the self pairs) the ones whose
    bounding-sphere bound is tightest at contact are kept (plus the first candidate), so that a cull that is a few
    millimetres too tight loses the contact.
    -> dict(x [n, D] float32, target [n], kind_env [n] bool, pidx, oidx, cidx [n] long)"""
    m = R.get_model(r)
    scene = SCENES[scene_name](r)
    g = torch.Generator().manual_seed(7 + len(scene_name) + 31 * ROBOTS.index(r))
    pool = random_configs(m, 6000, seed=300 + ROBOTS.index(r)).double()
    cu, Tc = scene.c64()
    ds = G.self_collision_distances(m, pool)
    de = torch.stack([G.env_collision_distances(m, pool, c, t) for c, t in zip(cu, Tc)], dim=1)  # [n, O, C]
    ns = n_static(m)
    cand = []  # (kind_env, p, o, c, qa index, qb index)

    def pick(dcol, n_take):
        bad = torch.nonzero(dcol < -0.005).flatten()
        good = torch.nonzero(dcol > 0.02).flatten()
        if len(bad) == 0 or len(good) == 0:
            return []
        ia = bad[torch.randperm(len(bad), generator=g)[:n_take]]
        ib = good[torch.randint(len(good), (len(ia),), generator=g)]
        return list(zip(ia.tolist(), ib.tolist()))

    groups = []
    for o in range(scene.n):
        rows = []
        for c in range(ns, len(m.capsules)):
            rows += [(True, 0, o, c, a, b) for a, b in pick(de[:, o, c], 8)]
        perm = torch.randperm(len(rows), generator=g)[:32].tolist()
        groups.append(([rows[i] for i in perm], 3))
    self_rows = []
    for p in range(len(m.pairs)):
        self_rows += [(False, p, 0, 0, a, b) for a, b in pick(ds[:, p], 4)]
    groups.append(([self_rows[i] for i in torch.randperm(len(self_rows), generator=g)[:48].tolist()], 6))

    def as_rows(sel):
        t = lambda k: torch.tensor([s[k] for s in sel])  # noqa: E731
        return (t(0).bool(), t(1).long(), t(2).long(), t(3).long()), pool[t(4)], pool[t(5)]

    chosen = []
    for sel, n_keep in groups:
        if not sel:
            continue
        rows, qa, qb = as_rows(sel)
        x = _bisect(m, scene, qa, qb, TARGETS[0], rows).double()
        gap = _bound_gap(m, x, scene, *rows)
        keep = [0] + [i for i in torch.argsort(gap).tolist() if i != 0][: n_keep - 1]
        chosen += [sel[i] for i in keep]
    rows, qa, qb = as_rows([s for s in chosen for _ in TARGETS])
    target = torch.tensor([tau for _ in chosen for tau in TARGETS], dtype=torch.float64)
    x = _bisect(m, scene, qa, qb, target, rows)
    d = _test_distance(m, x.double(), scene, *rows)
    gap = _bound_gap(m, x.double(), scene, *rows)
    kind_env, pidx, oidx, cidx = rows
    return dict(x=x, target=target, d=d, gap=gap, kind_env=kind_env, pidx=pidx, oidx=oidx, cidx=cidx)


def zero_family(model, n_per_joint=16):
    """q = 0 (clamped into the limits) and single-joint sweeps of it over each joint's range"""
    q0 = zero_config(model)
    lim = torch.tensor(model.actuated_joints_limits, dtype=torch.float64)
    xs = [q0[None]]
    for d in range(model.ndof):
        v = q0[None].repeat(n_per_joint, 1)
        v[:, d] = torch.linspace(float(lim[d, 0]), float(lim[d, 1]), n_per_joint, dtype=torch.float64)
        xs.append(v)
    return torch.cat(xs).float()


SCENES = {"crowded8": crowded8, "rotated8": rotated8, "degenerate": degenerate}


def scene_by_name(r, name):
    """'crowded8', 'rotated8', 'degenerate' or a prefix 'rotated8[:n]'"""
    if "[:" in name:
        base, n = name.split("[:")
        return SCENES[base](r).prefix(int(n[:-1]))
    return SCENES[name](r)


@functools.lru_cache(maxsize=None)
def waypoints(r, base_name, total):
    """`total` waypoints of a scene, shuffled: its near-contact configurations, q = 0 and its single-joint sweeps, and
    random configurations for the rest -> (x [total, D] float32, number of near-contact rows)"""
    m = R.get_model(r)
    nc = near_contacts(r, base_name)["x"]
    zf = zero_family(m)
    n_rand = total - len(nc) - len(zf)
    assert n_rand > 0
    x = torch.cat([nc, zf, random_configs(m, n_rand, seed=400 + ROBOTS.index(r))])
    perm = torch.randperm(total, generator=torch.Generator().manual_seed(500))
    return x[perm].contiguous(), len(nc)


@functools.lru_cache(maxsize=None)
def oracle_terms(r, base_name, total):
    """fp64 oracle of every collision test of the scene's waypoints (with gradients), plus fp32 gradients of the same
    closed form for the near-parallel criterion"""
    m = R.get_model(r)
    x, _ = waypoints(r, base_name, total)
    scene = SCENES[base_name](r)
    x64 = x.double()
    ds, Js = G.self_collision_distances(m, x64, with_jacobian=True)
    _, Js32 = G.self_collision_distances(m, x, with_jacobian=True)
    de, Je, Je32 = [], [], []
    for c, t in zip(scene.cuboids, scene.Tcuboids):
        d, J = G.env_collision_distances(m, x64, c.double(), t.double(), with_jacobian=True)
        _, J32 = G.env_collision_distances(m, x, c, t, with_jacobian=True)
        de.append(d), Je.append(J), Je32.append(J32)
    return dict(ds=ds, Js=Js, Js32=Js32.double(), de=torch.stack(de, 1), Je=torch.stack(Je, 1),
                Je32=torch.stack(Je32, 1).double())


# ------------------------------------------------------------------------------------------------------------------
# the per-waypoint fp64 assembly and its tolerances


W2 = 0.01 ** 2  # alpha_self_collision^2 = alpha_env_collision^2 of both parameter sets


def oracle_blocks(r, base_name, total, n_obst):
    """Collision part of the diagonal blocks: A = sum_active w^2 g g^T, b = -sum_active w^2 d g, with per-waypoint
    tolerances from per-term fp32 error bounds (distance TOL_D, gradient TOL_G_*), the masks of waypoints left out
    (sign band / ill-defined gradient) and the sensitivity of every waypoint (smallest active term / tolerance)."""
    m = R.get_model(r)
    o = oracle_terms(r, base_name, total)
    ns = n_static(m)
    ds, Js, Js32 = o["ds"], o["Js"], o["Js32"]
    de, Je, Je32 = (o["de"][:, :n_obst, ns:].flatten(1, 2), o["Je"][:, :n_obst, ns:].flatten(1, 2),
                    o["Je32"][:, :n_obst, ns:].flatten(1, 2))
    radii = torch.tensor([c.radius for c in m.capsules], dtype=torch.float64)[ns:].repeat(n_obst)
    d = torch.cat([ds, de], 1)
    J = torch.cat([Js, Je], 1)
    eg = torch.cat([torch.full((ds.shape[1],), TOL_G_SELF), torch.full((de.shape[1],), TOL_G_ENV)]).double()
    act = d < 0
    in_band = (d.abs() < SIGN_BAND).any(1)
    axis = de + radii
    axis_edge = (act[:, ds.shape[1]:] & (axis > 0) & (axis < AXIS_BAND)).any(1)
    parallel = (act & ((J - torch.cat([Js32, Je32], 1)).abs().amax(-1) > 0.25 * eg)).any(1)
    wJ = W2 * J * act[..., None]
    A = torch.einsum("nsi,nsj->nij", wJ, J)
    b = -(W2 * d[..., None] * J * act[..., None]).sum(1)
    # per entry: |w^2 (g_i g_j - g'_i g'_j)| <= w^2 ((|g_i| + |g_j|) eg + eg^2), |w^2 (d g_i - d' g'_i)| <= w^2 (|d| eg + TOL_D (|g_i| + eg))
    wa = W2 * act.double()
    u = torch.einsum("ns,nsi->ni", wa * eg, J.abs())
    tolA = u[:, :, None] + u[:, None, :] + (wa * eg ** 2).sum(1)[:, None, None]
    tolb = TOL_D * torch.einsum("ns,nsi->ni", wa, J.abs()) + (wa * (d.abs() * eg + TOL_D * eg)).sum(1)[:, None]
    # sensitivity: what dropping each active term (with a non-zero gradient) moves, against the tolerance of the entries
    # it moves; the smallest over the waypoint's terms
    n_idx, s_idx = torch.nonzero(act & (J.abs().amax(-1) > 1e-6), as_tuple=True)
    g = J[n_idx, s_idx]
    mv = ((W2 * g[:, :, None] * g[:, None, :]).abs() / tolA[n_idx]).flatten(1).amax(1)
    mv = torch.maximum(mv, (W2 * d[n_idx, s_idx, None] * g).abs().div(tolb[n_idx]).amax(1))
    sens = torch.full((x_n := d.shape[0],), float("inf"), dtype=torch.float64).scatter_reduce(0, n_idx, mv, "amin")
    has_term = torch.zeros(x_n, dtype=torch.bool)
    has_term[n_idx] = True
    return dict(A=A, b=b, tolA=tolA, tolb=tolb, in_band=in_band, axis_edge=axis_edge, parallel=parallel,
                has_term=has_term, sens=sens, n_active=act.sum(1))


def band_report(r, name, ob):
    excl = ob["in_band"] | ob["axis_edge"] | ob["parallel"]
    checked = ~excl
    with_terms = checked & ob["has_term"]
    insensitive = with_terms & (ob["sens"] < 10.0)
    rep = dict(waypoints=len(excl), sign_band=int(ob["in_band"].sum()), axis_band=int(ob["axis_edge"].sum()),
               near_parallel=int(ob["parallel"].sum()), excluded=int(excl.sum()), with_active_terms=int(with_terms.sum()),
               insensitive=int(insensitive.sum()))
    return checked, rep


BLOCK_P, BLOCK_T = 37, 160  # ragged path count (not a multiple of the 16-path groups), T in the hundreds
BLOCK_SCENES = ["crowded8", "rotated8", "rotated8[:OGRP]", "rotated8[:OGRP+1]", "degenerate"]


def _resolve(r, name):
    return name.replace("OGRP+1", str(ogrp(r) + 1)).replace("OGRP", str(ogrp(r)))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the scenes are not vacuous


@pytest.mark.parametrize("r", ROBOTS)
def test_scenes_are_not_vacuous(r):
    """Every obstacle of every scene is hit; the near-contact configurations land in their bands, on every obstacle,
    the second mask group included; the bands leave most waypoints checked and most checked terms are sensitive."""
    m = R.get_model(r)
    ns = n_static(m)
    for base in ("crowded8", "rotated8", "degenerate"):
        scene = SCENES[base](r)
        assert scene.n == (3 if base == "degenerate" else 8)
        nc = near_contacts(r, base)
        # landed: within 10 % of the target after rounding to float32, and outside the sign band
        assert ((nc["d"] - nc["target"]).abs() <= 0.1 * nc["target"].abs()).all(), (base, (nc["d"] - nc["target"]).abs().max())
        assert (nc["d"].abs() > SIGN_BAND).all()
        env = nc["kind_env"]
        assert set(nc["oidx"][env].tolist()) == set(range(scene.n)), base  # contacts on every obstacle
        assert (~env).sum() >= 6 * len(TARGETS)                              # and on self pairs
        assert (nc["cidx"][env] >= ns).all()
        # some contacts have a bound within 3 mm of tight: a cull 5 mm too tight loses them
        assert int(((nc["gap"] < 3e-3) & (nc["target"] < 0) & env).sum()) >= 3, base
        total = BLOCK_P * BLOCK_T
        o = oracle_terms(r, base, total)
        hit = (o["de"][:, :, ns:] < 0).any(2).any(0)
        assert bool(hit.all()), (base, hit)  # every obstacle is hit by a moving capsule
        if scene.n == 8:
            assert bool((o["de"][:, ogrp(r):, ns:] < 0).any()), "contacts in the second mask group"
        for name in BLOCK_SCENES:
            if not name.startswith(base):
                continue
            sc = scene_by_name(r, _resolve(r, name))
            ob = oracle_blocks(r, base, total, sc.n)
            checked, rep = band_report(r, sc.name, ob)
            assert rep["excluded"] <= MAX_EXCLUDED * rep["waypoints"], (sc.name, rep)
            assert rep["insensitive"] <= MAX_INSENSITIVE * rep["with_active_terms"], (sc.name, rep)
            assert rep["with_active_terms"] >= 0.1 * rep["waypoints"], (sc.name, rep)
    # the degenerate geometry is really there: capsule axes inside the box, parallel to the plate at q = 0
    sc = degenerate(r)
    q0 = zero_config(m)[None]
    c, t = sc.c64()
    assert int(((sc.cuboids[0][:3] == sc.cuboids[0][3:]).sum())) == 1 and float(sc.cuboids[1][0]) == float(sc.cuboids[1][3])
    radii = torch.tensor([cap.radius for cap in m.capsules], dtype=torch.float64)
    d_box = G.env_collision_distances(m, q0, c[2], t[2])[0]
    assert (d_box[:2] + radii[:2]).abs().max() == 0.0  # base and first link: axis inside, d = -radius
    assert float(G.env_collision_distances(m, q0, c[0], t[0]).min()) < 0


# ------------------------------------------------------------------------------------------------------------------
# GPU


@pytest.fixture(scope="module")
def robots():
    from cppflow_b200.robot import get_robot

    return {r: get_robot(r) for r in ROBOTS}


def _collision_only_params():
    from cppflow_b200.lm_hyper_parameters import OptimizationParameters

    return OptimizationParameters(alpha_self_collision=0.01, use_self_collisions=True, alpha_env_collision=0.01,
                                  use_env_collisions=True, use_pose=False, use_differencing=False,
                                  use_virtual_configs=False)


def _assemble(rob, pm, x, xv, P, T, scene):
    """cppflow_lm_full_assemble -> packed blocks [P, T, NW] (workspace layout [path / 16][t][k][path % 16] float4)"""
    from cppflow_b200 import ops, _lib

    lib = _lib.load()
    D = rob.ndof
    NT = D * (D + 1) // 2
    NW = (NT + D + 3) // 4 * 4
    ws = torch.full((lib.cppflow_lm_full_workspace_bytes(rob.robot_id, P, T) // 4,), float("nan"), device=DEV)
    tg = torch.zeros((T, 7), device=DEV)
    tg[:, 3] = 1.0
    prm = ops.make_params(pm)
    cu, tc, no = ops._obs(scene.ops_obstacles())
    xd, xvd = x.to(DEV), (xv.to(DEV) if xv is not None else None)
    _lib.check(lib.cppflow_lm_full_assemble(rob.robot_id, prm, _lib.ptr(xd), _lib.ptr(xvd), _lib.ptr(tg), P, T, cu, tc, no,
                                            _lib.ptr(ws), ws.numel() * 4, _lib.stream_ptr(DEV)))
    torch.cuda.synchronize()
    groups = (P + 15) // 16
    blk = ws[: groups * T * NW * 16].cpu().double().reshape(groups, T, NW // 4, 16, 4)
    return blk.permute(0, 3, 1, 2, 4).reshape(groups * 16, T, NW)[:P], NT


def _tri(D):
    return [(i, j) for i in range(D) for j in range(i + 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("r", ROBOTS)
@pytest.mark.parametrize("scene_name", BLOCK_SCENES)
def test_lm_assembly_blocks_vs_fp64(robots, r, scene_name):
    """Every (A_tt, b_t) block the assembly kernel writes, for P = 37 paths x T = 160 waypoints, against a per-waypoint
    fp64 assembly: first with only the collision terms on (A = lambda I + sum_active w^2 g g^T, b = -sum_active w^2 d g),
    then with ALT_LOSS_V2_1_DIFF (+ beta n_t, the differencing right-hand side and the virtual-config terms, xv = x)."""
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF

    m = R.get_model(r)
    rob = robots[r]
    D = m.ndof
    P, T = BLOCK_P, BLOCK_T
    name = _resolve(r, scene_name)
    base = name.split("[")[0]
    scene = scene_by_name(r, name)
    x, _ = waypoints(r, base, P * T)
    ob = oracle_blocks(r, base, P * T, scene.n)
    checked, rep = band_report(r, name, ob)
    assert rep["excluded"] <= MAX_EXCLUDED * rep["waypoints"], rep
    assert rep["insensitive"] <= MAX_INSENSITIVE * rep["with_active_terms"], rep
    tri = _tri(D)
    ti, tj = torch.tensor([i for i, _ in tri]), torch.tensor([j for _, j in tri])
    x64 = x.double().reshape(P, T, D)
    pm_diff = ALT_LOSS_V2_1_DIFF
    beta = torch.tensor([(pm_diff.alpha_differencing * (pm_diff.alpha_differencing_prismatic_scaling
                                                        if d in m.prismatic_joint_idxs else 1.0)) ** 2 for d in range(D)],
                        dtype=torch.float64)
    gamma2 = (pm_diff.alpha_virtual_configs * pm_diff.alpha_differencing) ** 2
    worst = {}
    for mode, pm in (("collision", _collision_only_params()), ("diff", pm_diff)):
        blk, NT = _assemble(rob, pm, x, x if mode == "diff" else None, P, T, scene)
        A_got = blk[..., :NT].reshape(P * T, NT)
        b_got = blk[..., NT:NT + D].reshape(P * T, D)
        A_ref = ob["A"] + pm.lm_lambda * torch.eye(D, dtype=torch.float64)
        b_ref = ob["b"].clone()
        if mode == "diff":
            w = L.angular_changes(x64.transpose(0, 1)).transpose(0, 1)  # [P, T-1, D] wrapped x[t+1] - x[t]
            z = torch.zeros((P, 1, D), dtype=torch.float64)
            dw = (torch.cat([w, z], 1) - torch.cat([z, w], 1)).reshape(P * T, D)
            nt = torch.full((P, T), 2.0, dtype=torch.float64)
            nt[:, 0] = nt[:, -1] = 1.0
            tt = torch.arange(T)
            virt = ((tt < pm.n_virtual_configs) | (tt >= T - pm.n_virtual_configs)).double().repeat(P)
            A_ref = A_ref + torch.diag_embed(beta * nt.reshape(-1, 1) + gamma2 * virt[:, None])
            b_ref = b_ref + beta * dw
            # a difference within rounding of +-pi may wrap either way in float32: leave such waypoints out
            near_pi = ((w.abs() - np.pi).abs() < 1e-5).any(-1)
            amb = torch.zeros((P, T), dtype=torch.bool)
            amb[:, 1:] |= near_pi
            amb[:, :-1] |= near_pi
            ok = checked & ~amb.reshape(-1)
        else:
            ok = checked
        A_ref = A_ref[:, ti, tj]
        # per-term bounds plus fp32 rounding of the accumulation
        tolA = ob["tolA"][:, ti, tj] + 1e-6 * A_ref.abs().amax(1, keepdim=True) + 1e-12
        tolb = ob["tolb"] + 1e-6 * b_ref.abs().amax(1, keepdim=True) + 1e-13
        rA = ((A_got - A_ref).abs() / tolA).amax(1)
        rb = ((b_got - b_ref).abs() / tolb).amax(1)
        ratio = torch.maximum(rA, rb)
        assert torch.isfinite(A_got).all() and torch.isfinite(b_got).all()
        bad = torch.nonzero(ok & (ratio > 1.0)).flatten()
        assert len(bad) == 0, (mode, name, f"{len(bad)} waypoints beyond tolerance, e.g. waypoint {int(bad[0])}: "
                               f"ratio {float(ratio[bad[0]]):.3g}, {int(ob['n_active'][bad[0]])} active terms")
        worst[mode] = float(ratio[ok].max())
    print(f"lm assembly {r} {name}: {rep}; worst error / tolerance: "
          + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))


# ---- the LM step on the new scenes


def _planted_paths(r, scene, P, T, seed):
    """P smooth paths of T waypoints with near-contact configurations (+-2e-4 / +-2e-3 m, on self pairs and on
    obstacles of both mask groups) and deep contacts with the last obstacle planted"""
    m, target, x0 = synthetic_problem(r, P, T, seed=seed)
    nc = near_contacts(r, "rotated8")
    big = nc["target"].abs() >= 2e-4
    env_hi = torch.nonzero(big & nc["kind_env"] & (nc["oidx"] >= ogrp(r))).flatten()
    env_lo = torch.nonzero(big & nc["kind_env"] & (nc["oidx"] < ogrp(r))).flatten()
    slf = torch.nonzero(big & ~nc["kind_env"]).flatten()
    cu, Tc = scene.c64()
    cand = random_configs(m, 4000, seed=seed + 1)
    deep = cand[G.env_collision_distances(m, cand.double(), cu[-1], Tc[-1]).min(dim=1).values < -0.01]
    x = x0.reshape(P, T, -1).clone()
    for p in range(P):
        for k, t in enumerate((3, 9, 14, 20, 26, 33)):
            src = (env_hi, env_lo, slf)[k % 3]
            x[p, t] = nc["x"][src[(p * 7 + k) % len(src)]]
        x[p, 17] = deep[p % len(deep)]
    return m, target, x.reshape(P * T, -1).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("r", ROBOTS)
def test_lm_step_vs_dense_oracle_on_crowded_scene(robots, r):
    """lm_full_step (ALT_LOSS_V2_1_DIFF) on rotated8 with near-contact and second-group contacts planted against the dense
    fp64 get_r_and_J + _lm_full_step: 1e-4 rad.  The fused and overlapped launches give the same bits; the segmented
    solve stays within the tolerance of test_segmented_solve_long_paths."""
    from cppflow_b200 import ops
    from cppflow_b200.lm_hyper_parameters import ALT_LOSS_V2_1_DIFF

    P, T = 4, 40
    rob = robots[r]
    scene = rotated8(r)
    m, target, x0 = _planted_paths(r, scene, P, T, seed=61)
    cu, Tc = scene.c64()
    # no waypoint in the sign band: the active set is unambiguous
    ds = G.self_collision_distances(m, x0.double())
    de = torch.stack([G.env_collision_distances(m, x0.double(), c, t) for c, t in zip(cu, Tc)], 1)
    assert ds.abs().min() > SIGN_BAND and de.abs().min() > SIGN_BAND
    n_hi = int((de[:, ogrp(r):, n_static(m):] < 0).any(-1).any(-1).sum())
    assert n_hi >= P
    prm = ops.make_params(ALT_LOSS_V2_1_DIFF)
    ob = scene.ops_obstacles()
    x, tg = x0.to(DEV), target.to(DEV)
    out = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, x, tg, P, T, ob, False)
    worst = 0.0
    for p in range(P):
        sl = slice(p * T, (p + 1) * T)
        xp = x0[sl].double()
        opms = L.LmParams(virtual_configs=xp.clone())
        Jd, rd = L.get_r_and_J(opms, m, xp, target.double(), Tc, cu)
        ref = L.lm_full_step(L.stack_rows(Jd), L.stack_rows(rd), xp, opms.lm_lambda)
        err = float((out[sl].cpu().double() - ref).abs().max())
        worst = max(worst, err)
        assert err < 1e-4, (p, err)
    for fused, overlap in ((True, False), (True, True), (False, True)):
        got = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, x, tg, P, T, ob, False, fused=fused, overlap=overlap)
        assert torch.equal(got, out), (fused, overlap)
    seg = ops.lm_full_step(rob.robot_id, rob.ndof, prm, x, x, tg, P, T, ob, False, segments=4)
    step = float((out - x).abs().max())
    assert float((seg - out).abs().max()) < 1e-4 + 1e-3 * step
    print(f"lm step {r} rotated8: max |dq| vs fp64 oracle = {worst:.2e} rad, {n_hi} waypoints touch the second mask group")


# ---- collision flags


FLAG_SCENES = ["crowded8", "rotated8", "degenerate", "rotated8[:0]", "rotated8[:1]", "rotated8[:OGRP]",
               "rotated8[:OGRP+1]"]


@pytest.mark.gpu
@pytest.mark.parametrize("r", ROBOTS)
@pytest.mark.parametrize("scene_name", FLAG_SCENES)
def test_collision_flags_vs_oracle_signs(robots, r, scene_name):
    """ops.collision_flags against the signs of the oracle's minimum distances, outside the sign band"""
    from cppflow_b200 import ops

    m = R.get_model(r)
    rob = robots[r]
    name = _resolve(r, scene_name)
    base = name.split("[")[0]
    scene = scene_by_name(r, name)
    total = BLOCK_P * BLOCK_T
    x, n_near = waypoints(r, base, total)
    o = oracle_terms(r, base, total)
    s, e = ops.collision_flags(rob.robot_id, rob.ndof, x.to(DEV), scene.ops_obstacles())
    s, e = s.cpu().bool(), e.cpu().bool()
    dmin_s = o["ds"].min(1).values
    dmin_e = o["de"][:, :scene.n].flatten(1).min(1).values if scene.n else torch.full((total,), float("inf"), dtype=torch.float64)
    for flag, dmin, what in ((s, dmin_s, "self"), (e, dmin_e, "env")):
        ok = dmin.abs() > SIGN_BAND
        assert ok.double().mean() > 1 - MAX_EXCLUDED
        wrong = torch.nonzero(ok & (flag != (dmin < 0))).flatten()
        assert len(wrong) == 0, (name, what, f"{len(wrong)} wrong flags, e.g. waypoint {int(wrong[0])}: "
                                 f"flag {bool(flag[wrong[0]])}, oracle min {float(dmin[wrong[0]]):.3g}")
    assert bool(s.any()) and not bool(s.all())
    if scene.n:
        assert bool(e.any()) and (base == "degenerate" or not bool(e.all()))
    else:
        assert not bool(e.any())


# ---- path metrics


def _metric_paths(r, P, T, seed):
    """P paths of T waypoints at least 1 cm clear of everything in rotated8, each with one near-contact waypoint (self or
    env, obstacle 7 included) where the path's minimum is attained"""
    m = R.get_model(r)
    scene = rotated8(r)
    cu, Tc = scene.c64()
    pool = random_configs(m, 8000, seed=seed)
    ds = G.self_collision_distances(m, pool.double()).min(1).values
    de = torch.stack([G.env_collision_distances(m, pool.double(), c, t).min(1).values for c, t in zip(cu, Tc)], 1).min(1).values
    clear = pool[(ds > 0.01) & (de > 0.01)]
    nc = near_contacts(r, "rotated8")
    g = torch.Generator().manual_seed(seed)
    x = clear[torch.randint(len(clear), (P, T), generator=g)]
    on7 = torch.nonzero(nc["kind_env"] & (nc["oidx"] == 7)).flatten()
    for p in range(P):
        k = on7[p % len(on7)] if p % 3 == 0 else (p * 11) % len(nc["x"])
        x[p, (p * 37) % T] = nc["x"][k]
    return m, x.reshape(P * T, -1).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("r", ROBOTS)
def test_path_metrics_minima_at_near_contact(robots, r):
    """Columns 5 / 6 (minimum self / env distance) of the exact metrics = the oracle's minimum to 1e-5 m, for the
    one-CTA-per-path launch (64 paths) and the cluster launch (one path); the sign-only variant is bit-identical where
    the exact minimum is negative, non-negative elsewhere, and bit-identical in columns 0-4."""
    from cppflow_b200 import ops

    rob = robots[r]
    P, T = 64, 300  # 64 x 5 cluster CTAs > 2 x 148: one CTA per path
    m, x = _metric_paths(r, P, T, seed=71)
    scene = rotated8(r)
    cu, Tc = scene.c64()
    x64 = x.double()
    ds = G.self_collision_distances(m, x64).min(1).values.reshape(P, T)
    de = torch.stack([G.env_collision_distances(m, x64, c, t).min(1).values for c, t in zip(cu, Tc)], 1).min(1).values.reshape(P, T)
    ref = torch.stack([ds.min(1).values, de.min(1).values], 1)
    assert int((ref < 0).any(1).sum()) >= P // 4 and int((ref >= 0).all(1).sum()) >= 4
    target = torch.zeros((T, 7))
    target[:, 3] = 1.0
    ob = scene.ops_obstacles()
    xd, td = x.to(DEV), target.to(DEV)
    many = ops.path_metrics(rob.robot_id, rob.ndof, xd, td, P, T, ob).cpu()
    err = (many[:, 5:7].double() - ref).abs()
    assert float(err.max()) < 1e-5, (float(err.max()), torch.nonzero(err > 1e-5)[:4].tolist())
    worst_one = 0.0
    for p in range(0, P, 5):
        one = ops.path_metrics(rob.robot_id, rob.ndof, xd[p * T:(p + 1) * T].contiguous(), td, 1, T, ob).cpu()[0]
        e1 = float((one[5:7].double() - ref[p]).abs().max())
        worst_one = max(worst_one, e1)
        assert e1 < 1e-5, (p, one[5:7], ref[p])
    sign = ops.path_metrics(rob.robot_id, rob.ndof, xd, td, P, T, ob, sign_only=True).cpu()
    assert torch.equal(sign[:, :5], many[:, :5])
    for k in (5, 6):
        neg = many[:, k] < 0
        assert torch.equal(sign[neg, k], many[neg, k])
        assert bool((sign[~neg, k] >= 0).all())
    print(f"path metrics {r}: max |min distance - oracle| = {float(err.max()):.2e} m (64 paths), {worst_one:.2e} m (cluster)")
