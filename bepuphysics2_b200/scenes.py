"""Seeded synthetic scenes for the BASELINE.json configs (SURVEY.md §8d).

The reference's collision detection cannot run here, so contact manifolds are synthesised directly in the prestep layouts the
narrow phase would write (Constraints/Contact/ContactConvexTypes.cs prestep structs), with the material the reference benchmarks use
(DemoBenchmarks/ShapePileBenchmark.cs:L54-66: SpringSettings(30 Hz, zeta 1), MaximumRecoveryVelocity 2, friction 1).
Every generator is a pure function of its arguments (numpy PCG64 with a fixed seed, default 5 like the reference's `new Random(5)`).

A scene is a dict: {"bodies": float32[n, 32] BodyDynamics records, "constraints": [(type_id, int32[m, bodies], float32[m, prestep])...],
"description": str}. `build(scene, ...)` adds it to a host `Simulation` in order, which assigns batches like Solver.Add does.
"""
import math

import numpy as np

TWO_PI = np.float32(6.283185307179586477)


def make_bodies(position, orientation=None, linear=None, angular=None, inverse_mass=None, inverse_inertia=None):
    """Packs BodyDynamics records (BepuPhysics/BodyProperties.cs:L11-46,L318-338): floats 0-3 orientation xyzw, 4-6 position, 8-10 linear,
    12-14 angular, 16-21 local inverse inertia (XX,YX,YY,ZX,ZY,ZZ), 22 inverse mass, 24-30 world inverse inertia + inverse mass (left zero)."""
    position = np.asarray(position, dtype=np.float32).reshape(-1, 3)
    n = position.shape[0]
    b = np.zeros((n, 32), dtype=np.float32)
    b[:, 3] = 1.0
    if orientation is not None:
        b[:, 0:4] = np.asarray(orientation, dtype=np.float32).reshape(n, 4)
    b[:, 4:7] = position
    if linear is not None:
        b[:, 8:11] = np.asarray(linear, dtype=np.float32).reshape(n, 3)
    if angular is not None:
        b[:, 12:15] = np.asarray(angular, dtype=np.float32).reshape(n, 3)
    if inverse_inertia is not None:
        b[:, 16:22] = np.asarray(inverse_inertia, dtype=np.float32).reshape(n, 6)
    if inverse_mass is not None:
        b[:, 22] = np.asarray(inverse_mass, dtype=np.float32).reshape(n)
    return b


def spring(frequency_hz, damping_ratio):
    """SpringSettings(frequency, dampingRatio) -> (AngularFrequency, TwiceDampingRatio) (Constraints/SpringSettings.cs:L75-80)."""
    return np.float32(frequency_hz) * TWO_PI, np.float32(damping_ratio) * np.float32(2)


def convex_prestep(offsets_a, depths, normal, offset_b=None, friction=1.0, spring_settings=None, max_recovery=2.0):
    """Rows of Contact{N}[OneBody]PrestepData: [OffsetA xyz, Depth] x N, (OffsetB xyz), Normal xyz, FrictionCoefficient, AngularFrequency,
    TwiceDampingRatio, MaximumRecoveryVelocity. offsets_a: [m, N, 3], depths: [m, N], normal: [m, 3], offset_b: [m, 3] or None (one body)."""
    offsets_a = np.asarray(offsets_a, dtype=np.float32)
    m, N, _ = offsets_a.shape
    af, tdr = spring_settings if spring_settings is not None else spring(30, 1)
    cols = []
    for i in range(N):
        cols.append(offsets_a[:, i, :])
        cols.append(np.asarray(depths, dtype=np.float32)[:, i : i + 1])
    if offset_b is not None:
        cols.append(np.asarray(offset_b, dtype=np.float32).reshape(m, 3))
    cols.append(np.asarray(normal, dtype=np.float32).reshape(m, 3))
    mat = np.empty((m, 4), dtype=np.float32)
    mat[:, 0], mat[:, 1], mat[:, 2], mat[:, 3] = friction, af, tdr, max_recovery
    cols.append(mat)
    return np.ascontiguousarray(np.concatenate(cols, axis=1), dtype=np.float32)


def nonconvex_prestep(offsets, depths, normals, offset_b=None, friction=1.0, spring_settings=None, max_recovery=2.0):
    """Rows of Contact{N}Nonconvex[OneBody]PrestepData: material (4), (OffsetB xyz), [Offset xyz, Depth, Normal xyz] x N."""
    offsets = np.asarray(offsets, dtype=np.float32)
    m, N, _ = offsets.shape
    af, tdr = spring_settings if spring_settings is not None else spring(30, 1)
    mat = np.empty((m, 4), dtype=np.float32)
    mat[:, 0], mat[:, 1], mat[:, 2], mat[:, 3] = friction, af, tdr, max_recovery
    cols = [mat]
    if offset_b is not None:
        cols.append(np.asarray(offset_b, dtype=np.float32).reshape(m, 3))
    for i in range(N):
        cols.append(offsets[:, i, :])
        cols.append(np.asarray(depths, dtype=np.float32)[:, i : i + 1])
        cols.append(np.asarray(normals, dtype=np.float32)[:, i, :])
    return np.ascontiguousarray(np.concatenate(cols, axis=1), dtype=np.float32)


CONVEX_ONE_BODY = {1: 0, 2: 1, 3: 2, 4: 3}
CONVEX_TWO_BODY = {1: 4, 2: 5, 3: 6, 4: 7}
NONCONVEX_ONE_BODY = {2: 8, 3: 9, 4: 10}
NONCONVEX_TWO_BODY = {2: 15, 3: 16, 4: 17}


def box_stacks(columns=16, height=16, penetration=0.01):
    """Config 1 (plumbing): `columns` stacks of `height` unit boxes (mass 1, inverse inertia diag 6) on one kinematic ground body.
    One Contact4 (type 7) per box: 4 corner contacts against the body below, normal (0,1,0), depth `penetration`."""
    n = columns * height
    pos = np.zeros((n + 1, 3), dtype=np.float32)
    pos[0] = (0, -0.5, 0)  # ground slab, top face at y = 0
    spacing = 1.0 - penetration
    idx = 1
    handles_a, handles_b = [], []
    for c in range(columns):
        for i in range(height):
            pos[idx] = (3.0 * c, 0.5 - penetration + i * spacing, 0.0)
            handles_a.append(idx)
            handles_b.append(idx - 1 if i > 0 else 0)
            idx += 1
    inv_mass = np.ones(n + 1, dtype=np.float32)
    inv_inertia = np.zeros((n + 1, 6), dtype=np.float32)
    inv_inertia[:, 0] = inv_inertia[:, 2] = inv_inertia[:, 5] = 6.0
    inv_mass[0] = 0
    inv_inertia[0] = 0
    bodies = make_bodies(pos, inverse_mass=inv_mass, inverse_inertia=inv_inertia)
    a = np.asarray(handles_a, dtype=np.int32)
    b = np.asarray(handles_b, dtype=np.int32)
    corners = np.array([[-0.5, -0.5, -0.5], [0.5, -0.5, -0.5], [-0.5, -0.5, 0.5], [0.5, -0.5, 0.5]], dtype=np.float32)
    offsets = np.broadcast_to(corners, (n, 4, 3)).copy()
    depths = np.full((n, 4), penetration, dtype=np.float32)
    normal = np.broadcast_to(np.array([0, 1, 0], dtype=np.float32), (n, 3))
    offset_b = pos[b] - pos[a]
    pre = convex_prestep(offsets, depths, normal, offset_b)
    return {"bodies": bodies, "constraints": [(7, np.stack([a, b], axis=1), pre)], "description": "%d columns x %d unit boxes, Contact4 only" % (columns, height)}


# ShapePileBenchmark shapes (DemoBenchmarks/ShapePileBenchmark.cs:L109-164), mass 1: local inverse inertia diagonals.
def _shape_inverse_inertias():
    def inv(ixx, iyy, izz):
        return np.array([1.0 / ixx, 0, 1.0 / iyy, 0, 0, 1.0 / izz], dtype=np.float32)

    r = 1.5
    sphere = inv(0.4 * r * r, 0.4 * r * r, 0.4 * r * r)
    # capsule radius 1, length 1 (axis y): approximate as cylinder + two hemispheres by volume-weighted mass split
    cr, cl = 1.0, 1.0
    vc, vs = math.pi * cr * cr * cl, 4.0 / 3.0 * math.pi * cr ** 3
    mc, ms = vc / (vc + vs), vs / (vc + vs)
    iyy = mc * 0.5 * cr * cr + ms * 0.4 * cr * cr
    ixx = mc * (cl * cl / 12.0 + cr * cr / 4.0) + ms * (0.4 * cr * cr + cl * cl / 4.0 + 3.0 * cl * cr / 8.0)
    capsule = inv(ixx, iyy, ixx)
    w, h, d = 1.0, 3.0, 2.0
    box = inv((h * h + d * d) / 12.0, (w * w + d * d) / 12.0, (w * w + h * h) / 12.0)
    cyr, cyl = 1.5, 0.3
    cylinder = inv(cyl * cyl / 12.0 + cyr * cyr / 4.0, 0.5 * cyr * cyr, cyl * cyl / 12.0 + cyr * cyr / 4.0)
    hull = inv(0.39, 0.39, 0.39)  # dodecahedron-ish hull, a little lighter in rotation than the unit sphere
    return np.stack([sphere, capsule, box, cylinder, hull])


_NEIGHBOR_OFFSETS = np.array(
    [(1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (1, -1, 0), (1, 0, 1), (1, 0, -1), (0, 1, 1), (0, 1, -1), (1, 1, 1), (1, 1, -1), (1, -1, 1), (1, -1, -1)],
    dtype=np.int64,
)


def _random_unit_quaternions(rng, n):
    q = rng.standard_normal((n, 4)).astype(np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True).astype(np.float32)
    return q.astype(np.float32)


def _tangent_frame(normal):
    ref = np.where(np.abs(normal[:, 0:1]) < 0.7, np.array([[1, 0, 0]], dtype=np.float32), np.array([[0, 1, 0]], dtype=np.float32))
    t1 = np.cross(normal, ref)
    t1 /= np.linalg.norm(t1, axis=1, keepdims=True)
    t2 = np.cross(normal, t1)
    return t1.astype(np.float32), t2.astype(np.float32)


def shape_pile(body_count=100_000, manifolds_per_body=3.5, one_body_fraction=0.10, seed=5, dims=None, nonconvex_fraction=0.0):
    """Config 2/4: a settled-pile contact graph on a jittered 3-D lattice. Bodies are the five ShapePileBenchmark shapes (mass 1) at random
    orientations; each body touches lattice neighbours (13 forward directions) with the probability that yields `manifolds_per_body`
    constraints per body; manifold contact counts are drawn {1: 15%, 2: 25%, 3: 15%, 4: 45%}; `one_body_fraction` of the manifolds are against
    the static world (one-body types 0-3). Optionally a fraction of the multi-contact manifolds use the nonconvex types (8-10, 15-17)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    if dims is None:
        ny = max(4, int(round((body_count / 100.0) ** (1.0 / 3.0) * 2.15)))  # 100k -> 100 x 10 x 100
        nx = int(math.ceil(math.sqrt(body_count / ny)))
        nz = int(math.ceil(body_count / (nx * ny)))
    else:
        nx, ny, nz = dims
    n = body_count
    ids = np.arange(n, dtype=np.int64)
    gx, gy, gz = ids % nx, (ids // nx) % ny, ids // (nx * ny)
    spacing = 2.0
    pos = np.stack([gx, gy, gz], axis=1).astype(np.float32) * np.float32(spacing)
    pos += rng.uniform(-0.25, 0.25, size=(n, 3)).astype(np.float32)
    shape = rng.integers(0, 5, size=n)
    inv_inertia = _shape_inverse_inertias()[shape]
    bodies = make_bodies(
        pos,
        orientation=_random_unit_quaternions(rng, n),
        linear=rng.uniform(-0.3, 0.3, size=(n, 3)).astype(np.float32),
        angular=rng.uniform(-0.3, 0.3, size=(n, 3)).astype(np.float32),
        inverse_mass=np.ones(n, dtype=np.float32),
        inverse_inertia=inv_inertia,
    )
    two_body_target = manifolds_per_body * (1.0 - one_body_fraction)
    p_pair = min(1.0, two_body_target / len(_NEIGHBOR_OFFSETS))
    pairs_a, pairs_b = [], []
    for off in _NEIGHBOR_OFFSETS:
        ox, oy, oz = gx + off[0], gy + off[1], gz + off[2]
        valid = (ox >= 0) & (ox < nx) & (oy >= 0) & (oy < ny) & (oz >= 0) & (oz < nz)
        other = ox + oy * nx + oz * nx * ny
        valid &= other < n
        valid &= rng.random(n) < p_pair
        pairs_a.append(ids[valid])
        pairs_b.append(other[valid])
    a = np.concatenate(pairs_a)
    b = np.concatenate(pairs_b)
    order = np.argsort(a, kind="stable")  # narrow-phase-like order: by first body
    a, b = a[order].astype(np.int32), b[order].astype(np.int32)
    m2 = a.shape[0]
    m1 = int(round(n * manifolds_per_body * one_body_fraction))
    one_a = np.sort(rng.choice(n, size=m1, replace=m1 > n)).astype(np.int32)

    def manifold_geometry(count, pa, pb):
        counts = rng.choice(np.array([1, 2, 3, 4]), size=count, p=[0.15, 0.25, 0.15, 0.45])
        if pb is not None:
            d = pa - pb
            normal = d / np.linalg.norm(d, axis=1, keepdims=True)
            mid = 0.5 * (pa + pb)
        else:
            normal = np.tile(np.array([[0, 1, 0]], dtype=np.float32), (count, 1))
            mid = pa - normal * np.float32(0.9)
        normal = normal + rng.normal(0, 0.05, size=(count, 3)).astype(np.float32)
        normal = (normal / np.linalg.norm(normal, axis=1, keepdims=True)).astype(np.float32)
        t1, t2 = _tangent_frame(normal)
        ang = rng.uniform(0, 2 * math.pi, size=(count, 1)).astype(np.float32) + np.arange(4, dtype=np.float32)[None, :] * np.float32(math.pi / 2)
        rad = rng.uniform(0.15, 0.45, size=(count, 4)).astype(np.float32)
        pts = mid[:, None, :] + (np.cos(ang) * rad)[:, :, None] * t1[:, None, :] + (np.sin(ang) * rad)[:, :, None] * t2[:, None, :]
        offsets = (pts - pa[:, None, :]).astype(np.float32)
        depths = rng.uniform(-0.02, 0.05, size=(count, 4)).astype(np.float32)
        return counts, normal, offsets, depths

    constraints = []
    pa, pb = pos[a], pos[b]
    counts, normal, offsets, depths = manifold_geometry(m2, pa, pb)
    noncv = rng.random(m2) < nonconvex_fraction
    for N in (1, 2, 3, 4):
        sel = (counts == N) & ~(noncv & (N > 1))
        if sel.any():
            pre = convex_prestep(offsets[sel][:, :N], depths[sel][:, :N], normal[sel], (pb - pa)[sel])
            constraints.append((CONVEX_TWO_BODY[N], np.stack([a[sel], b[sel]], axis=1), pre))
        sel = (counts == N) & noncv & (N > 1)
        if N > 1 and sel.any():
            k = int(sel.sum())
            normals = normal[sel][:, None, :] + rng.normal(0, 0.03, size=(k, N, 3)).astype(np.float32)
            normals = (normals / np.linalg.norm(normals, axis=2, keepdims=True)).astype(np.float32)
            pre = nonconvex_prestep(offsets[sel][:, :N], depths[sel][:, :N], normals, (pb - pa)[sel])
            constraints.append((NONCONVEX_TWO_BODY[N], np.stack([a[sel], b[sel]], axis=1), pre))
    if m1 > 0:
        pa1 = pos[one_a]
        counts, normal, offsets, depths = manifold_geometry(m1, pa1, None)
        noncv = rng.random(m1) < nonconvex_fraction
        for N in (1, 2, 3, 4):
            sel = (counts == N) & ~(noncv & (N > 1))
            if sel.any():
                pre = convex_prestep(offsets[sel][:, :N], depths[sel][:, :N], normal[sel], None)
                constraints.append((CONVEX_ONE_BODY[N], one_a[sel].reshape(-1, 1), pre))
            sel = (counts == N) & noncv & (N > 1)
            if N > 1 and sel.any():
                k = int(sel.sum())
                normals = normal[sel][:, None, :] + rng.normal(0, 0.03, size=(k, N, 3)).astype(np.float32)
                normals = (normals / np.linalg.norm(normals, axis=2, keepdims=True)).astype(np.float32)
                pre = nonconvex_prestep(offsets[sel][:, :N], depths[sel][:, :N], normals, None)
                constraints.append((NONCONVEX_ONE_BODY[N], one_a[sel].reshape(-1, 1), pre))
    total = sum(c[1].shape[0] for c in constraints)
    return {
        "bodies": bodies,
        "constraints": constraints,
        "description": "shape pile: %d bodies on a %dx%dx%d jittered lattice, %d contact manifolds (types 0-7%s)" % (n, nx, ny, nz, total, ", 8-10, 15-17" if nonconvex_fraction > 0 else ""),
    }


def fallback_stress(body_count=50_000, hubs=50, seed=5, neighbour_manifolds_per_body=1.0):
    """Config 5: every body touches one of a few dynamic hub bodies, so hubs exceed FallbackBatchThreshold constraints and most constraints
    land in the sequential fallback batch; plus ordinary neighbour contacts."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n = body_count
    pos = rng.uniform(-50, 50, size=(n, 3)).astype(np.float32)
    inv_inertia = _shape_inverse_inertias()[rng.integers(0, 5, size=n)]
    inv_mass = np.ones(n, dtype=np.float32)
    inv_mass[:hubs] = 0.01  # heavy hubs
    inv_inertia[:hubs] *= 0.01
    bodies = make_bodies(pos, orientation=_random_unit_quaternions(rng, n), linear=rng.uniform(-0.3, 0.3, size=(n, 3)).astype(np.float32),
                         angular=rng.uniform(-0.3, 0.3, size=(n, 3)).astype(np.float32), inverse_mass=inv_mass, inverse_inertia=inv_inertia)
    others = np.arange(hubs, n, dtype=np.int32)
    hub_of = (rng.integers(0, hubs, size=others.shape[0])).astype(np.int32)
    constraints = []

    def add_pairs(a, b, label_rng):
        m = a.shape[0]
        counts = label_rng.choice(np.array([1, 2, 3, 4]), size=m, p=[0.15, 0.25, 0.15, 0.45])
        d = pos[a] - pos[b]
        normal = (d / np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-3)).astype(np.float32)
        t1, t2 = _tangent_frame(normal)
        ang = label_rng.uniform(0, 2 * math.pi, size=(m, 1)).astype(np.float32) + np.arange(4, dtype=np.float32)[None, :] * np.float32(math.pi / 2)
        rad = label_rng.uniform(0.15, 0.45, size=(m, 4)).astype(np.float32)
        offs = (-normal * np.float32(0.9))[:, None, :] + (np.cos(ang) * rad)[:, :, None] * t1[:, None, :] + (np.sin(ang) * rad)[:, :, None] * t2[:, None, :]
        depths = label_rng.uniform(-0.02, 0.05, size=(m, 4)).astype(np.float32)
        offset_b = (-normal * np.float32(1.8)).astype(np.float32)
        for N in (1, 2, 3, 4):
            sel = counts == N
            if sel.any():
                constraints.append((CONVEX_TWO_BODY[N], np.stack([a[sel], b[sel]], axis=1), convex_prestep(offs[sel][:, :N].astype(np.float32), depths[sel][:, :N], normal[sel], offset_b[sel])))

    add_pairs(others, hub_of, rng)
    k = int(round(n * neighbour_manifolds_per_body))
    na = rng.integers(hubs, n, size=k).astype(np.int32)
    nb_ = rng.integers(hubs, n, size=k).astype(np.int32)
    keep = na != nb_
    add_pairs(na[keep], nb_[keep], rng)
    total = sum(c[1].shape[0] for c in constraints)
    return {"bodies": bodies, "constraints": constraints, "description": "fallback stress: %d bodies, %d hubs, %d manifolds" % (n, hubs, total)}


# ---- quaternion helpers in the reference's conventions (BepuUtilities/QuaternionEx.cs) ----
def qcat(a, b):
    """QuaternionEx.Concatenate(a, b): the rotation a followed by the rotation b. Arrays [..., 4] as xyzw."""
    ax, ay, az, aw = a[..., 0], a[..., 1], a[..., 2], a[..., 3]
    bx, by, bz, bw = b[..., 0], b[..., 1], b[..., 2], b[..., 3]
    return np.stack([aw * bx + ax * bw + az * by - ay * bz, aw * by + ay * bw + ax * bz - az * bx, aw * bz + az * bw + ay * bx - ax * by,
                     aw * bw - ax * bx - ay * by - az * bz], axis=-1).astype(np.float32)


def qconj(q):
    return (q * np.array([-1, -1, -1, 1], dtype=np.float32)).astype(np.float32)


def qrot(v, q):
    """QuaternionEx.Transform(v, q)."""
    u = q[..., :3]
    w = q[..., 3:4]
    t = 2.0 * np.cross(u, v)
    return (v + w * t + np.cross(u, t)).astype(np.float32)


def basis_quaternion(z, x):
    """RagdollDemo.CreateBasis(z, x) (Demos/Demos/RagdollDemo.cs:L183-192): quaternion whose local Z maps to z and local X towards x."""
    z = np.asarray(z, dtype=np.float64)
    x = np.asarray(x, dtype=np.float64)
    bz = z / np.linalg.norm(z)
    by = np.cross(bz, x)
    by /= np.linalg.norm(by)
    bx = np.cross(by, bz)
    m = np.stack([bx, by, bz], axis=1)  # columns = images of the unit axes
    tr = m[0, 0] + m[1, 1] + m[2, 2]
    if tr > 0:
        s = math.sqrt(tr + 1.0) * 2
        q = [(m[2, 1] - m[1, 2]) / s, (m[0, 2] - m[2, 0]) / s, (m[1, 0] - m[0, 1]) / s, 0.25 * s]
    elif m[0, 0] > m[1, 1] and m[0, 0] > m[2, 2]:
        s = math.sqrt(1.0 + m[0, 0] - m[1, 1] - m[2, 2]) * 2
        q = [0.25 * s, (m[0, 1] + m[1, 0]) / s, (m[0, 2] + m[2, 0]) / s, (m[2, 1] - m[1, 2]) / s]
    elif m[1, 1] > m[2, 2]:
        s = math.sqrt(1.0 + m[1, 1] - m[0, 0] - m[2, 2]) * 2
        q = [(m[0, 1] + m[1, 0]) / s, 0.25 * s, (m[1, 2] + m[2, 1]) / s, (m[0, 2] - m[2, 0]) / s]
    else:
        s = math.sqrt(1.0 + m[2, 2] - m[0, 0] - m[1, 1]) * 2
        q = [(m[0, 2] + m[2, 0]) / s, (m[1, 2] + m[2, 1]) / s, 0.25 * s, (m[1, 0] - m[0, 1]) / s]
    return np.asarray(q, dtype=np.float32)


# Ragdoll skeleton (Demos/Demos/RagdollDemo.cs:L428-545 AddRagdoll): 16 bodies, 15 connections, 58 joints =
# 11 BallSocket + 15 SwingLimit + 9 TwistLimit + 4 TwistServo + 2 SwivelHinge + 2 Hinge + 15 AngularMotor.
# (name, local position, half extents used for the inertia box, mass)
_RAGDOLL_BODIES = [
    ("hips", (0, 1.1, 0), (0.2, 0.1, 0.12), 8), ("abdomen", (0, 1.3, 0), (0.18, 0.1, 0.11), 7), ("chest", (0, 1.6, 0), (0.22, 0.18, 0.13), 10), ("head", (0, 1.95, 0), (0.1, 0.12, 0.1), 5),
    ("upper_arm_r", (0.45, 1.7, 0), (0.225, 0.1, 0.1), 5), ("lower_arm_r", (0.9, 1.7, 0), (0.225, 0.09, 0.09), 5), ("hand_r", (1.225, 1.7, 0), (0.1, 0.05, 0.1), 2),
    ("upper_arm_l", (-0.45, 1.7, 0), (0.225, 0.1, 0.1), 5), ("lower_arm_l", (-0.9, 1.7, 0), (0.225, 0.09, 0.09), 5), ("hand_l", (-1.225, 1.7, 0), (0.1, 0.05, 0.1), 2),
    ("upper_leg_r", (0.15, 0.8, 0), (0.12, 0.25, 0.12), 5), ("lower_leg_r", (0.15, 0.3, 0), (0.11, 0.25, 0.11), 5), ("foot_r", (0.15, -0.025, 0.05), (0.1, 0.075, 0.15), 2),
    ("upper_leg_l", (-0.15, 0.8, 0), (0.12, 0.25, 0.12), 5), ("lower_leg_l", (-0.15, 0.3, 0), (0.11, 0.25, 0.11), 5), ("foot_l", (-0.15, -0.025, 0.05), (0.1, 0.075, 0.15), 2),
]
# (body a, body b, anchor, position joint, twist joint, swing axis, max swing angle, twist axis)
_RAGDOLL_CONNECTIONS = [
    (0, 1, (0, 1.2, 0), "ball", "limit", (0, 1, 0), 0.25 * math.pi, (0, 1, 0)), (1, 2, (0, 1.4, 0), "ball", "limit", (0, 1, 0), 0.25 * math.pi, (0, 1, 0)),
    (2, 3, (0, 1.8, 0), "ball", "limit", (0, 1, 0), 0.35 * math.pi, (0, 1, 0)),
    (2, 4, (0.225, 1.7, 0), "ball", "limit", (1, 0, 0), 0.56 * math.pi, (1, 0, 0)), (4, 5, (0.675, 1.7, 0), "swivel", "limit", (1, 0, 0), 0.5 * math.pi, (1, 0, 0)),
    (5, 6, (1.125, 1.7, 0), "ball", "servo", (1, 0, 0), 0.5 * math.pi, (1, 0, 0)),
    (2, 7, (-0.225, 1.7, 0), "ball", "limit", (-1, 0, 0), 0.56 * math.pi, (-1, 0, 0)), (7, 8, (-0.675, 1.7, 0), "swivel", "limit", (-1, 0, 0), 0.5 * math.pi, (-1, 0, 0)),
    (8, 9, (-1.125, 1.7, 0), "ball", "servo", (-1, 0, 0), 0.5 * math.pi, (-1, 0, 0)),
    (0, 10, (0.15, 1.05, 0), "ball", "limit", (0, -1, 0), 0.45 * math.pi, (0, -1, 0)), (10, 11, (0.15, 0.55, 0), "hinge", None, (0, -1, 0), 0.5 * math.pi, (0, -1, 0)),
    (11, 12, (0.15, 0.05, 0), "ball", "servo", (0, -1, 0), 0.3 * math.pi, (0, -1, 0)),
    (0, 13, (-0.15, 1.05, 0), "ball", "limit", (0, -1, 0), 0.45 * math.pi, (0, -1, 0)), (13, 14, (-0.15, 0.55, 0), "hinge", None, (0, -1, 0), 0.5 * math.pi, (0, -1, 0)),
    (14, 15, (-0.15, 0.05, 0), "ball", "servo", (0, -1, 0), 0.3 * math.pi, (0, -1, 0)),
]


def ragdolls(count=10_000, seed=5, contacts_per_body=2.0, motor="motor", spacing=2.5, pose_noise=0.15):
    """Config 3: `count` ragdolls with the RagdollDemo.AddRagdoll joint topology at random poses in a kinematic rotating tube, joint springs
    SpringSettings(15 Hz, 1) (RagdollDemo.cs:L443), AngularMotor settings MotorSettings(float.MaxValue, 0.01) (L200) or, with motor="servo", the
    AngularServo variant the demo comments mention (L199). Plus `contacts_per_body` contact manifolds per body: against the kinematic tube
    (two-body contacts with a kinematic B, tube material spring 10 Hz / friction 2, RagdollTubeDemo.cs:L29) and against other ragdolls."""
    rng = np.random.Generator(np.random.PCG64(seed))
    nb = len(_RAGDOLL_BODIES)
    n = count * nb + 1  # + the kinematic tube (body 0)
    local_pos = np.array([b[1] for b in _RAGDOLL_BODIES], dtype=np.float32)
    half = np.array([b[2] for b in _RAGDOLL_BODIES], dtype=np.float32)
    mass = np.array([b[3] for b in _RAGDOLL_BODIES], dtype=np.float32)
    # box inertia about the body's own axes; bodies are axis aligned in the ragdoll frame, so the body orientation is the ragdoll's
    full = 2 * half
    ixx = mass / 12 * (full[:, 1] ** 2 + full[:, 2] ** 2)
    iyy = mass / 12 * (full[:, 0] ** 2 + full[:, 2] ** 2)
    izz = mass / 12 * (full[:, 0] ** 2 + full[:, 1] ** 2)
    inv_inertia_local = np.zeros((nb, 6), dtype=np.float32)
    inv_inertia_local[:, 0], inv_inertia_local[:, 2], inv_inertia_local[:, 5] = 1 / ixx, 1 / iyy, 1 / izz
    side = int(math.ceil(count ** (1.0 / 3.0)))
    rid = np.arange(count)
    base = np.stack([rid % side, (rid // side) % side, rid // (side * side)], axis=1).astype(np.float32) * np.float32(spacing)
    base += rng.uniform(-0.2, 0.2, size=(count, 3)).astype(np.float32)
    rq = _random_unit_quaternions(rng, count)
    pos = base[:, None, :] + qrot(np.broadcast_to(local_pos, (count, nb, 3)), rq[:, None, :])
    orient = np.broadcast_to(rq[:, None, :], (count, nb, 4))
    if pose_noise > 0:
        # ragdolls in motion, not in their exact rest pose: every body is rotated a little about a random axis (rest pose makes the twist/servo angle
        # measurements sit exactly on acos(1), where the reference's formulation is numerically ill-conditioned)
        axis = rng.standard_normal((count, nb, 3)).astype(np.float32)
        axis /= np.linalg.norm(axis, axis=2, keepdims=True)
        half = (rng.uniform(-pose_noise, pose_noise, size=(count, nb, 1)) * 0.5).astype(np.float32)
        dq = np.concatenate([axis * np.sin(half), np.cos(half)], axis=2).astype(np.float32)
        orient = qcat(dq, orient)
    lin = rng.uniform(-0.5, 0.5, size=(count, 1, 3)).astype(np.float32) + rng.uniform(-0.2, 0.2, size=(count, nb, 3)).astype(np.float32)
    ang = rng.uniform(-0.5, 0.5, size=(count, nb, 3)).astype(np.float32)
    bodies = np.zeros((n, 32), dtype=np.float32)
    bodies[0] = make_bodies(np.array([[0, 0, 0]], dtype=np.float32), angular=np.array([[0, 0, 0.25]], dtype=np.float32))[0]  # kinematic tube, rotating
    bodies[1:] = make_bodies(pos.reshape(-1, 3), orientation=orient.reshape(-1, 4), linear=lin.reshape(-1, 3), angular=ang.reshape(-1, 3),
                             inverse_mass=np.broadcast_to(1 / mass, (count, nb)).reshape(-1), inverse_inertia=np.broadcast_to(inv_inertia_local, (count, nb, 6)).reshape(-1, 6))
    handle = 1 + rid[:, None] * nb + np.arange(nb)[None, :]  # [count, nb]
    joint_spring = spring(15, 1)
    fmax = np.float32(np.finfo(np.float32).max)
    per_type = {22: [], 25: [], 26: [], 27: [], 29: [], 30: [], 46: [], 47: []}

    def add(type_id, a, b, row):
        row = np.asarray(row, dtype=np.float32)
        per_type[type_id].append((handle[:, a], handle[:, b], np.broadcast_to(row, (count, row.shape[0]))))

    ident = np.array([0, 0, 0, 1], dtype=np.float32)
    for a, b, anchor, pos_joint, twist, swing_axis, swing_angle, twist_axis in _RAGDOLL_CONNECTIONS:
        anchor = np.asarray(anchor, dtype=np.float32)
        off_a, off_b = anchor - local_pos[a], anchor - local_pos[b]  # bodies share the ragdoll frame, so local offsets are frame offsets
        if pos_joint == "ball":
            add(22, a, b, np.r_[off_a, off_b, joint_spring])
        elif pos_joint == "swivel":
            add(46, a, b, np.r_[off_a, np.asarray(twist_axis, np.float32), off_b, [0, 1, 0], joint_spring])
        else:
            add(47, a, b, np.r_[off_a, [1, 0, 0], off_b, [1, 0, 0], joint_spring])
        add(25, a, b, np.r_[np.asarray(swing_axis, np.float32), np.asarray(swing_axis, np.float32), [math.cos(swing_angle)], joint_spring])
        tz = np.asarray(twist_axis, dtype=np.float32)
        tx = np.array([0, 0, -1], dtype=np.float32)
        basis = basis_quaternion(tz, tx)
        if twist == "limit":
            add(27, a, b, np.r_[basis, basis, [-0.55 * math.pi, 0.55 * math.pi], joint_spring])
        elif twist == "servo":
            add(26, a, b, np.r_[basis, basis, [0.0], joint_spring, [fmax, 0.0, fmax]])
        if motor == "servo":
            add(29, a, b, np.r_[ident, joint_spring, [fmax, 0.0, fmax]])
        else:
            add(30, a, b, np.r_[[0, 0, 0], [fmax, 100.0]])
    # Interleave like AddRagdoll does (all joints of ragdoll 0, then ragdoll 1, ...) is what the reference's batching would see; adding type by type
    # is equally valid input and keeps generation vectorised. Constraints of one type are ordered by ragdoll, then connection.
    constraints = []
    for type_id, items in per_type.items():
        if not items:
            continue
        ha = np.stack([i[0] for i in items], axis=1).reshape(-1)
        hb = np.stack([i[1] for i in items], axis=1).reshape(-1)
        pre = np.stack([i[2] for i in items], axis=1).reshape(ha.shape[0], -1)
        constraints.append((type_id, np.stack([ha, hb], axis=1).astype(np.int32), np.ascontiguousarray(pre, dtype=np.float32)))
    # contacts
    body_pos = bodies[1:, 4:7]
    total_dyn = count * nb
    m = int(round(total_dyn * contacts_per_body))
    m_tube = m // 2
    m_pair = m - m_tube
    tube_spring = spring(10, 1)

    def geometry(k, pa, normal):
        counts = rng.choice(np.array([1, 2, 3, 4]), size=k, p=[0.3, 0.3, 0.1, 0.3])
        t1, t2 = _tangent_frame(normal)
        ang_ = rng.uniform(0, 2 * math.pi, size=(k, 1)).astype(np.float32) + np.arange(4, dtype=np.float32)[None, :] * np.float32(math.pi / 2)
        rad = rng.uniform(0.02, 0.08, size=(k, 4)).astype(np.float32)
        offs = (-normal * np.float32(0.1))[:, None, :] + (np.cos(ang_) * rad)[:, :, None] * t1[:, None, :] + (np.sin(ang_) * rad)[:, :, None] * t2[:, None, :]
        return counts, offs.astype(np.float32), rng.uniform(-0.01, 0.03, size=(k, 4)).astype(np.float32)

    if m_tube > 0:
        ta = rng.integers(0, total_dyn, size=m_tube)
        normal = rng.standard_normal((m_tube, 3)).astype(np.float32)
        normal /= np.linalg.norm(normal, axis=1, keepdims=True)
        counts, offs, depths = geometry(m_tube, body_pos[ta], normal)
        offset_b = bodies[0, 4:7][None, :] - body_pos[ta]
        for N in (1, 2, 3, 4):
            sel = counts == N
            if sel.any():
                pre = convex_prestep(offs[sel][:, :N], depths[sel][:, :N], normal[sel], offset_b[sel], friction=2.0, spring_settings=tube_spring, max_recovery=fmax)
                constraints.append((CONVEX_TWO_BODY[N], np.stack([ta[sel] + 1, np.zeros(int(sel.sum()), dtype=np.int64)], axis=1).astype(np.int32), pre))
    if m_pair > 0 and count > 1:
        pa_ = rng.integers(0, total_dyn, size=m_pair)
        shift = rng.integers(nb, min(total_dyn - 1, 4 * nb) + 1, size=m_pair)  # a body of a nearby but different ragdoll
        pb_ = (pa_ + shift) % total_dyn
        d = body_pos[pa_] - body_pos[pb_]
        normal = (d / np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-3)).astype(np.float32)
        counts, offs, depths = geometry(m_pair, body_pos[pa_], normal)
        offset_b = (-normal * np.float32(0.2)).astype(np.float32)
        for N in (1, 2, 3, 4):
            sel = counts == N
            if sel.any():
                pre = convex_prestep(offs[sel][:, :N], depths[sel][:, :N], normal[sel], offset_b[sel])
                constraints.append((CONVEX_TWO_BODY[N], np.stack([pa_[sel] + 1, pb_[sel] + 1], axis=1).astype(np.int32), pre))
    total = sum(c[1].shape[0] for c in constraints)
    return {"bodies": bodies, "constraints": constraints,
            "description": "%d ragdolls (%d bodies, %d joints) + kinematic tube, %d constraints total" % (count, total_dyn, 58 * count, total)}


# (type id, bodies per constraint) of every joint / motor / servo / limit type of DefaultTypes.cs beyond the ragdoll set.
JOINT_ZOO_TYPES = {23: 2, 24: 2, 28: 2, 31: 2, 32: 4, 33: 2, 34: 2, 35: 2, 36: 3, 37: 2, 38: 2, 39: 2, 40: 2, 41: 2, 42: 1, 43: 1, 44: 1, 45: 1, 52: 2, 53: 2, 54: 2, 55: 2}


def joint_zoo(body_count=2000, per_type=200, seed=5, kinematic_fraction=0.05, types=None):
    """Random bodies on a jittered grid, connected by `per_type` constraints of each type in JOINT_ZOO_TYPES (or `types`) with randomised
    but physically sensible prestep data (Weld, AngularHinge, AngularSwivelHinge, TwistMotor, AngularAxisMotor, AngularAxisGearMotor,
    BallSocketServo/Motor, DistanceServo/Limit, PointOnLineServo, LinearAxisServo/Motor/Limit, CenterDistance constraint/limit, the four
    one-body servos/motors, AreaConstraint (3 bodies) and VolumeConstraint (4 bodies)). A fraction of the bodies is kinematic; no constraint
    gets more than one kinematic body and one-body constraints only go on dynamic bodies."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n = body_count
    side = int(math.ceil(n ** (1.0 / 3.0)))
    idx = np.arange(n)
    pos = np.stack([idx % side, (idx // side) % side, idx // (side * side)], axis=1).astype(np.float32) * np.float32(1.5)
    pos += rng.uniform(-0.3, 0.3, size=(n, 3)).astype(np.float32)
    inv_inertia = _shape_inverse_inertias()[rng.integers(0, 5, size=n)]
    inv_mass = rng.uniform(0.5, 2.0, size=n).astype(np.float32)
    kinematic = rng.random(n) < kinematic_fraction
    inv_mass[kinematic] = 0
    inv_inertia[kinematic] = 0
    bodies = make_bodies(pos, orientation=_random_unit_quaternions(rng, n), linear=rng.uniform(-0.5, 0.5, size=(n, 3)).astype(np.float32),
                         angular=rng.uniform(-0.5, 0.5, size=(n, 3)).astype(np.float32), inverse_mass=inv_mass, inverse_inertia=inv_inertia)
    dynamic = np.flatnonzero(~kinematic).astype(np.int32)
    fmax = np.float32(np.finfo(np.float32).max)

    def f32(x):
        return np.asarray(x, dtype=np.float32)

    def offsets(m):
        return rng.uniform(-0.5, 0.5, size=(m, 3)).astype(np.float32)

    def axes(m):
        a = rng.standard_normal((m, 3)).astype(np.float32)
        return (a / np.linalg.norm(a, axis=1, keepdims=True)).astype(np.float32)

    def scalars(m, lo, hi):
        return rng.uniform(lo, hi, size=(m, 1)).astype(np.float32)

    def springs(m):
        return np.concatenate([scalars(m, 5, 30) * TWO_PI, scalars(m, 0.3, 1.5) * np.float32(2)], axis=1).astype(np.float32)

    def servos(m):  # MaximumSpeed, BaseSpeed, MaximumForce; a third of them unlimited like ServoSettings.Default
        s = np.concatenate([scalars(m, 0.5, 5), scalars(m, 0, 0.5), scalars(m, 10, 1000)], axis=1)
        unlimited = rng.random(m) < 0.33
        s[unlimited] = (fmax, 0, fmax)
        return s.astype(np.float32)

    def motors(m):  # MaximumForce, Damping (MotorSettings softness)
        s = np.concatenate([scalars(m, 10, 1000), scalars(m, 0.1, 100)], axis=1)
        s[rng.random(m) < 0.33, 0] = fmax
        return s.astype(np.float32)

    def pick(m, count):
        """`count` distinct nearby bodies per constraint (consecutive grid indices from a random start), at most one kinematic: the first is dynamic."""
        first = dynamic[rng.integers(0, dynamic.shape[0], size=m)]
        cols = [first]
        for k in range(1, count):
            cand = (first + k * (1 + rng.integers(0, 3, size=m))) % n
            # replace kinematic partners of slots >= 2 (and duplicates) by the next dynamic body
            for _ in range(8):
                bad = np.zeros(m, dtype=bool)
                for c in cols:
                    bad |= cand == c
                if k >= 2:
                    bad |= kinematic[cand]
                if not bad.any():
                    break
                cand = np.where(bad, (cand + 1) % n, cand)
            cols.append(cand.astype(np.int32))
        return np.stack(cols, axis=1).astype(np.int32)

    constraints = []
    chosen = JOINT_ZOO_TYPES if types is None else {t: JOINT_ZOO_TYPES[t] for t in types}
    for type_id, nb in chosen.items():
        m = per_type
        h = pick(m, nb)
        if nb >= 2:  # at most one kinematic body: slot 1 may be kinematic, slots 0 and >= 2 are dynamic
            assert not kinematic[h[:, 0]].any() and not kinematic[h[:, 2:]].any()
        p0 = pos[h[:, 0]]
        if type_id in (23, 24):
            pre = np.concatenate([axes(m), axes(m), springs(m)], axis=1)
        elif type_id == 28:
            pre = np.concatenate([axes(m), axes(m), scalars(m, -2, 2), motors(m)], axis=1)
        elif type_id == 31:
            pre = np.concatenate([offsets(m) * 2, _random_unit_quaternions(rng, m), springs(m)], axis=1)
        elif type_id == 32:
            ab, ac, ad = pos[h[:, 1]] - p0, pos[h[:, 2]] - p0, pos[h[:, 3]] - p0
            volume = np.einsum("ij,ij->i", np.cross(ab, ac), ad)[:, None]
            pre = np.concatenate([volume * scalars(m, 0.8, 1.2), springs(m)], axis=1)
        elif type_id == 33:
            pre = np.concatenate([offsets(m), offsets(m), scalars(m, 0.5, 3), servos(m), springs(m)], axis=1)
        elif type_id == 34:
            lo = scalars(m, 0.2, 1.5)
            pre = np.concatenate([offsets(m), offsets(m), lo, lo + scalars(m, 0.5, 2), springs(m)], axis=1)
        elif type_id == 35:
            pre = np.concatenate([scalars(m, 0.5, 3), springs(m)], axis=1)
        elif type_id == 36:
            area = np.linalg.norm(np.cross(pos[h[:, 1]] - p0, pos[h[:, 2]] - p0), axis=1)[:, None]
            pre = np.concatenate([area * scalars(m, 0.8, 1.2), springs(m)], axis=1)
        elif type_id == 37:
            pre = np.concatenate([offsets(m), offsets(m), axes(m), servos(m), springs(m)], axis=1)
        elif type_id == 38:
            pre = np.concatenate([offsets(m), offsets(m), axes(m), scalars(m, -1, 1), servos(m), springs(m)], axis=1)
        elif type_id == 39:
            pre = np.concatenate([offsets(m), offsets(m), axes(m), scalars(m, -2, 2), motors(m)], axis=1)
        elif type_id == 40:
            pre = np.concatenate([offsets(m), offsets(m), axes(m), scalars(m, -1.5, 0), scalars(m, 0, 1.5), springs(m)], axis=1)
        elif type_id == 41:
            pre = np.concatenate([axes(m), scalars(m, -2, 2), motors(m)], axis=1)
        elif type_id == 42:
            pre = np.concatenate([_random_unit_quaternions(rng, m), springs(m), servos(m)], axis=1)
        elif type_id == 43:
            pre = np.concatenate([offsets(m) * 4, motors(m)], axis=1)
        elif type_id == 44:
            pre = np.concatenate([offsets(m), p0 + offsets(m) * 2, springs(m), servos(m)], axis=1)
        elif type_id == 45:
            pre = np.concatenate([offsets(m), offsets(m) * 4, motors(m)], axis=1)
        elif type_id == 52:
            pre = np.concatenate([offsets(m), offsets(m) * 4, motors(m)], axis=1)
        elif type_id == 53:
            pre = np.concatenate([offsets(m), offsets(m), springs(m), servos(m)], axis=1)
        elif type_id == 54:
            pre = np.concatenate([axes(m), scalars(m, 0.5, 3), motors(m)], axis=1)
        elif type_id == 55:
            lo = scalars(m, 0.2, 1.5)
            pre = np.concatenate([lo, lo + scalars(m, 0.5, 2), springs(m)], axis=1)
        else:
            raise ValueError("joint_zoo has no generator for type %d" % type_id)
        constraints.append((type_id, h, np.ascontiguousarray(f32(pre))))
    total = sum(c[1].shape[0] for c in constraints)
    return {"bodies": bodies, "constraints": constraints, "description": "joint zoo: %d bodies, %d constraints of %d types" % (n, total, len(constraints))}


def merge(*parts):
    """Concatenates scenes into one (body handles of later parts are shifted): independent islands in one simulation, so one solve exercises every
    constraint type, kinematic partners and unconstrained bodies together."""
    bodies, constraints, offset = [], [], 0
    for part in parts:
        bodies.append(part["bodies"])
        for type_id, handles, prestep in part["constraints"]:
            constraints.append((type_id, (handles + offset).astype(np.int32), prestep))
        offset += part["bodies"].shape[0]
    return {"bodies": np.concatenate(bodies), "constraints": constraints, "description": " + ".join(p.get("description", "?") for p in parts)}


def build(scene, simulation):
    """Adds a scene to a host Simulation (Bodies.Add, then Solver.Add per constraint in list order)."""
    simulation.add_bodies(scene["bodies"])
    for type_id, handles, prestep in scene["constraints"]:
        simulation.add_constraints(type_id, handles, prestep)
    return simulation


# ---- PredictBoundingBoxes worlds: every built-in shape type (bepucuda_set_shape_library / bepucuda_set_body_collidables) -----------------------
def bundle_hull_points(points, width):
    """ConvexHull.Points for a point set: Vector3Wide bundles [bundles, 3, width], the last bundle padded by repeating the last point
    (ConvexHullHelper.cs:L1050-1062). The bounds only read the points, so any point set will do; it need not be a hull."""
    points = np.asarray(points, dtype=np.float32).reshape(-1, 3)
    bundles = (points.shape[0] + width - 1) // width
    index = np.minimum(np.arange(bundles * width), points.shape[0] - 1)
    return np.ascontiguousarray(points[index].reshape(bundles, width, 3).transpose(0, 2, 1))


def shape_library(rng, hull_width=8, primitives=64, hulls=32, hull_points=(20, 64), compounds=32, big_compounds=8, compound_children=(2, 16), mesh_triangle_counts=(),
                  mesh_triangles_shared=None):
    """A random shape library: `primitives` shapes of each primitive type and triangles, hulls of hull_points[0]..[1] points, compounds and big
    compounds of compound_children[0]..[1] children of every convex type (hulls included), one mesh per entry of mesh_triangle_counts with a
    non-uniform scale."""
    from .native import ShapeLibrary, COMPOUND_CHILD_DTYPE, typed_index

    u = lambda lo, hi, *shape: rng.uniform(lo, hi, size=shape).astype(np.float32)
    bundles, hull_records, first = [], [], 0
    for _ in range(hulls):
        pts = bundle_hull_points(u(-1.5, 1.5, int(rng.integers(hull_points[0], hull_points[1] + 1)), 3), hull_width)
        bundles.append(pts)
        hull_records.append((first, pts.shape[0]))
        first += pts.shape[0]
    counts = {0: primitives, 1: primitives, 2: primitives, 3: primitives, 4: primitives, 5: hulls}
    children, records = [], [[], []]
    for kind, how_many in ((0, compounds), (1, big_compounds)):
        for _ in range(how_many):
            k = int(rng.integers(compound_children[0], compound_children[1] + 1))
            c = np.zeros(k, dtype=COMPOUND_CHILD_DTYPE)
            q = rng.normal(size=(k, 4))
            c["local_orientation"] = q / np.linalg.norm(q, axis=1, keepdims=True)
            c["local_position"] = u(-3, 3, k, 3)
            types = rng.choice([t for t in range(6) if counts[t] > 0], size=k)
            c["shape"] = typed_index(types, [int(rng.integers(0, counts[t])) for t in types])
            records[kind].append((sum(len(x) for x in children), k))
            children.append(c)
    mesh_pool, mesh_records = [], []
    for count in mesh_triangle_counts:
        tri = mesh_triangles_shared[:count] if mesh_triangles_shared is not None else u(-4, 4, count, 9)
        mesh_records.append((sum(len(x) for x in mesh_pool), count, tuple(u(0.2, 3.0, 3))))
        mesh_pool.append(tri)
    return ShapeLibrary(spheres=u(0.05, 2, primitives), capsules=u(0.05, 2, primitives, 2), boxes=u(0.05, 2, primitives, 3), triangles=u(-2, 2, primitives, 9),
                        cylinders=u(0.05, 2, primitives, 2), hull_points=np.concatenate(bundles) if bundles else None, hull_bundle_width=hull_width, hulls=hull_records,
                        compound_children=np.concatenate(children) if children else (), compounds=records[0], big_compounds=records[1],
                        mesh_triangles=np.concatenate(mesh_pool) if mesh_pool else (), meshes=mesh_records)


def shape_world(body_count, seed=5, library=None, type_weights=None, kinematic_fraction=0.1, **library_args):
    """Random bodies over a shape library (shape_library(**library_args) unless one is given): BodyDynamics records, one BODY_COLLIDABLE_DTYPE
    and one BODY_ACTIVITY_DTYPE record per body. type_weights: relative frequency of the shape types 0-8, plus 'none' (no shape) and 'user'
    (a user-registered type id, which has no built-in bounds). Spins range from still to fast enough for the pi/3 clamp."""
    from .native import BODY_ACTIVITY_DTYPE, BODY_COLLIDABLE_DTYPE, typed_index

    rng = np.random.default_rng(seed)
    library = library if library is not None else shape_library(rng, **library_args)
    weights = dict(type_weights or {0: 1, 1: 1, 2: 1, 3: 1, 4: 1, 5: 2, 6: 2, 7: 1, 8: 0.2, "none": 0.3, "user": 0.2})
    for t in list(weights):
        if isinstance(t, int) and library.count(t) == 0:
            weights.pop(t)
    keys = list(weights)
    p = np.array([weights[k] for k in keys], dtype=np.float64)
    kinds = rng.choice(len(keys), size=body_count, p=p / p.sum())
    collidables = np.zeros(body_count, dtype=BODY_COLLIDABLE_DTYPE)
    for j, k in enumerate(keys):
        sel = kinds == j
        m = int(sel.sum())
        if k == "none":
            collidables["shape"][sel] = rng.integers(0, 1 << 31, size=m).astype(np.uint32) & np.uint32(0x7FFFFFFF)
        elif k == "user":
            collidables["shape"][sel] = typed_index(rng.integers(9, 128, size=m), rng.integers(0, 1 << 24, size=m))
        else:
            collidables["shape"][sel] = typed_index(np.full(m, k), rng.integers(0, library.count(k), size=m))
    collidables["minimum_speculative_margin"] = rng.choice([0.0, 0.01, 0.2], size=body_count)
    collidables["maximum_speculative_margin"] = rng.choice([0.05, 1.0, 3.40282347e+38], size=body_count)
    collidables["allow_expansion_beyond_speculative_margin"] = rng.integers(0, 2, size=body_count)
    q = _random_unit_quaternions(rng, body_count)
    bodies = make_bodies(rng.uniform(-50, 50, size=(body_count, 3)), orientation=q,
                         linear=rng.normal(size=(body_count, 3)) * rng.choice([0.0, 0.1, 5.0, 80.0], size=(body_count, 1)),
                         angular=rng.normal(size=(body_count, 3)) * rng.choice([0.0, 0.3, 10.0, 200.0], size=(body_count, 1)),
                         inverse_mass=np.ones(body_count), inverse_inertia=np.tile(np.array([[1, 0, 1, 0, 0, 1]], dtype=np.float32), (body_count, 1)))
    bodies[rng.random(body_count) < kinematic_fraction, 16:23] = 0.0
    activities = np.zeros(body_count, dtype=BODY_ACTIVITY_DTYPE)
    activities["sleep_threshold"] = rng.choice([-1.0, 0.01, 5.0], size=body_count)
    activities["minimum_timesteps_under_threshold"] = rng.integers(1, 40, size=body_count)
    activities["timesteps_under_threshold_count"] = rng.integers(0, 256, size=body_count)
    return {"bodies": bodies, "library": library, "collidables": collidables, "activities": activities}
