"""Float64 reference geometry for tests/test_geometry_primitives.py, written from the geometric definitions of Box2D
2.3.x's shapes, manifolds, distance and time of impact (SURVEY.md Appendix B), plus the drivers of the two probes
(kb_probe_geometry on the device, kbo_probe_geometry in the oracle) that run the float32 routines one case at a time."""
import ctypes as C
import math

import numpy as np
from scipy.spatial import ConvexHull

from gym_kilobots_b200 import _abi as abi

F32 = np.float32
EPS = float(np.finfo(np.float32).eps)
SLOP = float(F32(0.005))
POLY_RADIUS = float(F32(2.0) * F32(0.005))           # b2_polygonRadius as the float32 both sides store
K_TOL = float(F32(0.1) * F32(0.005))                  # b2CollidePolygons' reference-face tolerance
ANGULAR_SLOP = float(F32(2.0) / F32(180.0) * F32(3.14159265359))
# Margin of a float32 result: every checked quantity is reached through at most 128 float32 roundings (two transforms,
# differences, dot products, a normalisation, one clip), each off by at most eps/2 of the case's scale S, so the float32
# value is within 64 * eps * S of the float64 one.  Decisions closer than that to their threshold are not checked.
MARGIN_K = 64.0

MANIFOLD_CIRCLES, MANIFOLD_FACE_A, MANIFOLD_FACE_B = 0, 1, 2


def margin(scale):
    return MARGIN_K * EPS * scale


def make_id(ia, ib, ta, tb):
    return (ia & 0xFF) | ((ib & 0xFF) << 8) | ((ta & 0xFF) << 16) | ((tb & 0xFF) << 24)


def swap_id(i):
    return ((i >> 8) & 0xFF) | ((i & 0xFF) << 8) | ((i >> 8) & 0xFF0000) | ((i & 0xFF0000) << 8)


# ------------------------------------------------------------------------------------------------ shapes
class Shape:
    """One probe shape: its KbProbeShape and its float64 reference geometry.
    kind 'circle' (pts = the centre), 'poly' (pts CCW, normals), 'edge' (pts = v1, v2; ghosts v0 / v3)."""

    def __init__(self, kind, radius, pts, normals=None, centroid=None, ghost0=None, ghost3=None, desc=None, name=""):
        self.kind, self.radius, self.pts, self.normals, self.centroid = kind, radius, pts, normals, centroid
        self.ghost0, self.ghost3, self.desc, self.name = ghost0, ghost3, desc, name

    @property
    def extent(self):
        return float(np.abs(self.pts).max()) + self.radius


def weld(points):
    """b2PolygonShape::Set's weld: a point is dropped when its squared distance to a kept point is below
    0.5 * b2_linearSlop (Box2D 2.3.x compares the squared distance with half the slop, in float32)."""
    kept = []
    for p in points:
        p32 = p.astype(np.float32)
        if all(float(np.dot((p32 - q).astype(np.float32), (p32 - q).astype(np.float32))) >= 0.5 * SLOP for q in kept):
            kept.append(p32)
    return np.array(kept, np.float64)


def reference_polygon(points):
    """Hull, normals, area centroid in float64.  Vertices CCW from the right-most point (lowest y on a tie), the start
    vertex of b2PolygonShape::Set's gift wrap; collinear points are not vertices."""
    ps = weld(np.asarray(points, np.float32))
    hull = ConvexHull(ps)
    idx = list(hull.vertices)                      # counter-clockwise for 2-D input
    xs = ps[idx]
    start = min(range(len(idx)), key=lambda k: (-xs[k, 0], xs[k, 1]))
    V = np.roll(xs, -start, axis=0)
    E = np.roll(V, -1, axis=0) - V
    N = np.stack([E[:, 1], -E[:, 0]], 1) / np.linalg.norm(E, axis=1)[:, None]
    cross = V[:, 0] * np.roll(V, -1, 0)[:, 1] - V[:, 1] * np.roll(V, -1, 0)[:, 0]
    area = 0.5 * cross.sum()
    centroid = ((V + np.roll(V, -1, 0)) * cross[:, None]).sum(0) / (6.0 * area)
    return V, N, centroid


def circle_shape(radius, name="circle"):
    fd = abi.KbFixtureDef()
    fd.shape = abi.KB_SHAPE_CIRCLE
    fd.radius = radius
    return Shape("circle", float(F32(radius)), np.zeros((1, 2)), desc=_fixture_desc(fd), name=name)


def box_shape(hx, hy, name="box"):
    fd = abi.KbFixtureDef()
    fd.shape = abi.KB_SHAPE_BOX
    fd.hx, fd.hy = hx, hy
    hx, hy = float(F32(hx)), float(F32(hy))
    V = np.array([[-hx, -hy], [hx, -hy], [hx, hy], [-hx, hy]])
    N = np.array([[0.0, -1.0], [1.0, 0.0], [0.0, 1.0], [-1.0, 0.0]])
    return Shape("poly", POLY_RADIUS, V, N, np.zeros(2), desc=_fixture_desc(fd), name=name)


def polygon_shape(points, name="polygon"):
    points = np.asarray(points, np.float64)
    fd = abi.KbFixtureDef()
    fd.shape = abi.KB_SHAPE_POLYGON
    fd.vertex_count = len(points)
    for k, (x, y) in enumerate(points):
        fd.vx[k], fd.vy[k] = x, y
    V, N, c = reference_polygon(points)
    return Shape("poly", POLY_RADIUS, V, N, c, desc=_fixture_desc(fd), name=name)


def _fixture_desc(fd):
    d = abi.KbProbeShape()
    d.kind = abi.KB_PROBE_FIXTURE
    d.fixture = fd
    return d


TABLE = (-25.0, -18.75, 25.0, 18.75)   # the default 2.0 m x 1.5 m arena in b2 units


def chain_edge(i, edges, box=TABLE):
    """Child i of the table chain (x0,y1) -> (x0,y0) -> (x1,y0) -> (x1,y1) [-> (x0,y1)]; ghosts from the neighbours."""
    x0, y0, x1, y1 = [float(F32(v)) for v in box]
    v = np.array([[x0, y1], [x0, y0], [x1, y0], [x1, y1], [x0, y1]])
    count = 5 if edges == 4 else 4
    loop = edges == 4
    g0 = v[i - 1] if i > 0 else (v[count - 2] if loop else None)
    g3 = v[i + 2] if i < count - 2 else (v[1] if loop else None)
    d = abi.KbProbeShape()
    d.kind = abi.KB_PROBE_EDGE
    d.edge, d.wall_edges = i, edges
    d.wall_x0, d.wall_y0, d.wall_x1, d.wall_y1 = box
    return Shape("edge", POLY_RADIUS, np.array([v[i], v[i + 1]]), ghost0=g0, ghost3=g3, desc=d,
                 name="edge%d/%d%s" % (i, edges, "" if box == TABLE else " of %s" % (box,)))


# ------------------------------------------------------------------------------------------------ probes
CASE_WORDS = 28


def pack_cases(rows):
    """rows: dicts with a, b and xf_a / xf_b (x, y, s, c) or sweep_a / sweep_b (lc.xy c0.xy c.xy a0 a), fixed_rot_*."""
    arr = np.zeros((len(rows), CASE_WORDS), np.float32)
    ints = arr.view(np.int32)
    for k, r in enumerate(rows):
        ints[k, 0], ints[k, 1] = r["a"], r["b"]
        ints[k, 2], ints[k, 3] = r.get("fixed_rot_a", 0), r.get("fixed_rot_b", 0)
        arr[k, 4:8] = r.get("xf_a", (0, 0, 0, 1))
        arr[k, 8:12] = r.get("xf_b", (0, 0, 0, 1))
        arr[k, 12:20] = r.get("sweep_a", (0,) * 8)
        arr[k, 20:28] = r.get("sweep_b", (0,) * 8)
    return arr


def run_probe(fn, err, op, shapes, cases=None):
    """fn: the bound kb_probe_geometry / kbo_probe_geometry; returns u32[rows, KB_PROBE_OUT_WORDS]."""
    descs = (abi.KbProbeShape * len(shapes))(*[s.desc for s in shapes])
    n = len(shapes) if op == abi.KB_PROBE_SHAPE else len(cases)
    out = np.zeros((n, abi.KB_PROBE_OUT_WORDS), np.uint32)
    cp = None if cases is None else cases.ctypes.data_as(C.c_void_p)
    rc = fn(-1, op, 0 if cases is None else len(cases), C.cast(descs, C.c_void_p), len(shapes), cp,
            out.ctypes.data_as(C.c_void_p))
    assert rc == 0, err().decode()
    return out


def f32(words):
    return np.asarray(words, np.uint32).view(np.float32)


# ------------------------------------------------------------------------------------------------ transforms
def xf_from_angle(x, y, angle):
    """A body transform as the kernels hold it: float32 position, float32 sin / cos."""
    return (float(F32(x)), float(F32(y)), float(F32(math.sin(angle))), float(F32(math.cos(angle))))


def rot(xf):
    s, c = xf[2], xf[3]
    return np.array([[c, -s], [s, c]])


def apply(xf, pts):
    return np.asarray(pts, np.float64) @ rot(xf).T + np.array(xf[:2])


def apply_t(xf, pts):
    return (np.asarray(pts, np.float64) - np.array(xf[:2])) @ rot(xf)


# ------------------------------------------------------------------------------------------------ distances
def seg_point_dist(a, b, q):
    e = b - a
    den = float(e @ e)
    t = 0.0 if den == 0.0 else min(1.0, max(0.0, float((q - a) @ e) / den))
    return float(np.linalg.norm(q - (a + t * e)))


def poly_signed_distance(V, N, q):
    """Signed distance from q to a convex polygon: the largest face separation inside, the Euclidean distance outside."""
    s = ((q - V) * N).sum(1)
    if s.max() <= 0.0:
        return float(s.max())
    return min(seg_point_dist(V[i], V[(i + 1) % len(V)], q) for i in range(len(V)))


def _edges(P):
    if len(P) == 1:
        return []
    if len(P) == 2:
        return [(P[0], P[1])]
    return [(P[i], P[(i + 1) % len(P)]) for i in range(len(P))]


def _axes(P):
    out = []
    for a, b in _edges(P):
        e = b - a
        n = np.array([e[1], -e[0]])
        L = np.linalg.norm(n)
        if L > 0:
            out.append(n / L)
    return out


def core_distance(PA, PB):
    """Exact distance between the convex hulls of two point sets (1 point, a segment or a CCW polygon): 0 when they
    overlap (no separating axis among the edge normals), else the minimum over vertex-edge and vertex-vertex pairs."""
    PA, PB = np.asarray(PA, np.float64), np.asarray(PB, np.float64)
    if len(PA) == 1 and len(PB) >= 3:
        return max(0.0, poly_signed_distance(PB, np.array(_axes(PB)), PA[0]))
    if len(PB) == 1 and len(PA) >= 3:
        return max(0.0, poly_signed_distance(PA, np.array(_axes(PA)), PB[0]))
    if len(PA) >= 2 and len(PB) >= 2:
        if not any((PB @ n).min() > (PA @ n).max() or (PA @ n).min() > (PB @ n).max() for n in _axes(PA) + _axes(PB)):
            return 0.0
    best = min(float(np.linalg.norm(p - q)) for p in PA for q in PB)
    for P, Q in ((PA, PB), (PB, PA)):
        for a, b in _edges(Q):
            for p in P:
                best = min(best, seg_point_dist(a, b, p))
    return best


def _batch_edges(P):
    n = P.shape[1]
    if n == 1:
        return None
    if n == 2:
        return P[:, :1], P[:, 1:]
    return P, np.roll(P, -1, axis=1)


def _points_to_segments(P, a, b):
    """min over points P (T, n, 2) and segments a -> b (T, m, 2) of the point-segment distance, per T."""
    e = (b - a)[:, None]                                   # (T, 1, m, 2)
    d = P[:, :, None] - a[:, None]                         # (T, n, m, 2)
    den = np.maximum((e * e).sum(-1), 1e-300)
    t = np.clip((d * e).sum(-1) / den, 0.0, 1.0)
    return np.linalg.norm(d - t[..., None] * e, axis=-1).min(axis=(1, 2))


def core_distance_batch(PA, PB):
    """core_distance over a batch: PA (T, nA, 2), PB (T, nB, 2) -> (T,)."""
    best = np.linalg.norm(PA[:, :, None] - PB[:, None], axis=-1).min(axis=(1, 2))
    overlap = np.zeros(len(PA), bool)
    for P, Q in ((PA, PB), (PB, PA)):
        eq = _batch_edges(Q)
        if eq is not None:
            best = np.minimum(best, _points_to_segments(P, *eq))
    if PA.shape[1] >= 2 and PB.shape[1] >= 2 or PA.shape[1] >= 3 or PB.shape[1] >= 3:
        separated = np.zeros(len(PA), bool)
        for Q in (PA, PB):
            eq = _batch_edges(Q)
            if eq is None:
                continue
            e = eq[1] - eq[0]
            n = np.stack([e[..., 1], -e[..., 0]], -1)       # (T, k, 2)
            pa = np.einsum("tkd,tnd->tkn", n, PA)
            pb = np.einsum("tkd,tnd->tkn", n, PB)
            separated |= ((pb.min(2) > pa.max(2)) | (pa.min(2) > pb.max(2))).any(1)
        overlap = ~separated
    return np.where(overlap, 0.0, best)


def world_core(shape, xf):
    return apply(xf, shape.pts)


# ------------------------------------------------------------------------------------------------ manifolds
def world_manifold(m, sA, xfA, sB, xfB):
    """b2WorldManifold::Initialize in float64: (normal, [(point, separation)])."""
    ln, lp = np.array(m["ln"]), np.array(m["lp"])
    rA, rB = sA.radius, sB.radius
    pts = []
    if m["type"] == MANIFOLD_CIRCLES:
        pA = apply(xfA, lp[None])[0]
        pB = apply(xfB, np.array(m["p"][0])[None])[0]
        d = pB - pA
        L = np.linalg.norm(d)
        n = d / L if L > EPS else np.array([1.0, 0.0])
        return n, [(0.5 * (pA + pB), float(d @ n) - rA - rB)], L
    if m["type"] == MANIFOLD_FACE_A:
        n = rot(xfA) @ ln
        plane = apply(xfA, lp[None])[0]
        for k in range(m["count"]):
            c = apply(xfB, np.array(m["p"][k])[None])[0]
            pts.append((c, float((c - plane) @ n) - rA - rB))
        return n, pts, None
    n = rot(xfB) @ ln
    plane = apply(xfB, lp[None])[0]
    for k in range(m["count"]):
        c = apply(xfA, np.array(m["p"][k])[None])[0]
        pts.append((c, float((c - plane) @ n) - rA - rB))
    return -n, pts, None


def decode_manifold(row):
    fl = f32(row)
    return {"type": int(row[0]), "count": int(row[1]), "ln": (float(fl[2]), float(fl[3])),
            "lp": (float(fl[4]), float(fl[5])),
            "p": [(float(fl[6]), float(fl[7])), (float(fl[9]), float(fl[10]))], "id": [int(row[8]), int(row[11])]}


class Choices:
    """The decisions of one evaluation of a float64 reference.  A decision whose value lies within `tol` of its
    threshold can go either way in float32; it takes the branch that the next bit of `bits` names, so that evaluating
    the reference once per bit pattern (admissible) yields every answer the float32 routine may legitimately give.
    With tol = 0 the decisions are the exact float64 ones."""

    def __init__(self, tol, bits=0):
        self.tol, self.bits, self.n = tol, bits, 0

    def _bit(self):
        b = (self.bits >> self.n) & 1
        self.n += 1
        return b

    def le(self, x):
        """x <= 0"""
        if self.tol > 0.0 and abs(x) <= self.tol:
            return self._bit() == 1
        return x <= 0.0

    def gt(self, x):
        return not self.le(x)

    def ge(self, x):
        return self.le(-x)

    def lt(self, x):
        return not self.le(-x)

    def sign(self, x):
        """-1, 0 or +1; near zero any of the three (a float32 difference can be exactly zero)"""
        if self.tol > 0.0 and abs(x) <= self.tol:
            return (-1, 1, 0, 0)[self._bit() | (self._bit() << 1)]
        return (x > 0.0) - (x < 0.0)


def admissible(reference, tol, max_ambiguous=10):
    """(every answer of reference(choices) when each decision within tol of its threshold goes either way,
    the answer with the exact float64 decisions)"""
    exact = reference(Choices(0.0))
    out, bits, limit = [], 0, 1
    while bits < limit:
        ch = Choices(tol, bits)
        out.append(reference(ch))
        limit = max(limit, 1 << min(ch.n, max_ambiguous))
        bits += 1
    return out, exact


def clip_segment(ch, vin, normal, offset, index_a):
    """b2ClipSegmentToLine in float64: keep the vertices with dot(normal, v) <= offset, and the crossing point when
    the two lie strictly on opposite sides."""
    d0 = float(normal @ vin[0][0]) - offset
    d1 = float(normal @ vin[1][0]) - offset
    s0, s1 = ch.sign(d0), ch.sign(d1)
    out = [v for v, sg in ((vin[0], s0), (vin[1], s1)) if sg <= 0]
    if s0 * s1 < 0:
        t = d0 / (d0 - d1) if d0 != d1 else 0.5
        out.append((vin[0][0] + t * (vin[1][0] - vin[0][0]), make_id(index_a, (vin[0][1] >> 8) & 0xFF, 0, 1)))
    return out


def clip_face(ch, ref_v1, ref_v2, ref_i1, ref_i2, incident, radius, side=None):
    """Clip the incident segment to the side planes of the reference face (offsets widened by `side`, default `radius`:
    b2CollidePolygons widens them, b2EPCollider does not) and keep the points within `radius` of the face.
    -> ([(point, id, separation from the face)], the face normal)."""
    t = ref_v2 - ref_v1
    t = t / np.linalg.norm(t)
    n = np.array([t[1], -t[0]])
    side = radius if side is None else side
    c1 = clip_segment(ch, incident, -t, -float(t @ ref_v1) + side, ref_i1)
    if len(c1) < 2:
        return [], n
    c2 = clip_segment(ch, c1, t, float(t @ ref_v2) + side, ref_i2)
    if len(c2) < 2:
        return [], n
    pts = []
    for p, pid in c2:
        s = float(n @ (p - ref_v1))
        if ch.le(s - radius):
            pts.append((p, pid, s))
    return pts, n
