"""The narrowphase, distance and time-of-impact routines one case at a time, against float64 geometry.

Whole-step parity tests compare the CUDA kernels with the CPU oracle; both restate Box2D 2.3.x from memory, so they can
agree and both be wrong.  Here the float32 routines run through a test-only probe (kbo_probe_geometry in the oracle,
kb_probe_geometry on the device: the production device functions of kb_narrow.cuh / kb_toi.cuh, one thread per case)
and are checked against float64 geometry written from the definitions (tests/geometry_ref.py):
  * without a GPU: the oracle against the float64 reference, and the shapes kb_create builds (SHAPE runs on the host);
  * on the GPU: the device against the oracle, bit for bit, on every case of every family, and the claims of the kernel
    code that rest on arguments: time_of_impact_edge_circle == time_of_impact, fixedRot == the rotated sweep.
Cases are seeded random ones at the table's scale (coordinates up to about +-40 b2 units) and at unit scale, plus families
aimed at the branches where manifold code goes wrong.  Every float tolerance is geometry_ref.margin(scale): see MARGIN_K.
A decision within that margin of its threshold may go either way in float32, so the reference is evaluated for both
branches of every such decision (geometry_ref.Choices) and the float32 manifold must equal one of the admissible
answers in every respect -- point count, type, normal, points, ids and separations.  Nothing is exempt; how many cases
had more than one admissible answer is reported.
"""
import ctypes as C
import math

import numpy as np
import pytest

from gym_kilobots_b200 import _abi as abi
from gym_kilobots_b200 import scene as S
import geometry_ref as G

KILOBOT_R = float(np.float32(S.KILOBOT_RADIUS * S.WORLD_SCALE))


# ------------------------------------------------------------------------------------------------ shapes
def template_polygons():
    out = []
    for name, tpl in (("triangle", S.TRIANGLE_TEMPLATE), ("lform", S.LFORM_TEMPLATE), ("tform", S.TFORM_TEMPLATE),
                      ("cform", S.CFORM_TEMPLATE)):
        for w, h in ((0.15, 0.15), (0.1, 0.2)):
            for k, sub in enumerate(S.polygon_local_vertices(tpl, w, h)):
                out.append(G.polygon_shape(np.asarray(sub) * S.WORLD_SCALE, "%s%d(%g,%g)" % (name, k, w, h)))
    return out


def random_convex(rng, n, scale):
    ang = np.sort(rng.uniform(0, 2 * np.pi, n))
    rad = scale * rng.uniform(0.5, 1.0, n)
    pts = np.stack([rad * np.cos(ang), rad * np.sin(ang)], 1)
    return pts[rng.permutation(n)]


def shape_set():
    rng = np.random.default_rng(7)
    shapes = template_polygons()
    shapes += [G.box_shape(1.875, 1.875, "quad.15"), G.box_shape(2.5, 1.25, "quad.2x.1")]
    for k in range(40):
        shapes.append(G.polygon_shape(random_convex(rng, 3 + k % 6, [0.5, 3.0][k % 2]), "random%d" % k))
    # points closer than the weld distance (|d|^2 < slop / 2, i.e. |d| < 0.05): the duplicates must disappear
    shapes.append(G.polygon_shape([(1, 0), (1.03, 0.0), (0, 1), (-1, 0), (-1, 0.02), (0, -1)], "weld"))
    shapes.append(G.polygon_shape([(1, 0), (1.06, 0.0), (0, 1), (-1, 0), (0, -1)], "no-weld"))
    # collinear points on the hull's edges are not vertices
    shapes.append(G.polygon_shape([(0, 0), (1, 0), (2, 0), (2, 1), (2, 2), (0, 2), (1, 1)], "collinear"))
    shapes.append(G.polygon_shape([(-1, -1), (0, -1), (1, -1), (1, 1), (-1, 1), (-1, 0)], "collinear2"))
    for e in (3, 4):
        shapes += [G.chain_edge(i, e) for i in range(e)]
    return shapes


def test_shapes_match_the_float64_hull(oracle, native):
    """kb_create's buildPolygon / buildBox / chain edges (the SHAPE op runs on the host) against the float64 hull of the
    welded input, and the oracle's own shape code against the same.  Vertices are input points, so they must be equal;
    normals unit, outward and perpendicular to their edge; the centroid the area centroid; the radius b2_polygonRadius."""
    shapes = shape_set()
    _, fo = oracle.load()
    for who, fn, err in (("device", native._fn["probe_geometry"], native._fn["last_error"]),
                         ("oracle", fo["probe_geometry"], fo["last_error"])):
        out = G.run_probe(fn, err, abi.KB_PROBE_SHAPE, shapes)
        fl = G.f32(out)
        for s, row, frow in zip(shapes, out, fl):
            where = "%s shape %s" % (who, s.name)
            assert frow[1] == np.float32(s.radius), where
            if s.kind == "edge":
                vs = np.stack([frow[6:10], frow[14:18]], 1)
                assert row[0] == 2 and np.array_equal(vs[1:3], s.pts), where
                assert row[2] == (s.ghost0 is not None) and row[3] == (s.ghost3 is not None), where
                if s.ghost0 is not None:
                    assert np.array_equal(vs[0], s.ghost0), where
                if s.ghost3 is not None:
                    assert np.array_equal(vs[3], s.ghost3), where
                continue
            m = int(row[0])
            V = np.stack([frow[6:6 + m], frow[14:14 + m]], 1).astype(np.float64)
            N = np.stack([frow[22:22 + m], frow[30:30 + m]], 1).astype(np.float64)
            assert m == len(s.pts), "%s: %d vertices, float64 hull has %d" % (where, m, len(s.pts))
            assert np.array_equal(V, s.pts), "%s: vertices %s, float64 hull %s" % (where, V, s.pts)
            tol = G.margin(s.extent)
            assert np.all(np.abs(np.linalg.norm(N, axis=1) - 1.0) <= 4 * G.EPS), where
            assert np.all(np.abs(N - s.normals).max(1) <= 4 * G.EPS), "%s: normals %s vs %s" % (where, N, s.normals)
            c = frow[4:6].astype(np.float64)
            assert np.abs(c - s.centroid).max() <= tol, "%s: centroid %s vs %s" % (where, c, s.centroid)


def test_probes_refuse_pairs_without_a_narrowphase_routine(oracle, native):
    """COLLIDE takes only the pairs the contact register forms: a circle as A only against a circle, never an edge as B.
    (The check is on the host: no GPU needed.)"""
    shapes = [G.circle_shape(0.5), G.box_shape(1.0, 1.0), G.chain_edge(0, 3)]
    _, fo = oracle.load()
    descs = (abi.KbProbeShape * len(shapes))(*[s.desc for s in shapes])
    for fn in (native._fn["probe_geometry"], fo["probe_geometry"]):
        for a, b, ok in ((0, 0, True), (1, 0, True), (1, 1, True), (2, 0, True), (2, 1, True),
                         (0, 1, False), (0, 2, False), (1, 2, False), (2, 2, False)):
            if ok and fn is native._fn["probe_geometry"]:
                continue   # a valid pair goes on to the device
            out = np.zeros((1, abi.KB_PROBE_OUT_WORDS), np.uint32)
            cases = G.pack_cases([{"a": a, "b": b}])
            rc = fn(-1, abi.KB_PROBE_COLLIDE, 1, C.cast(descs, C.c_void_p), len(shapes), cases.ctypes.data_as(C.c_void_p),
                    out.ctypes.data_as(C.c_void_p))
            assert (rc == 0) == ok, (shapes[a].name, shapes[b].name, rc)


# ------------------------------------------------------------------------------------------------ manifold cases
class Cases:
    """Shapes (indices into one list) and collide cases, with the family each case belongs to."""

    def __init__(self):
        self.shapes, self.rows, self.family = [], [], []
        self._index = {}

    def shape(self, s):
        if id(s) not in self._index:
            self._index[id(s)] = len(self.shapes)
            self.shapes.append(s)
        return self._index[id(s)]

    def add(self, family, sA, xfA, sB, xfB):
        self.rows.append({"a": self.shape(sA), "b": self.shape(sB), "xf_a": xfA, "xf_b": xfB})
        self.family.append(family)


def ulp_steps(x, k):
    return float(np.nextafter(np.float32(x), np.float32(np.inf if k > 0 else -np.inf))) if k else x


def collide_cases():
    rng = np.random.default_rng(2024)
    cs = Cases()
    kb = G.circle_shape(KILOBOT_R, "kilobot")
    big = G.circle_shape(1.25, "circle1.25")
    unit = G.circle_shape(0.5, "circle0.5")
    polys = [s for s in shape_set() if s.kind == "poly"]
    # the table, and the same chain mirrored (x0 > x1: it runs the other way round, every corner concave)
    mirrored = (G.TABLE[2], G.TABLE[1], G.TABLE[0], G.TABLE[3])
    edges = [G.chain_edge(i, e, box) for box in (G.TABLE, mirrored) for e in (3, 4) for i in range(e)]

    def rnd_xf(scale):
        return G.xf_from_angle(rng.uniform(-scale, scale), rng.uniform(-scale, scale), rng.uniform(-np.pi, np.pi))

    # -- circles: random, coincident centres, centres rA + rB apart plus or minus a few ulps
    for k in range(600):
        sc = [40.0, 1.0][k % 2]
        a, b = [(kb, kb), (kb, big), (unit, kb)][k % 3]
        xa = rnd_xf(sc)
        ang = rng.uniform(-np.pi, np.pi)
        d = (a.radius + b.radius) * rng.uniform(0.3, 1.5)
        cs.add("circles", a, xa, b, G.xf_from_angle(xa[0] + d * math.cos(ang), xa[1] + d * math.sin(ang), 0.0))
    for k in range(50):
        xa = rnd_xf(40.0)
        cs.add("circles/coincident", kb, xa, kb, (xa[0], xa[1], 0.0, 1.0))
    for k in range(200):
        a, b = [(kb, kb), (kb, big)][k % 2]
        R = np.float32(a.radius) + np.float32(b.radius)
        x = np.float32(rng.uniform(-40, 40))
        dx = ulp_steps(float(x + R), int(rng.integers(-3, 4)))
        cs.add("circles/rA+rB", a, (float(x), 5.0, 0.0, 1.0), b, (dx, 5.0, 0.0, 1.0))

    # -- circle against polygon: random, centre on a face, on a vertex, inside, on a Voronoi boundary
    for k in range(1500):
        p = polys[k % len(polys)]
        c = [kb, big][k % 2]
        sc = [40.0, 1.0][(k // 2) % 2]
        xa = rnd_xf(sc)
        local = rng.uniform(-1.6, 1.6, 2) * (p.extent + c.radius)
        w = G.apply(xa, local[None])[0]
        cs.add("poly-circle", p, xa, c, (float(w[0]), float(w[1]), 0.0, 1.0))
    for k in range(800):
        p = polys[k % len(polys)]
        c = kb
        xa = rnd_xf([40.0, 1.0][k % 2])
        i = int(rng.integers(len(p.pts)))
        v1, v2 = p.pts[i], p.pts[(i + 1) % len(p.pts)]
        kind = k % 4
        if kind == 0:    # on a face (outside by up to the radius)
            q = v1 + rng.uniform(0.05, 0.95) * (v2 - v1) + p.normals[i] * rng.uniform(-0.05, 1.2) * (c.radius + p.radius)
        elif kind == 1:  # on a vertex's Voronoi boundary: along the face normal through v1 (u1 == 0)
            q = v1 + p.normals[i] * rng.uniform(0.0, 1.2) * (c.radius + p.radius)
        elif kind == 2:  # around a vertex
            a = rng.uniform(0, 2 * np.pi)
            q = v1 + rng.uniform(0.0, 1.2) * (c.radius + p.radius) * np.array([math.cos(a), math.sin(a)])
        else:            # inside
            q = p.centroid + rng.uniform(-0.5, 0.5, 2) * (p.pts.max(0) - p.pts.min(0)) * 0.5
        w = G.apply(xa, q[None])[0]
        cs.add("poly-circle/targeted", p, xa, c, (float(w[0]), float(w[1]), 0.0, 1.0))

    # -- polygon against polygon
    for k in range(1500):
        pa, pb = polys[int(rng.integers(len(polys)))], polys[int(rng.integers(len(polys)))]
        sc = [40.0, 1.0][k % 2]
        xa = rnd_xf(sc)
        off = rng.uniform(-1, 1, 2) * (pa.extent + pb.extent) * 0.9
        w = G.apply(xa, off[None])[0]
        cs.add("poly-poly", pa, xa, pb, G.xf_from_angle(w[0], w[1], rng.uniform(-np.pi, np.pi)))
    boxes = [s for s in polys if s.name.startswith("quad")] + [polys[0]]
    for k in range(600):    # flush faces, and faces rotated +-1e-6 rad from flush; small / deep overlaps
        pa, pb = boxes[k % len(boxes)], boxes[(k // 3) % len(boxes)]
        xa = rnd_xf([40.0, 1.0][k % 2])
        i = int(rng.integers(len(pa.pts)))
        n = pa.normals[i]
        mid = 0.5 * (pa.pts[i] + pa.pts[(i + 1) % len(pa.pts)])
        # B's face j flush against A's face i: B rotated so that its normal j is -n
        j = int(rng.integers(len(pb.pts)))
        ang_b = math.atan2(-n[1], -n[0]) - math.atan2(pb.normals[j][1], pb.normals[j][0])
        ang_b += [0.0, 1e-6, -1e-6, 0.0][k % 4]
        depth = [0.0, 0.01, -0.015, 0.3, 0.021][k % 5]
        mb = 0.5 * (pb.pts[j] + pb.pts[(j + 1) % len(pb.pts)])
        rb = np.array([[math.cos(ang_b), -math.sin(ang_b)], [math.sin(ang_b), math.cos(ang_b)]])
        slide = rng.uniform(-0.8, 0.8) * np.array([-n[1], n[0]])
        pos_local = mid + n * (-depth) - rb @ mb + slide
        ang_a = math.atan2(xa[2], xa[3])
        pw = G.apply(xa, pos_local[None])[0]
        cs.add("poly-poly/flush", pa, xa, pb, G.xf_from_angle(pw[0], pw[1], ang_a + ang_b))
    for k in range(300):    # vertex-vertex near misses: SAT separation <= total radius, true distance larger
        pa, pb = boxes[k % len(boxes)], boxes[(k + 1) % len(boxes)]
        xa = rnd_xf([40.0, 1.0][k % 2])
        i = int(rng.integers(len(pa.pts)))
        va = pa.pts[i]
        dirn = va / np.linalg.norm(va)
        ang_b = rng.uniform(0.2, 1.3)
        rb = np.array([[math.cos(ang_b), -math.sin(ang_b)], [math.sin(ang_b), math.cos(ang_b)]])
        jb = int(np.argmin(pb.pts @ rb.T @ dirn))
        gap = rng.uniform(0.0, 0.03)
        pos_local = va + dirn * gap - rb @ pb.pts[jb]
        pw = G.apply(xa, pos_local[None])[0]
        cs.add("poly-poly/vertex", pa, xa, pb, G.xf_from_angle(pw[0], pw[1], math.atan2(xa[2], xa[3]) + ang_b))

    # -- against the table: random, every chain corner, and the open chain's ends
    for k in range(1500):
        e = edges[k % len(edges)]
        obj = [kb, big, polys[k % len(polys)], polys[(k * 7) % len(polys)]][k % 4]
        t = rng.uniform(-0.15, 1.15)
        base = e.pts[0] + t * (e.pts[1] - e.pts[0])
        q = base + rng.uniform(-1.3, 1.3, 2) * (obj.extent + e.radius)
        cs.add("edge-" + ("circle" if obj.kind == "circle" else "poly"), e, (0.0, 0.0, 0.0, 1.0), obj,
               G.xf_from_angle(q[0], q[1], rng.uniform(-np.pi, np.pi) if obj.kind == "poly" else 0.0))
    for e in edges:
        for end in (0, 1):
            corner = e.pts[end]
            for k in range(60):
                obj = [kb, big, polys[k % len(polys)]][k % 3]
                a = 2 * np.pi * k / 60 + 0.01
                r = (obj.extent + e.radius) * [0.5, 0.9, 1.02, 1.3][k % 4]
                q = corner + r * np.array([math.cos(a), math.sin(a)])
                cs.add("edge-corner", e, (0.0, 0.0, 0.0, 1.0), obj,
                       G.xf_from_angle(q[0], q[1], rng.uniform(-np.pi, np.pi) if obj.kind == "poly" else 0.0))
            # polygons around the corner on both sides of the chain, where the polygon axis and its adjacency filter
            # (the normal cone of the corner) decide
            for k in range(150):
                obj = polys[int(rng.integers(len(polys)))]
                q = corner + rng.uniform(-1.2, 1.2, 2) * obj.extent
                cs.add("edge-corner", e, (0.0, 0.0, 0.0, 1.0), obj, G.xf_from_angle(q[0], q[1], rng.uniform(-np.pi, np.pi)))
    return cs


# ------------------------------------------------------------------------------------------------ manifold reference
# Each reference below restates one narrowphase routine from its definition in float64 and returns the manifold it
# defines: an answer().  Every decision goes through `ch` (geometry_ref.Choices): a decision within the float margin of
# its threshold is evaluated both ways, so a case near a boundary is not exempt from anything -- the float32 manifold
# must equal one of the admissible answers in count, type, local normal and point, points, ids and separations.
class Tally(dict):
    def hit(self, key, n=1):
        self[key] = self.get(key, 0) + n


def answer(labels, mtype=None, ln=None, lp=None, ntol=0.0, pts=()):
    """pts: [(world point, feature id, separation as b2WorldManifold gives it)]"""
    return {"labels": [labels] if isinstance(labels, str) else list(labels), "count": len(pts), "type": mtype,
            "ln": None if ln is None else np.asarray(ln, np.float64), "lp": None if lp is None else np.asarray(lp, np.float64),
            "ntol": ntol, "pts": list(pts)}


def unit(v):
    L = float(np.linalg.norm(v))
    return v / L if L > 0.0 else v, L


def ref_circle_circle(ch, sA, xfA, sB, xfB, tol):
    pA, pB = np.array(xfA[:2]), np.array(xfB[:2])
    sep = float(np.linalg.norm(pB - pA)) - sA.radius - sB.radius
    if ch.gt(sep):
        return answer("separate")
    return answer("touching", G.MANIFOLD_CIRCLES, lp=(0.0, 0.0), pts=[(pB, 0, sep)])


def ref_poly_circle(ch, sA, xfA, sB, xfB, tol):
    """Face of largest separation (early out when any face separates by more than the radius); the centre inside the
    polygon (separation < b2_epsilon), or in the Voronoi region of the face's first vertex, its second vertex, or the face."""
    cw = np.array(xfB[:2])
    c = G.apply_t(xfA, cw[None])[0]
    V, N = sA.pts, sA.normals
    R = sA.radius + sB.radius
    s = ((c - V) * N).sum(1)
    i, separation = 0, -np.inf
    for j in range(len(V)):
        if ch.gt(s[j] - R):
            return answer("separate")
        if ch.gt(s[j] - separation):
            i, separation = j, s[j]
    v1, v2 = V[i], V[(i + 1) % len(V)]
    mid = 0.5 * (v1 + v2)
    L = float(np.linalg.norm(v2 - v1))
    if ch.lt(separation - G.EPS):
        return answer("inside", G.MANIFOLD_FACE_A, N[i], mid, 4 * G.EPS + tol / L, [(cw, 0, separation - R)])
    for name, v, u in (("vertex1", v1, float((c - v1) @ (v2 - v1)) / L), ("vertex2", v2, float((c - v2) @ (v1 - v2)) / L)):
        if ch.le(u):
            n, d = unit(c - v)
            if ch.gt(d - R):
                return answer(name + ", separate")
            return answer(name, G.MANIFOLD_FACE_A, n, v, 4 * G.EPS + tol / d if d > 0 else np.inf, [(cw, 0, d - R)])
    sf = float((c - mid) @ N[i])
    if ch.gt(sf - R):
        return answer("face, separate")
    return answer("face", G.MANIFOLD_FACE_A, N[i], mid, 4 * G.EPS + tol / L, [(cw, 0, sf - R)])


def ref_edge_circle(ch, sA, xfA, sB, xfB, tol):
    """Region A / B / AB of the segment.  A vertex region with a ghost vertex belongs to the neighbouring edge when the
    centre projects strictly inside that edge's span (the neighbour's face region), and then this edge reports nothing.
    At a convex corner, where the centre is in both edges' vertex regions, both edges report the shared vertex."""
    cw = np.array(xfB[:2])
    Q = G.apply_t(xfA, cw[None])[0]
    A, B = sA.pts
    e, L = unit(B - A)
    R = sA.radius + sB.radius
    for name, P, along, ghost, index in (("A", A, float(e @ (Q - A)), sA.ghost0, 0), ("B", B, float(e @ (B - Q)), sA.ghost3, 1)):
        if ch.le(along):
            d = float(np.linalg.norm(Q - P))
            if ch.gt(d - R):
                return answer("separate")
            if ghost is not None:
                g, _ = unit(P - ghost if index == 0 else ghost - P)
                if ch.gt(float(g @ (P - Q)) if index == 0 else float(g @ (Q - P))):
                    return answer("region %s ghost-rejected" % name)
            return answer("region " + name, G.MANIFOLD_CIRCLES, lp=P, pts=[(cw, G.make_id(index, 0, 0, 0), d - R)])
    P = A + float(e @ (Q - A)) * e
    if ch.gt(float(np.linalg.norm(Q - P)) - R):
        return answer("separate")
    n = np.array([-e[1], e[0]])
    if ch.lt(float(n @ (Q - A))):
        n = -n
    return answer("region AB", G.MANIFOLD_FACE_A, n, A, 4 * G.EPS + tol / L, [(cw, G.make_id(0, 0, 1, 0), float(n @ (Q - A)) - R)])


def poly_max_separation(P1, xf1, P2, xf2):
    """Per face of polygon 1: the smallest separation of polygon 2's vertices from it (float64, world frame)."""
    V1, N1 = G.apply(xf1, P1.pts), P1.normals @ G.rot(xf1).T
    V2 = G.apply(xf2, P2.pts)
    return np.array([float(((V2 - V1[i]) @ N1[i]).min()) for i in range(len(V1))])


def ref_poly_poly(ch, sA, xfA, sB, xfB, tol):
    """b2CollidePolygons: largest separation both ways against the total radius; B's face is the reference only if its
    separation exceeds A's by k_tol; the incident edge is the most anti-parallel one; its segment is clipped to the
    reference face's side planes (widened by the total radius) and keeps the points within the total radius."""
    tR = sA.radius + sB.radius

    def max_separation(P1, xf1, P2, xf2):
        best, index = -np.inf, 0
        for i, s in enumerate(poly_max_separation(P1, xf1, P2, xf2)):
            if ch.gt(s - best):
                best, index = s, i
        return best, index

    sa, ea = max_separation(sA, xfA, sB, xfB)
    if ch.gt(sa - tR):
        return answer("separate")
    sb, eb = max_separation(sB, xfB, sA, xfA)
    if ch.gt(sb - tR):
        return answer("separate")
    flip = ch.gt(sb - sa - G.K_TOL)
    P1, xf1, P2, xf2, e1 = (sB, xfB, sA, xfA, eb) if flip else (sA, xfA, sB, xfB, ea)
    label = "reference face %s" % ("B" if flip else "A")
    n1 = G.rot(xf1) @ P1.normals[e1]
    dots = (P2.normals @ G.rot(xf2).T) @ n1
    j, best = 0, np.inf
    for i, d in enumerate(dots):
        if ch.lt(d - best):
            j, best = i, d
    V1, V2 = G.apply(xf1, P1.pts), G.apply(xf2, P2.pts)
    j2, i2 = (j + 1) % len(V2), (e1 + 1) % len(V1)
    inc = [(V2[j], G.make_id(e1, j, 1, 0)), (V2[j2], G.make_id(e1, j2, 1, 0))]
    pts, _ = G.clip_face(ch, V1[e1], V1[i2], e1, i2, inc, tR)
    L = float(np.linalg.norm(P1.pts[i2] - P1.pts[e1]))
    return answer(label, G.MANIFOLD_FACE_B if flip else G.MANIFOLD_FACE_A, P1.normals[e1], 0.5 * (P1.pts[e1] + P1.pts[i2]),
                  4 * G.EPS + tol / L, [(p, G.swap_id(pid) if flip else pid, s - tR) for p, pid, s in pts])


def ref_edge_poly(ch, sA, xfA, sB, xfB, tol):
    """b2EPCollider from its definition (SURVEY.md B.5.2): front side and normal cone from the ghost vertices, edge
    axis, polygon axis with the adjacency filter, the 0.98 * s + 0.001 hysteresis between them, reference face, clip
    (side planes not widened)."""
    radius = 2.0 * G.POLY_RADIUS
    VB = G.apply_t(xfA, G.apply(xfB, sB.pts))
    NB = sB.normals @ G.rot(xfB).T @ G.rot(xfA)
    c = G.apply_t(xfA, G.apply(xfB, sB.centroid[None]))[0]
    v1, v2 = sA.pts
    e1, _ = unit(v2 - v1)
    n1 = np.array([e1[1], -e1[0]])
    f1 = ch.ge(float(n1 @ (c - v1)))
    has0, has3 = sA.ghost0 is not None, sA.ghost3 is not None
    if has0:
        e0, _ = unit(v1 - sA.ghost0)
        n0 = np.array([e0[1], -e0[0]])
        convex1 = ch.ge(float(e0[0] * e1[1] - e0[1] * e1[0]))
        f0 = ch.ge(float(n0 @ (c - sA.ghost0)))
    if has3:
        e2, _ = unit(sA.ghost3 - v2)
        n2 = np.array([e2[1], -e2[0]])
        convex2 = ch.gt(float(e1[0] * e2[1] - e1[1] * e2[0]))
        f2 = ch.ge(float(n2 @ (c - v2)))
    if has0 and has3:
        if convex1 and convex2:
            front = f0 or f1 or f2
            lim = (n0, n2) if front else (-n1, -n1)
        elif convex1:
            front = f0 or (f1 and f2)
            lim = (n0, n1) if front else (-n2, -n1)
        elif convex2:
            front = f2 or (f0 and f1)
            lim = (n1, n2) if front else (-n1, -n0)
        else:
            front = f0 and f1 and f2
            lim = (n1, n1) if front else (-n2, -n0)
        label = "ghosts 0+3, %s/%s" % ("convex" if convex1 else "concave", "convex" if convex2 else "concave")
    elif has0:
        front = (f0 or f1) if convex1 else (f0 and f1)
        lim = ((n0 if convex1 else n1), -n1) if front else (n1, (-n1 if convex1 else -n0))
        label = "ghost 0, %s" % ("convex" if convex1 else "concave")
    elif has3:
        front = (f1 or f2) if convex2 else (f1 and f2)
        lim = (-n1, (n2 if convex2 else n1)) if front else ((-n1 if convex2 else -n2), n1)
        label = "ghost 3, %s" % ("convex" if convex2 else "concave")
    else:
        front = f1
        lim = (-n1, -n1) if front else (n1, n1)
        label = "no ghosts"
    labels = ["%s, %s" % (label, "front" if front else "back")]
    normal = n1 if front else -n1
    lower, upper = lim
    if ch.gt(float(((VB - v1) @ normal).min()) - radius):
        return answer(labels + ["separate"])
    edge_sep = float(((VB - v1) @ normal).min())
    perp = np.array([-normal[1], normal[0]])
    poly_idx, poly_sep = -1, -np.inf
    for i in range(len(VB)):
        n = -NB[i]
        s = min(float(n @ (VB[i] - v1)), float(n @ (VB[i] - v2)))
        if ch.gt(s - radius):
            return answer(labels + ["separate"])
        lim_i = upper if ch.ge(float(n @ perp)) else lower
        if ch.lt(float((n - lim_i) @ normal) + G.ANGULAR_SLOP):
            continue
        if ch.gt(s - poly_sep):
            poly_idx, poly_sep = i, s
    use_poly = poly_idx >= 0 and ch.gt(poly_sep - (0.98 * edge_sep + 0.001))
    labels.append("polygon axis" if use_poly else "edge axis")
    if not use_poly and poly_idx >= 0 and poly_sep > edge_sep:
        labels.append("hysteresis keeps the edge axis")
    if not use_poly:
        dots = NB @ normal
        j, best = 0, dots[0]
        for i in range(1, len(VB)):
            if ch.lt(dots[i] - best):
                j, best = i, dots[i]
        j2 = (j + 1) % len(VB)
        inc = [(VB[j], G.make_id(0, j, 1, 0)), (VB[j2], G.make_id(0, j2, 1, 0))]
        rv1, rv2, ri1, ri2, rn = (v1, v2, 0, 1, n1) if front else (v2, v1, 1, 0, -n1)
        ln, lp = rn, rv1
    else:
        inc = [(v1, G.make_id(0, poly_idx, 0, 1)), (v2, G.make_id(0, poly_idx, 0, 1))]
        ri1, ri2 = poly_idx, (poly_idx + 1) % len(VB)
        rv1, rv2 = VB[ri1], VB[ri2]
        ln, lp = sB.normals[ri1], sB.pts[ri1]
    pts, _ = G.clip_face(ch, rv1, rv2, ri1, ri2, inc, radius, side=0.0)
    return answer(labels, G.MANIFOLD_FACE_B if use_poly else G.MANIFOLD_FACE_A, ln, lp, 4 * G.EPS + tol,
                  [(G.apply(xfA, p[None])[0], G.swap_id(pid) if use_poly else pid, s - radius) for p, pid, s in pts])


REFERENCES = {("circle", "circle"): ref_circle_circle, ("poly", "circle"): ref_poly_circle,
              ("edge", "circle"): ref_edge_circle, ("poly", "poly"): ref_poly_poly, ("edge", "poly"): ref_edge_poly}


def mismatch(m, a, sA, xfA, sB, xfB, tol):
    """None if the float32 manifold m is the answer a, else what differs"""
    if m["count"] != a["count"]:
        return "pointCount %d, reference %d" % (m["count"], a["count"])
    if a["count"] == 0:
        return None
    if m["type"] != a["type"]:
        return "type %d, reference %d" % (m["type"], a["type"])
    if np.abs(np.array(m["lp"]) - a["lp"]).max() > tol:
        return "local point %s, reference %s" % (m["lp"], a["lp"])
    if a["type"] != G.MANIFOLD_CIRCLES:
        ln = np.array(m["ln"])
        if np.isfinite(a["ntol"]) and abs(np.linalg.norm(ln) - 1.0) > 4 * G.EPS:
            return "|local normal| = %r" % np.linalg.norm(ln)
        if np.abs(ln - a["ln"]).max() > a["ntol"]:
            return "local normal %s, reference %s" % (ln, a["ln"])
    _, wpts, _ = G.world_manifold(m, sA, xfA, sB, xfB)
    body = xfA if m["type"] == G.MANIFOLD_FACE_B else xfB
    for k, (p, pid, sep) in enumerate(a["pts"]):
        gp = G.apply(body, np.array(m["p"][k])[None])[0]
        if np.abs(gp - p).max() > tol:
            return "point %d at %s, reference %s" % (k, gp, p)
        if m["id"][k] != pid:
            return "point %d id %#x, reference %#x" % (k, m["id"][k], pid)
        if abs(wpts[k][1] - sep) > tol:
            return "point %d separation %.9g, reference %.9g" % (k, wpts[k][1], sep)
    return None


def check_manifolds(out, cs, who):
    tallies = {}
    for k, (row, r, fam) in enumerate(zip(out, cs.rows, cs.family)):
        sA, sB = cs.shapes[r["a"]], cs.shapes[r["b"]]
        xfA, xfB = r["xf_a"], r["xf_b"]
        m = G.decode_manifold(row)
        scale = max(sA.extent, sB.extent) + max(abs(xfA[0]), abs(xfA[1]), abs(xfB[0]), abs(xfB[1]))
        tol = G.margin(scale)
        ref = REFERENCES[(sA.kind, sB.kind)]
        answers, exact = G.admissible(lambda ch: ref(ch, sA, xfA, sB, xfB, tol), tol)
        tally = tallies.setdefault(fam, Tally())
        for label in exact["labels"]:
            tally.hit(label)
        why = [mismatch(m, a, sA, xfA, sB, xfB, tol) for a in answers]
        if len(answers) > 1:
            tally.hit("near a decision boundary")
        if all(w is not None for w in why):
            raise AssertionError("%s case %d (%s: %s at %s vs %s at %s): the manifold (type %d, %d points, ln %s, lp %s, "
                                 "ids %s) is none of the %d admissible answers: %s" % (
                                     who, k, fam, sA.name, xfA, sB.name, xfB, m["type"], m["count"], m["ln"], m["lp"],
                                     [hex(i) for i in m["id"][:m["count"]]], len(answers),
                                     "; ".join("%s: %s" % ("/".join(a["labels"]), w) for a, w in zip(answers, why))))
    return tallies


@pytest.fixture(scope="module")
def collide_set():
    return collide_cases()


def oracle_probe(oracle, op, shapes, cases=None):
    _, fo = oracle.load()
    return G.run_probe(fo["probe_geometry"], fo["last_error"], op, shapes, cases)


def _merge(t, families):
    out = Tally()
    for fam in families:
        for k, v in t.get(fam, {}).items():
            out.hit(k, v)
    return out


def test_oracle_manifolds_match_the_float64_reference(oracle, collide_set):
    cs = collide_set
    out = oracle_probe(oracle, abi.KB_PROBE_COLLIDE, cs.shapes, G.pack_cases(cs.rows))
    t = check_manifolds(out, cs, "oracle")
    print("manifold coverage: %s" % {k: dict(v) for k, v in t.items()})
    # the seeded random families seldom land near a boundary; the targeted ones are built to
    families = ("circles", "poly-circle", "poly-poly", "edge-circle", "edge-poly")
    random = _merge(t, families)
    total = sum(f in families for f in cs.family)
    assert random.get("near a decision boundary", 0) < 0.02 * total, random
    assert t["circles/rA+rB"].get("near a decision boundary", 0) >= 100, t["circles/rA+rB"]
    pc = _merge(t, ("poly-circle", "poly-circle/targeted"))
    for region in ("inside", "vertex1", "vertex2", "face"):
        assert pc.get(region, 0) >= 20, "polygon-circle region %s reached %d times: %s" % (region, pc.get(region, 0), pc)
    assert t["poly-circle/targeted"].get("near a decision boundary", 0) >= 50, t["poly-circle/targeted"]
    pp = _merge(t, ("poly-poly", "poly-poly/flush", "poly-poly/vertex"))
    assert pp.get("reference face A", 0) >= 50 and pp.get("reference face B", 0) >= 50, pp
    ec = _merge(t, ("edge-circle", "edge-corner"))
    for key in ("region A", "region B", "region AB", "region A ghost-rejected", "region B ghost-rejected"):
        assert ec.get(key, 0) >= 5, "edge-circle %s reached %d times: %s" % (key, ec.get(key, 0), ec)
    ep = _merge(t, ("edge-poly", "edge-corner"))
    # a chain round a rectangle turns the same way at every corner: convex/concave mixes cannot occur on the table
    for key in [g + ", " + c + ", " + fb for g in ("ghost 0", "ghost 3") for c in ("convex", "concave") for fb in ("front", "back")] + \
               ["ghosts 0+3, %s, %s" % (c, fb) for c in ("convex/convex", "concave/concave") for fb in ("front", "back")] + \
               ["edge axis", "polygon axis", "hysteresis keeps the edge axis"]:
        assert ep.get(key, 0) >= 3, "edge-polygon %s reached %d times: %s" % (key, ep.get(key, 0), ep)


# ------------------------------------------------------------------------------------------------ distance
def distance_cases():
    rng = np.random.default_rng(99)
    cs = Cases()
    kb = G.circle_shape(KILOBOT_R, "kilobot")
    polys = [s for s in shape_set() if s.kind == "poly"]
    edges = [G.chain_edge(i, 4) for i in range(4)]
    for k in range(2000):
        sc = [40.0, 1.0][k % 2]
        kind = k % 4
        if kind == 0:
            a, b = polys[k % len(polys)], polys[(k * 5 + 3) % len(polys)]
        elif kind == 1:
            a, b = polys[k % len(polys)], kb
        elif kind == 2:
            a, b = edges[k % 4], kb
        else:
            a, b = edges[k % 4], polys[k % len(polys)]
        xa = (0.0, 0.0, 0.0, 1.0) if a.kind == "edge" else G.xf_from_angle(rng.uniform(-sc, sc), rng.uniform(-sc, sc),
                                                                              rng.uniform(-np.pi, np.pi))
        anchor = G.apply(xa, a.pts)[int(rng.integers(len(a.pts)))]
        q = anchor + rng.uniform(-1.5, 1.5, 2) * (b.extent + 0.5)
        cs.add("distance", a, xa, b, G.xf_from_angle(q[0], q[1], rng.uniform(-np.pi, np.pi)))
    return cs


def test_oracle_distance_matches_the_float64_core_distance(oracle):
    cs = distance_cases()
    out = oracle_probe(oracle, abi.KB_PROBE_DISTANCE, cs.shapes, G.pack_cases(cs.rows))
    d = G.f32(out[:, 0]).astype(np.float64)
    n_overlap = 0
    for k, r in enumerate(cs.rows):
        sA, sB = cs.shapes[r["a"]], cs.shapes[r["b"]]
        ref = G.core_distance(G.world_core(sA, r["xf_a"]), G.world_core(sB, r["xf_b"]))
        scale = max(sA.extent, sB.extent) + max(np.abs(r["xf_a"][:2]).max(), np.abs(r["xf_b"][:2]).max())
        n_overlap += ref == 0.0
        assert abs(d[k] - ref) <= G.margin(scale), "oracle distance case %d (%s at %s vs %s at %s): %.9g, float64 %.9g" % (
            k, sA.name, r["xf_a"], sB.name, r["xf_b"], d[k], ref)
        assert 1 <= out[k, 1] <= 3, k
    print("distance: %d cases, %d overlapping" % (len(cs.rows), n_overlap))
    assert 100 <= n_overlap <= len(cs.rows) - 100


# ------------------------------------------------------------------------------------------------ time of impact
def sweep_of(lc, c0, c, a0, a):
    return (lc[0], lc[1], c0[0], c0[1], c[0], c[1], a0, a)


def toi_cases():
    """Table edges (the table's sweep: no motion, no rotation, fixedRot) against
      toi/circle        a kilobot or a circle object moving towards / along the wall, up to several radii per step, and
                        turning (angles beyond +-2 pi): centred on its body, so fixedRot = 1 as the step kernels set it;
      toi/graze         a kilobot sliding parallel to the wall at about contact distance, turning, fixedRot = 1;
      toi/circle-offset a circle whose body's centre of mass is off its centre, turning: the rotation moves the circle,
                        so fixedRot = 0 (the control: here the shortcut would be wrong);
      toi/polygon       rotating L-, T-, C-forms and quads, angles beyond +-2 pi."""
    rng = np.random.default_rng(31)
    cs = Cases()
    kb = G.circle_shape(KILOBOT_R, "kilobot")
    big = G.circle_shape(1.25, "circle1.25")
    forms = [s for s in shape_set() if s.kind == "poly" and s.name[:5] in ("lform", "tform", "cform", "quad.")]
    edges = [G.chain_edge(i, e) for e in (3, 4) for i in range(e)]
    table = [0.0] * 8
    for k in range(1800):
        e = edges[k % len(edges)]
        kind = k % 6
        v1, v2 = e.pts
        t = rng.uniform(-0.1, 1.1)
        base = v1 + t * (v2 - v1)
        n = np.array([(v2 - v1)[1], -(v2 - v1)[0]])
        n = n / np.linalg.norm(n)
        inward = -n
        a0 = rng.uniform(-12.0, 12.0)
        a1 = a0 + rng.uniform(-3.0, 3.0)
        if kind in (0, 1, 3):
            b = kb if kind != 1 else big
            d0 = rng.uniform(-0.2, 3.0) * b.radius + b.radius
            c0 = base + inward * d0
            c1 = c0 + rng.uniform(-5, 5, 2) * b.radius
            lc = (0.0, 0.0) if kind != 3 else rng.uniform(-0.6, 0.6, 2) * b.radius
            fixed = 1 if kind != 3 else 0
            fam = "toi/circle" if kind != 3 else "toi/circle-offset"
        elif kind == 2:
            b = kb
            c0 = base + inward * (b.radius + rng.uniform(-0.01, 0.03))
            c1 = c0 + (v2 - v1) / np.linalg.norm(v2 - v1) * rng.uniform(-3, 3)
            lc, fixed, fam = (0.0, 0.0), 1, "toi/graze"
        else:
            b = forms[k % len(forms)]
            lc = rng.uniform(-0.3, 0.3, 2)
            c0 = base + inward * rng.uniform(0.0, 2.0) * b.extent
            c1 = c0 + rng.uniform(-1.5, 1.5, 2) * b.extent
            a1 = a0 + rng.uniform(-1.5, 1.5)
            fixed, fam = 0, "toi/polygon"
        sw = tuple(float(np.float32(x)) for x in sweep_of(lc, c0, c1, a0, a1))
        cs.rows.append({"a": cs.shape(e), "b": cs.shape(b), "fixed_rot_a": 1, "fixed_rot_b": fixed,
                        "sweep_a": table, "sweep_b": sw})
        cs.family.append(fam)
    return cs


def sweep_core(shape, sw, t):
    """Core points of a shape at the times t (array) of its sweep, float64 (angle and position interpolated linearly):
    (T, n, 2)."""
    t = np.atleast_1d(np.asarray(t, np.float64))[:, None]
    lc, c0, c1, a0, a1 = np.array(sw[0:2]), np.array(sw[2:4]), np.array(sw[4:6]), sw[6], sw[7]
    a = ((1 - t) * a0 + t * a1)[:, 0]
    cs, sn = np.cos(a), np.sin(a)
    R = np.stack([np.stack([cs, -sn], -1), np.stack([sn, cs], -1)], -2)     # (T, 2, 2)
    p = (1 - t) * c0 + t * c1 - R @ lc
    return np.einsum("tij,nj->tni", R, shape.pts) + p[:, None]


def test_oracle_time_of_impact_matches_the_float64_sweep(oracle):
    """t >= 0: the float64 core distance at t is within target +- tolerance (or below target + tolerance when the sweep
    starts there, t = 0); a sweep that clearly crosses the target band returns t >= 0; one that never comes within
    target + 2 tolerance returns t < 0.  When the core shape only translates (a circle centred on its body, or no
    rotation), the distance is nowhere in [0, t) below target - tolerance: conservative advancement along a separating
    axis finds the first contact of a translating convex shape.  A rotating shape can touch the wall and leave it again
    before the returned t -- b2TimeOfImpact's contract (b2TimeOfImpact.h: "uses a swept separating axis and may miss some
    intermediate, non-tunneling collisions") allows that, so those cases are counted, not failed.  The distance is
    sampled on a 1025-point grid and its minimum bounded below by the sweep's largest point speed (grid error <=
    speed * h / 2)."""
    cs = toi_cases()
    out = oracle_probe(oracle, abi.KB_PROBE_TOI, cs.shapes, G.pack_cases(cs.rows))
    tt = G.f32(out[:, 0]).astype(np.float64)
    grid = np.linspace(0.0, 1.0, 1025)
    tally = Tally()
    for k, r in enumerate(cs.rows):
        sA, sB = cs.shapes[r["a"]], cs.shapes[r["b"]]
        target = max(G.SLOP, float(np.float32(sA.radius + sB.radius) - np.float32(3.0) * np.float32(G.SLOP)))
        tol = 0.25 * G.SLOP
        sw = r["sweep_b"]
        ext = float(np.abs(sB.pts - np.array(sw[:2])).max(initial=0.0) + np.linalg.norm(sw[:2]))
        scale = max(np.abs(sw[2:6]).max(), 25.0) + (abs(sw[6]) + abs(sw[7])) * ext
        m = G.margin(scale)
        core_a = sA.pts
        dist = G.core_distance_batch(np.broadcast_to(core_a, (len(grid),) + core_a.shape), sweep_core(sB, sw, grid))
        speed = float(np.linalg.norm(np.array(sw[4:6]) - np.array(sw[2:4]))) + abs(sw[7] - sw[6]) * ext
        slack = speed * (grid[1] - grid[0]) / 2 + m
        where = "oracle TOI case %d (%s, %s, sweep %s, state %d): t = %r" % (k, cs.family[k], sB.name, sw, out[k, 3], tt[k])
        state = int(out[k, 3])
        tally.hit({1: "failed", 2: "overlapped", 3: "touching", 4: "separated"}.get(state, "unknown"))
        if tt[k] >= 0:
            tally.hit("touching at t = 0" if tt[k] == 0 else "touching at t > 0")
            d_t = G.core_distance(core_a, sweep_core(sB, sw, tt[k])[0])
            if tt[k] == 0:
                assert -m < d_t < target + tol + m, "%s: distance %.9g at t = 0" % (where, d_t)
            else:
                assert target - tol - m <= d_t <= target + tol + m, "%s: distance %.9g at t, band %.9g +- %.9g" % (
                    where, d_t, target, tol)
                early = dist[grid < tt[k]].min(initial=np.inf)
                translating = sw[6] == sw[7] or (sB.kind == "circle" and sw[0] == 0.0 and sw[1] == 0.0)
                if translating:
                    assert early >= target - tol - slack, "%s: distance %.9g before t" % (where, early)
                elif early < target - tol - slack:
                    tally.hit("rotating: an intermediate contact before t")
        else:
            if dist[0] > target + 2 * tol + m and (dist < target - 2 * tol - slack).any():
                first = grid[np.argmax(dist < target - 2 * tol - slack)]
                # a sweep that tunnels through the band within one grid step of the start is not "clear"
                raise AssertionError("%s: the float64 distance falls from %.9g to below %.9g by t = %.4f" % (
                    where, dist[0], target - 2 * tol, first))
            if dist.min() - slack >= target + 2 * tol:
                tally.hit("never within the band")
    print("TOI outcomes: %s" % dict(tally))
    for key in ("touching at t = 0", "touching at t > 0", "separated", "never within the band", "overlapped"):
        assert tally.get(key, 0) >= 10, "TOI outcome %s reached %d times: %s" % (key, tally.get(key, 0), dict(tally))


# ------------------------------------------------------------------------------------------------ device (GPU)
def _same_bits(a, b):
    fa, fb = G.f32(a), G.f32(b)
    return (a == b) | (np.isnan(fa) & np.isnan(fb))


def defined_manifold(out):
    """The words of a manifold that are defined: pointCount, and type, local normal / point and the first pointCount
    points when it has points.  (Both routines may leave partial results in the rest, which nothing reads.)"""
    out = out[:, :12].copy()
    count = out[:, 1]
    out[count == 0, 0] = 0
    out[count == 0, 2:] = 0
    out[count < 2, 9:12] = 0
    return out


def _assert_same(dev, ora, words, what, cs):
    same = _same_bits(dev[:, :words], ora[:, :words])
    bad = np.argwhere(~same)
    if bad.size:
        k, w = bad[0]
        r = cs.rows[k]
        raise AssertionError("%s: device and oracle differ in case %d (%s: %s vs %s), word %d: %#x vs %#x (%d cases differ)" % (
            what, k, cs.family[k], cs.shapes[r["a"]].name, cs.shapes[r["b"]].name, w, dev[k, w], ora[k, w],
            len(np.unique(bad[:, 0]))))


@pytest.mark.gpu
def test_device_matches_the_oracle_bit_for_bit(oracle, native, collide_set):
    """Every output of every case: the defined words of the manifolds, distances and simplex counts, times of impact."""
    fn, err = native._fn["probe_geometry"], native._fn["last_error"]
    for op, cs, words, what in ((abi.KB_PROBE_COLLIDE, collide_set, 12, "collide"),
                                (abi.KB_PROBE_DISTANCE, distance_cases(), 2, "distance"),
                                (abi.KB_PROBE_TOI, toi_cases(), 1, "time of impact")):
        cases = G.pack_cases(cs.rows)
        dev = G.run_probe(fn, err, op, cs.shapes, cases)
        ora = oracle_probe(oracle, op, cs.shapes, cases)
        if op == abi.KB_PROBE_COLLIDE:
            dev, ora = defined_manifold(dev), defined_manifold(ora)
        _assert_same(dev, ora, words, what, cs)


@pytest.mark.gpu
def test_device_toi_specialisations_are_the_generic_routine(native):
    """time_of_impact_edge_circle (DProxyEdge / DProxyCircle) is bit-identical to time_of_impact on every edge-circle
    case, turning circles and circles off their body's centre included.  A sweep with fixedRot = 1 -- the table, and a
    turning circle centred on its body, as the step kernels set it -- is bit-identical to the same sweep rotated.  The
    control shows that the comparison can fail: set on a circle off its body's centre, the shortcut ignores the turn that
    moves the circle and changes the result."""
    fn, err = native._fn["probe_geometry"], native._fn["last_error"]
    cs = toi_cases()
    out = G.run_probe(fn, err, abi.KB_PROBE_TOI, cs.shapes, G.pack_cases(cs.rows))
    circ = np.array([cs.shapes[r["b"]].kind == "circle" for r in cs.rows])
    assert circ.sum() > 800
    assert np.array_equal(out[circ, 1], out[circ, 0]), "edge-circle specialisation differs in case %d" % (
        np.nonzero(circ & (out[:, 1] != out[:, 0]))[0][0])
    fixed = np.array([r["fixed_rot_a"] or r["fixed_rot_b"] for r in cs.rows], bool)
    turning = np.array([r["fixed_rot_b"] == 1 and r["sweep_b"][6] != r["sweep_b"][7] for r in cs.rows], bool)
    assert turning.sum() > 500 and (turning & (G.f32(out[:, 0]) >= 0)).sum() > 100
    assert np.array_equal(out[fixed, 2], out[fixed, 0]), "fixedRot changes the result of case %d" % (
        np.nonzero(fixed & (out[:, 2] != out[:, 0]))[0][0])
    offset = [dict(r, fixed_rot_b=1) for r, f in zip(cs.rows, cs.family) if f == "toi/circle-offset"]
    wrong = G.run_probe(fn, err, abi.KB_PROBE_TOI, cs.shapes, G.pack_cases(offset))
    differ = int((wrong[:, 0] != wrong[:, 2]).sum())
    print("fixedRot on %d off-centre circles: %d results change" % (len(offset), differ))
    assert differ >= 50
