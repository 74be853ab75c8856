"""Generate mc_table.h, the marching-cubes case table of iso_surface.cu and of the CPU oracle, from a rule.

    python genre_shapehd_b200/csrc/gen_mc_table.py            # rewrites mc_table.h next to this file
    python genre_shapehd_b200/csrc/gen_mc_table.py --stdout   # prints it instead

The table is derived, not transcribed from any library:
  1. on each of the 6 cube faces, find the crossed edges (0, 2 or 4);
  2. join them into segments; on an ambiguous face (two diagonal in-corners) always cut off each in-corner separately,
     a rule that reads only that face's four corner bits, so the two cells sharing a face agree and the mesh has no cracks;
  3. orient each segment so that the triangle normal will point from the "> level" side to the "<= level" side, and chain
     the segments into closed loops;
  4. fan-triangulate each loop from its lowest-numbered edge.
Unlike Lewiner's MC33 tables, cube-interior ambiguities are not resolved and no cell-centre vertex is added.
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "mc_table.h")


def corner_offset(c):
    """corner c of a cell -> (di, dj, dk); bit c of the case index is that corner's `value > level`"""
    return ((c >> 2) & 1, (c >> 1) & 1, c & 1)


def corner_index(o):
    return (o[0] << 2) | (o[1] << 1) | o[2]


def _other_axes(a):
    return [b for b in range(3) if b != a]


def edge_owner(e):
    """edge e -> (owner corner offset, axis a): the edge runs from the owner to owner + e_a"""
    a, r = divmod(e, 4)
    b, c = _other_axes(a)
    o = [0, 0, 0]
    o[b], o[c] = r >> 1, r & 1
    return tuple(o), a


def edge_corners(e):
    o, a = edge_owner(e)
    q = list(o)
    q[a] = 1
    return corner_index(o), corner_index(tuple(q))


def edge_midpoint(e):
    o, a = edge_owner(e)
    m = [float(x) for x in o]
    m[a] = 0.5
    return tuple(m)


FACES = [(a, v) for a in range(3) for v in (0, 1)]  # face (a, v): the corners whose coordinate a equals v


def face_corners_cyclic(face):
    """the face's 4 corners in cyclic order"""
    a, v = face
    b, c = _other_axes(a)
    out = []
    for sb, sc in ((0, 0), (1, 0), (1, 1), (0, 1)):
        o = [0, 0, 0]
        o[a], o[b], o[c] = v, sb, sc
        out.append(corner_index(tuple(o)))
    return out


def edge_between(c0, c1):
    for e in range(12):
        if set(edge_corners(e)) == {c0, c1}:
            return e
    raise AssertionError((c0, c1))


def face_segments(case, face):
    """the face rule: unordered pairs of crossed edges, from the face's own four corner bits only"""
    cyc = face_corners_cyclic(face)
    inside = [(case >> c) & 1 for c in cyc]
    edges = [edge_between(cyc[t], cyc[(t + 1) % 4]) for t in range(4)]
    crossed = [edges[t] for t in range(4) if inside[t] != inside[(t + 1) % 4]]
    if len(crossed) == 0:
        return []
    if len(crossed) == 2:
        return [tuple(crossed)]
    assert len(crossed) == 4
    # ambiguous face: cut off each in-corner separately (the two face edges at an in-corner are both crossed)
    segs = []
    for t in range(4):
        if inside[t]:
            segs.append((edges[(t - 1) % 4], edges[t]))
    assert len(segs) == 2
    return segs


def _sub(p, q):
    return tuple(x - y for x, y in zip(p, q))


def _cross(p, q):
    return (p[1] * q[2] - p[2] * q[1], p[2] * q[0] - p[0] * q[2], p[0] * q[1] - p[1] * q[0])


def _dot(p, q):
    return sum(x * y for x, y in zip(p, q))


def orient_segment(case, face, seg):
    """order (P, Q) so that the surface normal (pointing from the in-side to the out-side) crossed with Q - P points into the
    cube: then the loop runs counter-clockwise seen from the normal's tip, and fans along it have right-hand normals that point
    from the '> level' side to the '<= level' side"""
    a, v = face
    n_f = [0.0, 0.0, 0.0]
    n_f[a] = 1.0 if v else -1.0
    p, q = seg
    P, Q = edge_midpoint(p), edge_midpoint(q)
    T = _sub(Q, P)
    # the in-endpoints of both crossed edges lie on the in-side of the segment
    ins = []
    for e in seg:
        c0, c1 = edge_corners(e)
        ins.append(corner_offset(c0 if (case >> c0) & 1 else c1))
    mid = tuple((x + y) / 2 for x, y in zip(P, Q))
    inpt = tuple((x + y) / 2 for x, y in zip(*ins))
    m = _sub(mid, inpt)                      # from the in-side towards the segment
    s = _dot(_cross(m, T), n_f)
    assert s != 0
    return (p, q) if s < 0 else (q, p)


def case_loops(case):
    nxt = {}
    for face in FACES:
        for seg in face_segments(case, face):
            p, q = orient_segment(case, face, seg)
            assert p not in nxt, "two segments leave edge %d in case %d" % (p, case)
            nxt[p] = q
    assert sorted(nxt) == sorted(nxt.values()), "open chain in case %d" % case
    loops, seen = [], set()
    for start in sorted(nxt):
        if start in seen:
            continue
        loop, e = [], start
        while e not in seen:
            seen.add(e)
            loop.append(e)
            e = nxt[e]
        assert e == start
        loops.append(loop)
    return loops


def case_triangles(case):
    tris = []
    for loop in case_loops(case):
        r = loop.index(min(loop))
        loop = loop[r:] + loop[:r]           # start at the lowest-numbered edge
        for t in range(1, len(loop) - 1):
            tris.append((loop[0], loop[t], loop[t + 1]))
    return tris


def crossed_edges(case):
    return sorted(e for e in range(12) if ((case >> edge_corners(e)[0]) & 1) != ((case >> edge_corners(e)[1]) & 1))


def build_table():
    return [case_triangles(c) for c in range(256)]


def render(table):
    max_tris = max(len(t) for t in table)
    assert max_tris == max(len(crossed_edges(c)) - 2 * len(case_loops(c)) for c in range(256) if crossed_edges(c))
    lines = [
        "/* mc_table.h -- marching-cubes case table.  GENERATED by gen_mc_table.py; do not edit by hand.",
        " *",
        " * Cell corner c (0..7) sits at offset (di, dj, dk) = ((c >> 2) & 1, (c >> 1) & 1, c & 1) from the cell's lowest point",
        " * (i, j, k) of a C-order [D][H][W] volume.  Bit c of the case index is set when that corner's value > level (NaN: not set).",
        " * Edge e (0..11) runs along axis a = e / 4 (0 = i, 1 = j, 2 = k) from its owner corner; with (b, c) the other two axes in",
        " * increasing order, the owner's offset along b is (e % 4) >> 1 and along c is e & 1 (its offset along a is 0):",
        " *     e  0..3   along i, owner (0, dj, dk) with (dj, dk) = (0,0) (0,1) (1,0) (1,1)",
        " *     e  4..7   along j, owner (di, 0, dk) with (di, dk) = (0,0) (0,1) (1,0) (1,1)",
        " *     e  8..11  along k, owner (di, dj, 0) with (di, dj) = (0,0) (0,1) (1,0) (1,1)",
        " * Triangles (e0, e1, e2) have right-hand normals pointing from the '> level' side to the '<= level' side.",
        " * Ambiguous faces always cut off each in-corner separately; cube-interior ambiguities are not resolved (no MC33).",
        " */",
        "#ifndef GENRE_B200_MC_TABLE_H",
        "#define GENRE_B200_MC_TABLE_H",
        "",
        "#define MC_MAX_TRIS %d" % max_tris,
        "",
        "/* storage of the two arrays; a CUDA includer defines it as `static __device__ const` to get device copies */",
        "#ifndef MC_TABLE_QUAL",
        "#define MC_TABLE_QUAL static const",
        "#endif",
        "",
        "/* triangles per case */",
        "MC_TABLE_QUAL unsigned char mc_ntri[256] = {",
    ]
    for r in range(0, 256, 32):
        lines.append("    " + ", ".join(str(len(table[c])) for c in range(r, r + 32)) + ",")
    lines += ["};", "", "/* edge triples per case, rows padded with 0 */",
              "MC_TABLE_QUAL unsigned char mc_tri[256][MC_MAX_TRIS * 3] = {"]
    for c in range(256):
        flat = [e for tri in table[c] for e in tri]
        flat += [0] * (3 * max_tris - len(flat))
        lines.append("    {" + ", ".join(str(x) for x in flat) + "},  /* %3d */" % c)
    lines += ["};", "", "#endif /* GENRE_B200_MC_TABLE_H */", ""]
    return "\n".join(lines)


def main(argv):
    text = render(build_table())
    if "--stdout" in argv:
        sys.stdout.write(text)
    else:
        with open(OUT, "w", newline="\n") as f:
            f.write(text)


if __name__ == "__main__":
    main(sys.argv[1:])
