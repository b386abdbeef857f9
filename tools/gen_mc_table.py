"""Generate dynamicfusion_b200/csrc/mc_table.h, the marching-cubes case table of the mesh extraction (dfusion.h df_extract_mesh).

    python tools/gen_mc_table.py          # rewrites the header
    python tools/gen_mc_table.py --check  # exit 1 if the committed header differs from what this script writes

The table is derived, not typed in.  Conventions (shared with csrc/extract.cu and oracle/orc_mesh.c):
  corner c = 0..7 sits at (c & 1, (c >> 1) & 1, (c >> 2) & 1) from the cell's min corner; bit c of a case is set iff corner c is
  INSIDE (F < 0);
  edge e = 4 * axis + k runs from offset o(e) along +axis, with o = (0, k & 1, k >> 1) for axis 0, (k & 1, 0, k >> 1) for axis 1,
  (k & 1, k >> 1, 0) for axis 2 -- so the edge's vertex is keyed 3 * (linear index of min corner + o) + axis.
For every case the generator
  1. on each of the six faces joins the crossing edges into segments, from the face's four signs alone: two crossings make one segment;
     four (an ambiguous face: the inside corners on a diagonal) make two segments, each cutting off one inside corner, so the inside
     corners are always separated.  Neighbouring cells therefore agree on every shared face and the mesh has no cracks;
  2. directs every segment so that the surface is counter-clockwise seen from the outside (F > 0): the face normal then points from
     the inside corners to the outside ones, along the TSDF gradient;
  3. chains the directed segments into closed polygons (each crossing edge has one segment arriving and one leaving) and
     fan-triangulates each one from an apex whose diagonals do not lie in a cube face (a diagonal in a face could coincide with the
     neighbouring cell's and give that mesh edge four triangles).
Polygons are emitted in order of their smallest edge index, each starting from its apex.
"""
from __future__ import annotations

import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
HEADER = ROOT / "dynamicfusion_b200" / "csrc" / "mc_table.h"


def corner_pos(c: int):
    return (c & 1, (c >> 1) & 1, (c >> 2) & 1)


def edge_offset(e: int):
    axis, k = e >> 2, e & 3
    return [(0, k & 1, k >> 1), (k & 1, 0, k >> 1), (k & 1, k >> 1, 0)][axis], axis


def edge_corners(e: int):
    o, axis = edge_offset(e)
    hi = list(o)
    hi[axis] += 1
    idx = lambda p: p[0] | (p[1] << 1) | (p[2] << 2)
    return idx(o), idx(hi)


def edge_mid(e: int):
    o, axis = edge_offset(e)
    m = [float(v) for v in o]
    m[axis] += 0.5
    return m


def faces():
    """(axis, side, outward normal, corners, edges) of the six cube faces"""
    out = []
    for a in range(3):
        for s in range(2):
            f = [0, 0, 0]
            f[a] = 2 * s - 1
            cs = [c for c in range(8) if corner_pos(c)[a] == s]
            es = [e for e in range(12) if all(corner_pos(c)[a] == s for c in edge_corners(e))]
            out.append((a, s, f, cs, es))
    return out


FACES = faces()


def _sub(a, b):
    return [a[i] - b[i] for i in range(3)]


def _cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def _dot(a, b):
    return sum(a[i] * b[i] for i in range(3))


def share_face(e1: int, e2: int) -> bool:
    return any(e1 in es and e2 in es for (_, _, _, _, es) in FACES)


def crossing_edges(case: int):
    return [e for e in range(12) if ((case >> edge_corners(e)[0]) & 1) != ((case >> edge_corners(e)[1]) & 1)]


def face_segments(case: int):
    """directed segments (from edge, to edge, face index) of every face, decided from that face's signs alone"""
    inside = lambda c: (case >> c) & 1
    segs = []
    for fi, (a, s, f, cs, es) in enumerate(FACES):
        cross = [e for e in es if inside(edge_corners(e)[0]) != inside(edge_corners(e)[1])]
        pairs = []
        if len(cross) == 2:
            ref = [c for c in cs if inside(c)][0]                  # every inside corner of the face lies on the same side
            pairs.append((cross[0], cross[1], ref))
        elif len(cross) == 4:                                      # ambiguous face: cut off each inside corner on its own
            for c in cs:
                if inside(c):
                    inc = [e for e in cross if c in edge_corners(e)]
                    assert len(inc) == 2
                    pairs.append((inc[0], inc[1], c))
        else:
            assert not cross
        for e1, e2, ref in pairs:
            a_, b_ = edge_mid(e1), edge_mid(e2)
            m = [(a_[i] + b_[i]) / 2 for i in range(3)]
            side = _dot(f, _cross(_sub(b_, a_), _sub(m, list(corner_pos(ref)))))
            assert side != 0
            segs.append((e1, e2, fi) if side > 0 else (e2, e1, fi))
    return segs


def polygons(case: int):
    segs = face_segments(case)
    nxt = {}
    for e1, e2, _ in segs:
        assert e1 not in nxt, (case, "two segments leave one edge")
        nxt[e1] = e2
    assert sorted(nxt) == sorted(nxt.values()) == crossing_edges(case), case
    polys, seen = [], set()
    for start in sorted(nxt):
        if start in seen:
            continue
        cyc = [start]
        while nxt[cyc[-1]] != start:
            cyc.append(nxt[cyc[-1]])
        seen.update(cyc)
        polys.append(cyc)
    return polys


def fan(poly):
    """rotate the polygon to the first apex (in polygon order) none of whose diagonals joins two edges of one face"""
    n = len(poly)
    for r in range(n):
        p = poly[r:] + poly[:r]
        if all(not share_face(p[0], p[i]) for i in range(2, n - 1)):
            return [(p[0], p[i], p[i + 1]) for i in range(1, n - 1)]
    raise AssertionError(f"polygon {poly}: every apex has a diagonal in a face")


def build_table():
    """list of 256 lists of triangles (edge index triples)"""
    return [[t for poly in polygons(case) for t in fan(poly)] for case in range(256)]


def render(table) -> str:
    maxt = max(len(t) for t in table)
    lines = [
        "/* mc_table.h -- GENERATED by tools/gen_mc_table.py; do not edit.  Marching-cubes case table of the mesh extraction",
        " * (include/dfusion.h df_extract_mesh; the conventions are in the generator's docstring).  Shared by csrc/extract.cu and",
        " * oracle/orc_mesh.c: define DF_MC_CONST before including it to place the arrays (default: static const). */",
        "#ifndef DF_MC_TABLE_H",
        "#define DF_MC_TABLE_H",
        "#ifndef DF_MC_CONST",
        "#define DF_MC_CONST static const",
        "#endif",
        "",
        f"#define DF_MC_MAX_TRIS {maxt}    /* most triangles one cell emits */",
        "",
        "/* edge e: offset (dx, dy, dz) of its lower endpoint from the cell's min corner, then its axis */",
        "DF_MC_CONST signed char df_mc_edges[12][4] = {",
    ]
    lines.append("    " + ", ".join("{%d, %d, %d, %d}" % (*edge_offset(e)[0], edge_offset(e)[1]) for e in range(12)))
    lines.append("};")
    lines.append("")
    lines.append("/* triangles of case c (bit i = corner i inside) */")
    lines.append("DF_MC_CONST unsigned char df_mc_ntri[256] = {")
    for r in range(0, 256, 32):
        lines.append("    " + ", ".join(str(len(table[c])) for c in range(r, r + 32)) + ",")
    lines.append("};")
    lines.append("")
    lines.append("/* their edges, three per triangle, counter-clockwise seen from the outside (F > 0); -1 pads */")
    lines.append(f"DF_MC_CONST signed char df_mc_tris[256][{3 * maxt}] = {{")
    for c in range(256):
        flat = [e for t in table[c] for e in t] + [-1] * (3 * (maxt - len(table[c])))
        lines.append("    {" + ", ".join(str(v) for v in flat) + "},")
    lines.append("};")
    lines.append("")
    lines.append("#endif")
    return "\n".join(lines) + "\n"


def main(argv) -> int:
    table = build_table()
    text = render(table)
    assert max(len(t) for t in table) <= 5, "at most 5 triangles per cell: one cell's output, and the row width of df_mc_tris"
    if "--check" in argv:
        same = HEADER.exists() and HEADER.read_text() == text
        print("mc_table.h is up to date" if same else "mc_table.h differs from the generator's output")
        return 0 if same else 1
    HEADER.write_text(text)
    print(f"wrote {HEADER} ({sum(len(t) for t in table)} triangles over 256 cases, at most {max(len(t) for t in table)} per cell)")
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
