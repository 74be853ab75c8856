"""Marching cubes without a GPU: the generated case table (against the rule it comes from), the oracle's meshes of
analytic fields (closed, oriented, right topology and volume, vertices on crossed edges), write_obj, the C ABI's argument
checks and the skimage stand-in's argument handling."""
import collections
import ctypes
import functools
import importlib.util
import os

import numpy as np
import pytest
import torch

import oracle_mesh
from conftest import REPO
from genre_shapehd_b200 import _lib, compat, postprocess
from genre_shapehd_b200.synth import iso_field

CSRC = os.path.join(REPO, "genre_shapehd_b200", "csrc")


def _gen():
    spec = importlib.util.spec_from_file_location("gen_mc_table", os.path.join(CSRC, "gen_mc_table.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


GEN = _gen()


def test_generator_reproduces_committed_header():
    with open(os.path.join(CSRC, "mc_table.h"), newline="") as f:
        committed = f.read()
    assert GEN.render(GEN.build_table()) == committed


# ---- the table against the rule, restated here without the generator's helpers ------------------------------------
def _corner(o):
    return 4 * o[0] + 2 * o[1] + o[2]


def _edges():
    """edge e -> (corner at the owner, corner at owner + e_a), numbering of mc_table.h"""
    out = []
    for e in range(12):
        a, r = divmod(e, 4)
        b, c = [x for x in range(3) if x != a]
        o = [0, 0, 0]
        o[b], o[c] = r >> 1, r & 1
        q = list(o)
        q[a] = 1
        out.append((_corner(o), _corner(q)))
    return out


EDGES = _edges()


def _crossed(case):
    return {e for e, (p, q) in enumerate(EDGES) if ((case >> p) & 1) != ((case >> q) & 1)}


def _face_rule(case, a, v):
    """segments (frozensets of two edges) on face (axis a = v): cut off each in-corner when the face is ambiguous"""
    b, c = [x for x in range(3) if x != a]
    cyc = []
    for sb, sc in ((0, 0), (1, 0), (1, 1), (0, 1)):
        o = [0, 0, 0]
        o[a], o[b], o[c] = v, sb, sc
        cyc.append(_corner(o))
    ins = [(case >> x) & 1 for x in cyc]
    side = [EDGES.index(tuple(sorted((cyc[t], cyc[(t + 1) % 4])))) for t in range(4)]   # EDGES pairs are (low, high)
    crossed = [side[t] for t in range(4) if ins[t] != ins[(t + 1) % 4]]
    if len(crossed) == 2:
        return {frozenset(crossed)}
    if len(crossed) == 4:
        return {frozenset((side[(t - 1) % 4], side[t])) for t in range(4) if ins[t]}
    return set()


def _face_of(seg):
    """the cube face both edges of a segment lie on"""
    cs = [set(EDGES[e]) for e in seg]
    common = None
    for a in range(3):
        for v in (0, 1):
            face = {x for x in range(8) if ((x >> (2 - a)) & 1) == v}
            if cs[0] <= face and cs[1] <= face:
                assert common is None
                common = (a, v)
    return common


@functools.lru_cache(maxsize=None)
def _table():
    t = GEN.build_table()
    assert len(t) == 256
    return t


@pytest.mark.parametrize("case", range(256))
def test_case_uses_exactly_the_crossed_edges(case):
    tris = _table()[case]
    used = {e for tri in tris for e in tri}
    assert used == _crossed(case)
    assert all(len(set(tri)) == 3 for tri in tris)


@pytest.mark.parametrize("case", range(256))
def test_case_boundary_on_each_face_is_the_face_rule(case):
    tris = _table()[case]
    directed = collections.Counter((t[i], t[(i + 1) % 3]) for t in tris for i in range(3))
    assert all(n == 1 for n in directed.values())
    boundary = [d for d in directed if (d[1], d[0]) not in directed]
    per_face = collections.defaultdict(set)
    for p, q in boundary:
        face = _face_of((p, q))
        assert face is not None, "boundary segment %s of case %d is not on a cube face" % ((p, q), case)
        per_face[face].add(frozenset((p, q)))
    for a in range(3):
        for v in (0, 1):
            assert per_face.get((a, v), set()) == _face_rule(case, a, v), (case, a, v)


def test_table_header_constants():
    t = _table()
    with open(os.path.join(CSRC, "mc_table.h")) as f:
        text = f.read()
    assert "#define MC_MAX_TRIS %d" % max(len(x) for x in t) in text
    assert t[0] == [] and t[255] == []


# ---- oracle meshes of analytic fields ------------------------------------------------------------------------------
def _directed_edges(faces):
    f = faces.astype(np.int64)
    return np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])


def _signed_volume(verts, faces):
    a, b, c = (verts[faces[:, i]].astype(np.float64) for i in range(3))
    return np.einsum("ij,ij->i", a, np.cross(b, c)).sum() / 6.0


@pytest.mark.parametrize("res", [32, 64])
@pytest.mark.parametrize("kind,euler", [("sphere", 2), ("torus", 0), ("two_spheres", 4)])
def test_oracle_mesh_of_analytic_field(kind, euler, res):
    field, vol = iso_field(kind, (res, res, res))
    assert not (field == 0).any(), "the level must not be hit exactly"
    verts, faces = oracle_mesh.iso_surface(field, 0.0)
    assert len(verts) and len(faces)
    # closed and consistently oriented: every directed edge once, and its reverse once
    de = _directed_edges(faces)
    key = de[:, 0] * len(verts) + de[:, 1]
    rkey = de[:, 1] * len(verts) + de[:, 0]
    assert len(np.unique(key)) == len(key)
    assert np.array_equal(np.sort(key), np.sort(rkey))
    n_edges = len(key) // 2
    assert len(verts) - n_edges + len(faces) == euler
    # outward normals -> positive enclosed volume; fan triangulation of a sampled field: within 3% at 32^3, 1% at 64^3
    v = _signed_volume(verts, faces)
    assert v > 0
    assert abs(v / vol - 1) < (0.03 if res == 32 else 0.01), (v, vol)


@pytest.mark.parametrize("shape,spacing,offset", [((32, 32, 32), (1, 1, 1), (0, 0, 0)),
                                                  ((20, 27, 33), (0.5, 2.0, 0.25), (-3.0, 1.5, 0.125))])
def test_oracle_vertices_lie_on_crossed_edges(shape, spacing, offset):
    field, _ = iso_field("torus", shape)
    verts, faces, vals = oracle_mesh.iso_surface(field, 0.0, spacing, offset, values=True)
    inside = field > 0
    owners = []
    for a in range(3):
        sl0 = [slice(None)] * 3
        sl1 = [slice(None)] * 3
        sl0[a], sl1[a] = slice(0, -1), slice(1, None)
        crossed = np.zeros(shape, bool)
        crossed[tuple(sl0)] = inside[tuple(sl0)] != inside[tuple(sl1)]
        for p in np.argwhere(crossed):
            owners.append((tuple(p), a))
    owners.sort(key=lambda pa: (pa[0], pa[1]))      # C order of the owner, then the axis
    assert len(owners) == len(verts)
    sp, of = np.asarray(spacing, np.float64), np.asarray(offset, np.float64)
    for (p, a), v, val in zip(owners, verts.astype(np.float64), vals):
        q = list(p)
        q[a] += 1
        f0, f1 = float(field[p]), float(field[tuple(q)])
        grid = (v - of) / sp
        for b in range(3):
            if b != a:
                assert np.float32(p[b] * spacing[b] + offset[b]) == np.float32(v[b])
        t = grid[a] - p[a]
        assert -1e-5 <= t <= 1 + 1e-5
        interp = f0 + t * (f1 - f0)
        assert abs(interp) <= 1e-5 * max(1.0, abs(f0), abs(f1)), (p, a, interp)
        assert val == max(f0, f1)
    assert faces.min() >= 0 and faces.max() < len(verts)


def test_write_obj_round_trips(tmp_path):
    field, _ = iso_field("sphere", (24, 24, 24))
    verts, faces = oracle_mesh.iso_surface(field, 0.0, 1 / 128, -0.5)
    verts = verts * np.float32(np.pi)           # awkward mantissas
    path = tmp_path / "m.obj"
    postprocess.write_obj(str(path), verts, faces)
    vs, fs = [], []
    with open(path) as f:
        for line in f:
            tok = line.split()
            if tok[0] == "v":
                vs.append([np.float32(float(x)) for x in tok[1:]])
            elif tok[0] == "f":
                fs.append([int(x) - 1 for x in tok[1:]])
    assert np.array_equal(np.asarray(vs, np.float32), verts)
    assert np.array_equal(np.asarray(fs, np.int32), faces)


# ---- C ABI argument checks (fake device addresses: nothing is launched or dereferenced) ------------------------------
def _d(v=4096):
    return ctypes.c_void_p(v)


@pytest.mark.parametrize("shape,ws,code,needle", [
    ((1, 8, 8, 257), 1 << 30, -1, b"unsupported"),       # W > 256
    ((1, 1, 8, 8), 1 << 30, -1, b"unsupported"),         # D < 2
    ((1, 8, 8, 8), 16, -2, b"workspace"),                # short workspace
])
def test_iso_surface_abi_validates_before_launching(shape, ws, code, needle):
    lib = _lib.load()
    n, d, h, w = shape
    rc = lib.genre_b200_iso_surface_count(_d(), n, d, h, w, 0.5, _d(), ws, _d(), None)
    msg = lib.genre_b200_last_error()
    assert rc == code and needle in msg.lower(), (rc, msg)
    rc = lib.genre_b200_iso_surface_emit(_d(), n, d, h, w, 0.5, 1, 1, 1, 0, 0, 0, _d(), _d(), _d(), None, _d(), ws, None)
    msg = lib.genre_b200_last_error()
    assert rc == code and needle in msg.lower(), (rc, msg)


def test_iso_surface_workspace_bytes():
    lib = _lib.load()
    # one bit per voxel + two int2 per z row, each part 16-byte aligned
    assert lib.genre_b200_iso_surface_workspace_bytes(16, 128, 128, 128) == 16 * 128 * 128 * (4 * 4 + 16)
    assert lib.genre_b200_iso_surface_workspace_bytes(1, 8, 8, 257) == 0
    assert lib.genre_b200_iso_surface_workspace_bytes(0, 8, 8, 8) == 0


def test_iso_surface_refuses_cpu_tensors():
    with pytest.raises(RuntimeError):
        postprocess.iso_surface(torch.zeros(8, 8, 8), 0.5)


# ---- the skimage stand-in ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kw", [dict(step_size=2), dict(mask=np.ones((4, 4, 4), bool)),
                                dict(gradient_direction="ascent"), dict(allow_degenerate=False), dict(method="lorensen")])
def test_marching_cubes_stand_in_rejects_what_it_does_not_implement(kw):
    vol = np.zeros((4, 4, 4), np.float32)
    vol[1:3, 1:3, 1:3] = 1
    with pytest.raises(NotImplementedError):
        compat.marching_cubes(vol, 0.5, **kw)
    if "method" not in kw:
        with pytest.raises(NotImplementedError):
            compat.marching_cubes_lewiner(vol, 0.5, **kw)


def test_marching_cubes_stand_in_in_a_bad_fork(monkeypatch):
    monkeypatch.setattr(torch.cuda, "_is_in_bad_fork", lambda: True)
    vol = np.zeros((4, 4, 4), np.float32)
    with pytest.raises(RuntimeError, match="vis_workers 0") as e:
        compat.marching_cubes_lewiner(vol, 0.25, spacing=(1 / 128,) * 3)
    assert "fork" in str(e.value) and "export_obj" in str(e.value)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device message")
def test_marching_cubes_stand_in_without_a_device():
    with pytest.raises(RuntimeError, match="no CUDA device"):
        compat.marching_cubes(np.zeros((4, 4, 4), np.float32), 0.0)


def test_stub_skimage_measure_is_the_stand_in():
    import sys
    compat.stub_optional_modules(offline_resnet=False)
    measure = sys.modules["skimage.measure"]
    if getattr(sys.modules["skimage"], "__genre_b200_stub__", False):
        assert measure.marching_cubes_lewiner is compat.marching_cubes_lewiner
        assert measure.marching_cubes is compat.marching_cubes
