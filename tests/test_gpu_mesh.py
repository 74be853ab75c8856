"""Batched marching cubes on the GPU (postprocess.iso_surface / export_obj, the skimage stand-in) against the CPU oracle,
bit for bit: same vertices, same faces, same values, same order."""
import numpy as np
import pytest
import torch

import oracle_mesh
from genre_shapehd_b200 import compat, postprocess
from genre_shapehd_b200.synth import iso_field

pytestmark = pytest.mark.gpu


def _dev():
    return torch.device("cuda", torch.cuda.current_device())


def _same(a, b):
    """bitwise equality, NaN at the same places counting as equal (CPU and GPU NaN payloads differ)"""
    a = torch.as_tensor(a).cpu()
    b = torch.as_tensor(b).cpu()
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    if a.is_floating_point():
        na, nb = torch.isnan(a), torch.isnan(b)
        return torch.equal(na, nb) and torch.equal(a[~na], b[~nb])
    return torch.equal(a, b)


def _check(vols, level, spacing=(1.0, 1.0, 1.0), offset=(0.0, 0.0, 0.0)):
    """vols [B,D,H,W] numpy -> GPU meshes, each equal to the oracle's"""
    vols = np.ascontiguousarray(vols, dtype=np.float32)
    meshes = postprocess.iso_surface(torch.from_numpy(vols).to(_dev()), level, spacing, offset, values=True)
    assert len(meshes) == len(vols)
    for vol, (v, f, val) in zip(vols, meshes):
        ov, of, oval = oracle_mesh.iso_surface(vol, level, spacing, offset, values=True)
        assert v.shape == ov.shape and f.shape == of.shape, (v.shape, ov.shape, f.shape, of.shape)
        assert _same(v, torch.from_numpy(ov)), "vertices differ from the oracle"
        assert torch.equal(f.cpu(), torch.from_numpy(of)), "faces differ from the oracle"
        assert _same(val, torch.from_numpy(oval)), "values differ from the oracle"
    return meshes


@pytest.mark.parametrize("res", [32, 64, 128])
@pytest.mark.parametrize("kind", ["sphere", "torus"])
def test_analytic_fields_match_oracle(kind, res):
    field, _ = iso_field(kind, (res, res, res))
    meshes = _check(field[None], 0.0)
    assert len(meshes[0][1]) > 0


def _cases(vol, level):
    b = vol > level
    cs = np.zeros(tuple(n - 1 for n in vol.shape), np.int64)
    for c in range(8):
        di, dj, dk = (c >> 2) & 1, (c >> 1) & 1, c & 1
        cs |= b[di:di + cs.shape[0], dj:dj + cs.shape[1], dk:dk + cs.shape[2]].astype(np.int64) << c
    return cs


def test_noise_covers_every_case():
    vol = np.random.RandomState(7).rand(32, 32, 32).astype(np.float32)
    assert len(np.unique(_cases(vol, 0.5))) == 256
    _check(vol[None], 0.5)


@pytest.fixture(scope="module")
def genre_outputs():
    from genre_shapehd_b200.genre_models import GenReNet
    from genre_shapehd_b200.synth_genre import genre_inputs, init_genre_net_for_bench
    torch.manual_seed(0)
    net = init_genre_net_for_bench(GenReNet()).to(_dev()).eval()
    with torch.no_grad():
        out = net(genre_inputs(2, _dev(), seed=3))
    return {k: out[k].detach().float() for k in ("pred_voxel", "pred_proj_depth", "pred_proj_sph_full")}


@pytest.mark.parametrize("name,sigmoid", [("pred_voxel", True), ("pred_proj_depth", False), ("pred_proj_sph_full", False)])
def test_genre_outputs_match_oracle(genre_outputs, name, sigmoid):
    v = genre_outputs[name]
    v = torch.sigmoid(v) if sigmoid else v
    x = v[:, 0].cpu().numpy()
    # the visualiser's level (a seeded, untrained refiner may stay below it everywhere: then both meshes are empty) ...
    _check(x, 0.25, (1 / 128,) * 3, (-0.5,) * 3)
    # ... and a level inside the data range, for a dense mesh of the network's actual output
    level = float(np.median(x[x > x.min()])) if (x > x.min()).any() else float(x.min())
    meshes = _check(x, level, (1 / 128,) * 3, (-0.5,) * 3)
    assert sum(len(m[1]) for m in meshes) > 0


@pytest.mark.parametrize("shape", [(40, 72, 100), (17, 23, 33), (6, 10, 256), (3, 2, 2), (2, 5, 31)])
def test_non_cubic_shapes_match_oracle(shape):
    field, _ = iso_field("torus", shape, scale=max(shape))
    noise = np.random.RandomState(sum(shape)).rand(*shape).astype(np.float32) - 0.5
    _check(np.stack([field, noise]), 0.0)


def test_objects_touching_the_boundary():
    big, _ = iso_field("sphere", (48, 40, 36), center=(5.3, 20.1, 30.7), scale=80)
    full_slab = np.ones((48, 40, 36), np.float32)
    full_slab[:, :, 18:] = -1
    _check(np.stack([big, full_slab]), 0.0)


def test_voxels_equal_to_the_level():
    vol = np.random.RandomState(1).randint(0, 3, size=(2, 24, 24, 24)).astype(np.float32)
    assert (vol == 1).any()
    _check(vol, 1.0)


def test_one_nan_voxel():
    field, _ = iso_field("sphere", (32, 32, 32))
    r = int(0.3 * 32)
    field[16 + r, 16, 16] = np.nan       # on the surface: its edges give NaN vertices, the same ones on both sides
    field[16, 16, 16] = np.nan           # deep inside: the hole becomes a small closed bubble
    (v, f, val), = _check(field[None], 0.0)
    assert torch.isnan(v).any()


def test_spacing_and_offset():
    field, _ = iso_field("two_spheres", (30, 34, 50))
    _check(field[None], 0.0, (0.7, 1 / 128, 3.0), (-1.25, 0.5, 100.0))
    _check(field[None], 0.1, 1 / 128, -0.5)


def test_empty_and_full_volumes():
    vols = torch.stack([torch.zeros(20, 21, 22), torch.ones(20, 21, 22)]).to(_dev())
    for v, f in postprocess.iso_surface(vols, 0.5):
        assert v.shape == (0, 3) and f.shape == (0, 3)


def _batch():
    fields = [iso_field(k, (40, 36, 44))[0] for k in ("sphere", "torus", "two_spheres", "shell")]
    fields.append(np.zeros((40, 36, 44), np.float32) - 1)     # empty sample in the middle of a batch
    fields.append(np.random.RandomState(5).rand(40, 36, 44).astype(np.float32) - 0.5)
    return torch.from_numpy(np.stack(fields)).to(_dev())


def test_batched_equals_per_sample_and_repeats_bitwise():
    vols = _batch()
    batched = postprocess.iso_surface(vols, 0.0, 0.5, 1.0, values=True)
    again = postprocess.iso_surface(vols, 0.0, 0.5, 1.0, values=True)
    for i, m in enumerate(batched):
        single = postprocess.iso_surface(vols[i], 0.0, 0.5, 1.0, values=True)[0]
        for a, b, c in zip(m, single, again[i]):
            assert torch.equal(a, b) and torch.equal(a, c)


def test_permuting_the_batch_permutes_the_output():
    vols = _batch()
    perm = [3, 0, 5, 1, 4, 2]
    base = postprocess.iso_surface(vols, 0.0)
    permuted = postprocess.iso_surface(vols[perm], 0.0)
    for i, p in enumerate(perm):
        assert torch.equal(permuted[i][0], base[p][0]) and torch.equal(permuted[i][1], base[p][1])


def test_input_layouts():
    field = torch.from_numpy(iso_field("sphere", (20, 20, 20))[0]).to(_dev())
    a = postprocess.iso_surface(field, 0.0)[0]
    b = postprocess.iso_surface(field[None, None], 0.0)[0]
    c = postprocess.iso_surface(field.expand(2, 20, 20, 20), 0.0)[1]
    for x, y in ((a, b), (a, c)):
        assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])


def test_stand_in_matches_iso_surface_for_the_visualiser():
    """what Visualizer._save_iso_obj calls: marching_cubes_lewiner(df, 0.25, spacing=(1/128,)*3), then verts -= 0.5"""
    df = torch.sigmoid(torch.from_numpy(iso_field("torus", (64, 64, 64))[0] / 4)).numpy()
    verts, faces, normals, values = compat.marching_cubes_lewiner(df, 0.25, spacing=(1 / 128, 1 / 128, 1 / 128))
    assert verts.dtype == np.float32 and faces.dtype == np.int32 and normals.shape == verts.shape
    v, f, val = postprocess.iso_surface(torch.from_numpy(df).to(_dev()), 0.25, 1 / 128, -0.5, values=True)[0]
    assert np.array_equal(verts - np.float32(0.5), v.cpu().numpy())
    assert np.array_equal(faces, f.cpu().numpy()) and np.array_equal(values, val.cpu().numpy())
    assert np.allclose(np.linalg.norm(normals, axis=1), 1, atol=1e-5)
    # outward winding: the closed mesh encloses a positive volume
    a, b, c = (verts[faces[:, i]].astype(np.float64) for i in range(3))
    assert np.einsum("ij,ij->i", a, np.cross(b, c)).sum() > 0
    m = compat.marching_cubes(df, 0.25, spacing=(1 / 128,) * 3)
    assert np.array_equal(m[0], verts) and np.array_equal(m[1], faces)


def _parse_obj(path):
    vs, fs = [], []
    with open(path) as f:
        for line in f:
            tok = line.split()
            if tok and tok[0] == "v":
                vs.append([np.float32(float(x)) for x in tok[1:]])
            elif tok and tok[0] == "f":
                fs.append([int(x) - 1 for x in tok[1:]])
    return np.asarray(vs, np.float32).reshape(-1, 3), np.asarray(fs, np.int32).reshape(-1, 3)


def test_export_obj_writes_the_oracle_mesh(tmp_path):
    logits = torch.from_numpy(np.stack([iso_field("sphere", (32, 32, 32))[0], np.full((32, 32, 32), -3.0, np.float32),
                                        np.full((32, 32, 32), 3.0, np.float32)]))[:, None].to(_dev())
    paths = [str(tmp_path / ("%d.obj" % i)) for i in range(3)]
    before = logits.clone()
    postprocess.export_obj(logits, paths, 0.25, sigmoid=True)
    assert torch.equal(logits, before), "export_obj modified its input"
    probs = torch.sigmoid(logits[:, 0]).cpu().numpy()
    for p, vol in zip(paths, probs):
        vol = vol.copy()
        if 0.25 < vol.min():         # Visualizer._save_iso_obj's nudges
            vol[0, 0, 0] = 0.25 - 1
        if 0.25 > vol.max():
            vol[-1, -1, -1] = 0.25 + 1
        ov, of = oracle_mesh.iso_surface(vol, 0.25, 1 / 128, -0.5)
        v, f = _parse_obj(p)
        assert len(of) > 0
        assert np.array_equal(v, ov) and np.array_equal(f, of)
