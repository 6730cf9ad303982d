"""The volume's readers at the edges of block-key space.  An arena object's true block x lies in [-2^17, 2^17); the stored key
one past its last block is the next object's first block, so every reader must stop at the object's window: extraction,
point normals, ray casting and tracking of an object whose blocks reach the seam must equal the same blocks in a plain volume
of their own (which in turn equals the CPU references), bit for bit.  A plain volume's keys reach +-2^20 per axis: blocks at
exactly the limits load, sort and extract like the oracle, and one past is refused.  Synthetic blocks come from
tests/test_key_edges_oracle.py.  World coordinates here are 10 km and more from the origin, where FP32 resolves about a
quarter voxel: only parity is checked, not accuracy."""
import numpy as np
import pytest

import test_checkpoint_format as fmt
from conftest import canon_mesh, lexorder
from test_key_edges_oracle import KEY_LIMIT, OBJ_HALF, concat, corner_plane, oracle_volume, plane_blocks, unit, write_checkpoint

pytestmark = pytest.mark.gpu

VL, TRUNC = 0.005, 0.02
SEAM = 16 * OBJ_HALF                       # voxel x of the window edge: object o ends at +SEAM, object o + 1 starts at -SEAM
N_SEAM = unit([-1.0, 0.01, 0.005])         # free side towards -x
YZ = [(ky, kz) for ky in (0, 1) for kz in (0, 1)]


def seam_blocks():
    """object o: its last block column (true kx = 2^17 - 1), surface 0.8 voxel before the seam, last layer negative;
    object o + 1: its first column (true kx = -2^17), surface 1.2 voxels after the seam, first layer positive"""
    last = plane_blocks([(OBJ_HALF - 1, ky, kz) for ky, kz in YZ], VL, TRUNC, (SEAM, 0, 0), (-0.8, 16.0, 16.0), N_SEAM)
    first = plane_blocks([(-OBJ_HALF, ky, kz) for ky, kz in YZ], VL, TRUNC, (-SEAM, 0, 0), (1.2, 16.0, 16.0), N_SEAM)
    return last, first


def plain(path=None):
    from otslam_b200.volume import TSDFVolume
    v = TSDFVolume(VL, TRUNC)
    if path is not None:
        v.load(path)
    return v


def faces_in_range(v):
    """extract the mesh and check the face indices on the host before anything else reads them"""
    verts, cols, nrm, faces, ek = v.extract_triangle_mesh()
    assert ((faces >= 0) & (faces < len(verts))).all(), "face indices outside the mesh"
    return verts, cols, nrm, faces, ek


def canon_with_normals(m):
    verts, cols, nrm, faces, ek = m
    return canon_mesh(verts, cols, faces, ek) + (nrm[lexorder(ek)],)


def same_bits(x, y):
    x, y = np.ascontiguousarray(x), np.ascontiguousarray(y)
    return x.shape == y.shape and x.dtype == y.dtype and (x.view(np.uint8) == y.view(np.uint8)).all()


def assert_same_volume(v, ref):
    """export_blocks, stats, mesh (vertices, colours, faces, edge keys, vertex normals), points, their colours, keys and
    normals: bit for bit"""
    ea, eb = v.export_blocks(), ref.export_blocks()
    assert all(same_bits(x, y) for x, y in zip(ea, eb)), "export_blocks"
    assert v.stats() == ref.stats()
    A, B = canon_with_normals(faces_in_range(v)), canon_with_normals(faces_in_range(ref))
    assert len(A[0]) == len(B[0]) > 0 and all(same_bits(x, y) for x, y in zip(A, B)), "mesh"
    pa, pb = v.extract_point_cloud(normals=True), ref.extract_point_cloud(normals=True)
    ia, ib = lexorder(pa[2]), lexorder(pb[2])
    assert len(ia) == len(ib) > 0 and all(same_bits(x[ia], y[ib]) for x, y in zip(pa, pb)), "points"


def assert_equals_oracle(v, ov):
    """mesh and points of GPU volume v against the oracle's: as tests/test_gpu_extract_cloud.py checks them"""
    from oracle import oracle
    verts, cols, nrm, faces, ek = faces_in_range(v)
    A, B = canon_mesh(*ov.extract_triangle_mesh()), canon_mesh(verts, cols, faces, ek)
    assert len(A[0]) == len(B[0]) > 0 and (A[3] == B[3]).all() and (A[0] == B[0]).all() and (A[2] == B[2]).all()
    assert np.abs(A[1] - B[1]).max() <= 1e-9
    assert (oracle.vertex_normals(verts, faces) == nrm).all()
    gp, gc, gpe, gpn = v.extract_point_cloud(normals=True)
    op, oc, ope = ov.extract_point_cloud()
    a, b = lexorder(ope), lexorder(gpe)
    assert len(gp) == len(op) > 0 and (ope[a] == gpe[b]).all() and (op[a] == gp[b]).all() and np.abs(oc[a] - gc[b]).max() <= 2e-7
    assert np.abs(ov.point_normals(gp) - gpn).max() <= 1e-12


def seam_arena(o, tmp_path):
    """objects o and o + 1 of an arena loaded with the seam blocks, and each set in a plain volume of its own"""
    from otslam_b200.volume import ArenaView
    last, first = seam_blocks()
    files = [tmp_path / "last.otslam", tmp_path / "first.otslam"]
    for b, p in zip((last, first), files):
        write_checkpoint(p, b, VL, TRUNC)
    arena = plain()
    arena.set_objects(o + 2)
    views = [ArenaView(arena, o), ArenaView(arena, o + 1)]
    for w, p in zip(views, files):
        assert w.load(p) == len(YZ)
    return arena, views, [plain(p) for p in files], [oracle_volume(b, VL, TRUNC) for b in (last, first)], files


def assert_seam_precondition(views):
    """the facing layers across the seam -- x = 15 of object o's blocks, x = 0 of object o + 1's -- are observed and of
    opposite signs, read back from the arena itself"""
    ka, ta, wa, _ = views[0].export_blocks()
    kb, tb, wb, _ = views[1].export_blocks()
    assert (ka[:, 0] == OBJ_HALF - 1).all() and (kb[:, 0] == -OBJ_HALF).all() and (ka[:, 1:] == kb[:, 1:]).all()
    la, lb = (a.reshape(-1, 16, 16, 16) for a in (ta, tb))
    wla, wlb = (a.reshape(-1, 16, 16, 16) for a in (wa, wb))
    facing = (wla[:, 15] > 0) & (wlb[:, 0] > 0) & (la[:, 15] * lb[:, 0] < 0)
    assert facing.sum() == len(YZ) * 256


@pytest.mark.parametrize("o", [0, 6])
def test_seam_extraction_equals_own_volume(o, tmp_path):
    """mesh, points and point normals of objects o and o + 1: no triangle or point across the seam (object o's +x
    marching-cubes neighbour), no normal from the other object's voxels (object o + 1's -x samples of GetTSDFAt)"""
    arena, views, own, ovs, _ = seam_arena(o, tmp_path)
    assert_seam_precondition(views)
    for w, ref, ov in zip(views, own, ovs):
        assert_equals_oracle(ref, ov)
        assert_same_volume(w, ref)
    for v in [arena] + own:
        v.close()


def look_plus_x(eye):
    """world->camera extrinsic of a camera at `eye` (metres) looking along +x, image y along -z: exact entries"""
    e = np.zeros((4, 4))
    R = np.array([[0.0, 1.0, 0.0], [0.0, 0.0, -1.0], [1.0, 0.0, 0.0]])      # rows: camera x, y, z axes in the world
    e[:3, :3] = R
    e[:3, 3] = -(R @ np.asarray(eye, np.float64))
    e[3, 3] = 1.0
    return e


def turned(e, deg_y, deg_x):
    """the same camera turned about its own y and x axes"""
    a, b = np.radians(deg_y), np.radians(deg_x)
    ry = np.array([[np.cos(a), 0, np.sin(a), 0], [0, 1, 0, 0], [-np.sin(a), 0, np.cos(a), 0], [0, 0, 0, 1]])
    rx = np.array([[1, 0, 0, 0], [0, np.cos(b), -np.sin(b), 0], [0, np.sin(b), np.cos(b), 0], [0, 0, 0, 1]])
    return rx @ ry @ e


W, H = 64, 48
INTR = (60.0, 60.0, 31.5, 23.5)


def seam_views():
    """for object o: a camera 100 voxels before its surface; for object o + 1: 100 voxels before the seam, so its rays
    cross the window edge (true kx = -2^17 - 1 is object o's last block in stored keys) before they reach the surface"""
    eyes = [np.array([(SEAM - 100) * VL, 16 * VL, 16 * VL]), np.array([(-SEAM - 100) * VL, 16 * VL, 16 * VL])]
    return [np.stack([turned(look_plus_x(eye), a, b) for a, b in ((0, 0), (6, -4), (-5, 7))]) for eye in eyes]


@pytest.mark.parametrize("o", [0, 6])
def test_seam_ray_cast_and_track_equal_own_volume(o, tmp_path):
    """ray casting: hit refinement and normals within 1.5 voxels of the seam; arena object, own volume and the CPU model
    (depth, vertex, normal bit for bit, colour within one level).  Tracking against the same surfaces: the same bits."""
    from test_gpu_raycast import assert_equals_oracle as assert_equals_model
    from test_gpu_track import same_bits as same_track, seeded_starts
    from test_raycast_oracle import raycast
    from test_track_oracle import track
    arena, views, own, ovs, _ = seam_arena(o, tmp_path)
    for k, (w, ref, ov, ext) in enumerate(zip(views, own, ovs, seam_views())):
        g = w.ray_cast(INTR, ext, W, H)
        r = ref.ray_cast(INTR, ext, W, H)
        for a in ("depth", "vertex", "normal", "color"):
            assert same_bits(g[a], r[a]), a
        assert_equals_model(r, raycast(ov, INTR, ext, W, H))
        edge = (SEAM if k == 0 else -SEAM) * VL
        hit = r["depth"] > 0
        assert (np.abs(r["vertex"][..., 0][hit] - edge) <= 1.5 * VL).sum() >= 100, "hits near the seam"
        # frames: the rendered depth in 0.1 mm units, tracked from seeded starts a few millimetres and tenths of a degree off
        frames = np.round(r["depth"] * 10000.0).astype(np.uint16)
        inits = seeded_starts(ext, 11 + k, cm=(0.2, 0.5), deg=(0.2, 0.5))
        kw = dict(depth_scale=10000.0)
        tg, tr = w.track(frames, INTR, inits, **kw), ref.track(frames, INTR, inits, **kw)
        same_track(tg, tr)
        same_track(tr, track(ov, frames, INTR, inits, **kw))
        assert (tr["fitness"] > 0).any()
    for v in [arena] + own:
        v.close()


@pytest.mark.parametrize("o", [0, 6])
def test_seam_checkpoint_round_trip(o, tmp_path):
    """object o saved from the arena is the file it was loaded from; loaded into object o of a fresh arena whose object
    o + 1 is already there, it equals the original and object o + 1 is untouched"""
    from otslam_b200.volume import ArenaView
    arena, views, own, _, files = seam_arena(o, tmp_path)
    p = tmp_path / "saved.otslam"
    views[0].save(p)
    assert p.read_bytes() == files[0].read_bytes()
    fresh = plain()
    fresh.set_objects(o + 2)
    nxt = ArenaView(fresh, o + 1)
    nxt.load(files[1])
    before = nxt.export_blocks()
    assert ArenaView(fresh, o).load(p) == len(YZ)
    assert_same_volume(ArenaView(fresh, o), own[0])
    assert all(same_bits(x, y) for x, y in zip(before, nxt.export_blocks()))
    assert_same_volume(nxt, own[1])
    for v in [arena, fresh] + own:
        v.close()


def band_frames(surface_vox, cam_vox, n=3):
    """n u16 frames (0.1 mm units) of the plane x = surface_vox voxels seen fronto-parallel from cameras at x = cam_vox
    looking +x, each moved a little in y and z, with their extrinsics and a colour pattern"""
    depth_m = (surface_vox - cam_vox) * VL
    assert 0.0 < depth_m < 3.0
    d = np.full((n, H, W), round(depth_m * 10000.0), np.uint16)
    rgb = np.zeros((n, H, W, 3), np.uint8)
    rgb[..., 0] = (np.arange(W) * 4)[None, None]
    rgb[..., 1] = (np.arange(H) * 5)[None, :, None]
    rgb[..., 2] = (np.arange(n) * 60 + 30)[:, None, None]
    # camera x chosen so that the quantised depth lands the surface where asked: x = surface - depth
    cam_x = surface_vox * VL - d[0, 0, 0] / 10000.0
    ext = np.stack([look_plus_x([cam_x, (16 + 2 * k) * VL, (16 - 3 * k) * VL]) for k in range(n)])
    return d, rgb, ext


@pytest.mark.parametrize("o", [0, 6])
def test_seam_integration_matches_the_oracle(o):
    """object o integrates a surface whose truncation band ends in block 2^17 - 1, object o + 1 one whose band starts in
    block -2^17, in one batch.  Each object equals its oracle volume; a surface one voxel further out is refused."""
    from oracle import oracle
    from otslam_b200.volume import ArenaView
    # band of a surface at x: [x - 4, x + 4) voxels; object o: x + 4 = SEAM - 0.2 (last layer, centre SEAM - 0.5, is behind the
    # surface and observed); object o + 1: x - 4 = -SEAM + 0.2 (first layer, centre -SEAM + 0.5, in front and observed)
    surf = (SEAM - 4.2, -SEAM + 4.2)
    frames = [band_frames(surf[0], surf[0] - 100), band_frames(surf[1], surf[1] - 100)]
    d = np.concatenate([f[0] for f in frames])
    rgb = np.concatenate([f[1] for f in frames])
    ext = np.concatenate([f[2] for f in frames])
    ids = np.repeat(np.array([o, o + 1], np.int32), 3)
    arena = plain()
    arena.set_objects(o + 2)
    arena.integrate_batch(d, rgb, INTR, ext, depth_scale=10000.0, object_ids=ids)
    views = [ArenaView(arena, o), ArenaView(arena, o + 1)]
    keys = [w.export_blocks()[0] for w in views]
    assert (keys[0][:, 0] == OBJ_HALF - 1).all() and (keys[1][:, 0] == -OBJ_HALF).all()
    assert_seam_precondition_integrated(views)
    for k, w in enumerate(views):
        ov = oracle.Volume(VL, TRUNC)
        nupd = 0
        for j in range(3):
            nupd += ov.integrate(oracle.depth_convert(frames[k][0][j], 10000.0), frames[k][1][j], INTR, frames[k][2][j])[1]
        gk, gt, gw, gc = w.export_blocks()
        ok_, ot, ow, oc = ov.export_blocks()
        assert gk.shape == ok_.shape and (gk == ok_).all() and (gw == ow).all() and (gt == ot).all()
        assert np.abs(gc - oc)[ow > 0].max() <= 1.0
        assert w.stats()["weight_sum"] == nupd
        assert_equals_oracle(w, ov)
    # one voxel further out: the band leaves the window on either side; the batch is refused before it is integrated
    before = [w.stats() for w in views]
    for k, far in ((0, surf[0] + 1), (1, surf[1] - 1)):
        fd, fc, fe = band_frames(far, far - 100, 1)
        with pytest.raises(RuntimeError, match="block key outside"):
            arena.integrate_batch(fd, fc, INTR, fe, depth_scale=10000.0, object_ids=np.array([o + k], np.int32))
        after = [w.stats() for w in views]
        assert [a["weight_sum"] for a in after] == [b["weight_sum"] for b in before]
        assert [a["n_observed"] for a in after] == [b["n_observed"] for b in before]
    arena.close()


def assert_seam_precondition_integrated(views):
    """as assert_seam_precondition, over the voxels both frames observed"""
    ka, ta, wa, _ = views[0].export_blocks()
    kb, tb, wb, _ = views[1].export_blocks()
    ia = {tuple(k[1:]): i for i, k in enumerate(ka)}
    n = 0
    for j, k in enumerate(kb):
        i = ia.get(tuple(k[1:]))
        if i is None:
            continue
        la, lb = ta[i].reshape(16, 16, 16)[15], tb[j].reshape(16, 16, 16)[0]
        wla, wlb = wa[i].reshape(16, 16, 16)[15], wb[j].reshape(16, 16, 16)[0]
        n += int(((wla > 0) & (wlb > 0) & (la * lb < 0)).sum())
    assert n >= 256, n


def test_plain_checkpoint_key_limits(tmp_path):
    """keys at exactly -2^20 and 2^20 - 1 on each axis load; one past either refuses the file and leaves the volume as it was"""
    from otslam_b200 import _lib
    n = unit([1.0, 1.0, 1.0])
    lim = []
    for a in range(3):
        for x in (-KEY_LIMIT, KEY_LIMIT - 1):
            k = [0, 0, 0]
            k[a] = x
            lim.append(k)
    good = plane_blocks(lim, VL, TRUNC, (8, 8, 8), (0.0, 0.0, 0.0), n)
    write_checkpoint(tmp_path / "good.otslam", good, VL, TRUNC)
    v = plain()
    assert v.load(tmp_path / "good.otslam") == 6
    assert (v.export_blocks()[0] == good[0]).all()
    before, exp = v.stats(), v.export_blocks()
    for a in range(3):
        for x in (-KEY_LIMIT - 1, KEY_LIMIT):
            k = [1, 2, 3]
            k[a] = x
            p = tmp_path / f"past{a}_{x}.otslam"
            write_checkpoint(p, plane_blocks([k], VL, TRUNC, (0, 0, 0), (0.0, 0.0, 0.0), n), VL, TRUNC)
            assert _lib.lib.otslam_volume_load(v._h, str(p).encode(), None) == _lib.ERR_OVERFLOW, (a, x, _lib.last_error())
            assert v.stats() == before and all(same_bits(y, z) for y, z in zip(exp, v.export_blocks()))
    v.close()


@pytest.mark.parametrize("o", [0, 7])
def test_arena_checkpoint_key_limits(o, tmp_path):
    """arena object o: true x at exactly -2^17 and 2^17 - 1 loads; one past refuses the file and leaves the arena as it was"""
    from otslam_b200 import _lib
    from otslam_b200.volume import ArenaView
    blocks = plane_blocks([(-OBJ_HALF, 5, -5), (OBJ_HALF - 1, 5, -5)], VL, TRUNC, (0, 80, -72), (0.0, 0.3, 0.1), unit([0.0, 1.0, 1.0]))
    write_checkpoint(tmp_path / "good.otslam", blocks, VL, TRUNC)
    arena = plain()
    arena.set_objects(8)
    view = ArenaView(arena, o)
    assert view.load(tmp_path / "good.otslam") == 2
    assert (view.export_blocks()[0] == blocks[0]).all()
    own = plain(tmp_path / "good.otslam")
    assert_same_volume(view, own)
    before, exp = view.stats(), view.export_blocks()
    for x in (-OBJ_HALF - 1, OBJ_HALF):
        p = tmp_path / f"past{x}.otslam"
        write_checkpoint(p, plane_blocks([(x, 5, -5)], VL, TRUNC, (0, 80, -72), (0.0, 0.3, 0.1), unit([0.0, 1.0, 1.0])), VL, TRUNC)
        arena.select_object(o)
        assert _lib.lib.otslam_volume_load(arena._h, str(p).encode(), None) == _lib.ERR_OVERFLOW
        assert view.stats() == before and all(same_bits(y, z) for y, z in zip(exp, view.export_blocks()))
        assert sum(ArenaView(arena, j).num_blocks() for j in range(8)) == 2
    arena.close(); own.close()


def test_plain_volume_at_opposite_corners(tmp_path):
    """planes in the 2x2x2 blocks at (-2^20, -2^20, -2^20) and at (2^20 - 1, 2^20 - 1, 2^20 - 1), plus two blocks at the
    keys the top corner's +y and +z neighbours would pack to without the range check: export order is lexicographic
    (spans of 2^21 - 1 blocks on every axis: the full 63-bit sort key), and mesh, points and normals equal the oracle's"""
    top = KEY_LIMIT - 2
    alias = [(top, top + 1, -KEY_LIMIT),              # pack_key(top, top, 2^20): +z neighbour of (top, top, top + 1)
             (top + 1, -KEY_LIMIT, top)]              # pack_key(top, 2^20, top): +y neighbour of (top, top + 1, top)
    assert fmt.pack_key(top, top, KEY_LIMIT) == fmt.pack_key(*alias[0])
    assert fmt.pack_key(top, KEY_LIMIT, top) == fmt.pack_key(*alias[1])
    aliases = [plane_blocks([k], VL, TRUNC, (16 * k[0], 16 * k[1], 16 * k[2]), (3.3, 5.1, 0.6), unit([-1.0, 0.5, -2.0])) for k in alias]
    blocks = concat(corner_plane(-KEY_LIMIT), corner_plane(top), *aliases)
    assert all((b[2] > 0).any() for b in aliases)
    write_checkpoint(tmp_path / "corners.otslam", blocks, VL, TRUNC)
    v = plain(tmp_path / "corners.otslam")
    keys = v.export_blocks()[0]
    assert len(keys) == 18 and (keys == blocks[0]).all() and (lexorder(keys) == np.arange(18)).all()
    assert keys.min() == -KEY_LIMIT and keys.max() == KEY_LIMIT - 1
    ov = oracle_volume(blocks, VL, TRUNC)
    assert_equals_oracle(v, ov)
    v.close()
