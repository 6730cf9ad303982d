"""Blocks anywhere in block-key space, without a camera: synthetic blocks holding the analytic TSDF of a plane, in the three
forms the volume's readers are checked with -- a checkpoint file (what a GPU volume loads), the arrays of export_blocks
(what the ray-cast and tracking models take) and an oracle volume (oracle.Volume.import_blocks).  These CPU tests pin the
helpers and the oracle's block import, and extract planes placed at the corners of the key range (+-2^20 blocks per axis).
tests/test_gpu_key_edges.py uses the helpers at the arena seams and key limits."""
import numpy as np

import test_checkpoint_format as fmt
from conftest import lexorder
from oracle import oracle

KEY_LIMIT = 1 << 20          # plain volume: block keys in [-2^20, 2^20) on every axis
OBJ_HALF = 1 << 17           # arena object: true block x in [-2^17, 2^17)
COUNT = 3                    # integration count of every observed synthetic voxel

_L = np.arange(16)
LOCAL = np.stack(np.meshgrid(_L, _L, _L, indexing="ij"), -1).reshape(4096, 3)     # voxel index x*256 + y*16 + z


def unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v)


def plane_blocks(keys, vl, trunc, anchor, frac, normal):
    """Blocks at integer keys [n,3] (sorted lexicographically here) holding the plane through voxel coordinate anchor + frac
    (anchor integer, frac real; voxel g's centre is at g + 0.5) with unit normal `normal` pointing to the free side.
    sdf = vl * normal . ((g - anchor) + 0.5 - frac) in FP64 from the integer offset g - anchor, so the same plane moved by
    whole blocks gives the same voxels; tsdf = clip(sdf / trunc, -1, 1); weight COUNT where |sdf| < trunc, else 0; colour
    sums = rgb * weight, rgb a pattern of the voxel's place in its block.  Returns (keys i32 [n,3], tsdf f32 [n,4096],
    weight f32 [n,4096], colour sums u32 [n,4096,3]), voxel index x*256 + y*16 + z."""
    keys = np.asarray(keys, np.int64).reshape(-1, 3)
    keys = keys[lexorder(keys)]
    rel = (keys[:, None, :] * 16 - np.asarray(anchor, np.int64)) + LOCAL[None]
    r = (rel + 0.5) - np.asarray(frac, np.float64)
    n = np.asarray(normal, np.float64)
    sdf = vl * ((r[..., 0] * n[0] + r[..., 1] * n[1]) + r[..., 2] * n[2])
    tsdf = np.clip(sdf / trunc, -1.0, 1.0).astype(np.float32)
    weight = np.where(np.abs(sdf) < trunc, COUNT, 0).astype(np.float32)
    rgb = (LOCAL * np.array([37, 11, 5]) + np.array([40, 90, 150])) % 256
    sums = (rgb[None] * weight[..., None].astype(np.int64)).astype(np.uint32)
    return keys.astype(np.int32), tsdf, weight, sums


def concat(*blocks):
    """several block sets as one, sorted by key"""
    keys = np.concatenate([b[0] for b in blocks])
    o = lexorder(keys)
    return tuple(np.concatenate([b[i] for b in blocks])[o] for i in range(4))


def export_arrays(blocks):
    """(keys, tsdf, weight, colour f64 on the 0..255 scale): export_blocks' form, what raycast_model and track_model take"""
    keys, tsdf, weight, sums = blocks
    return keys, tsdf, weight, sums / np.maximum(weight, 1.0).astype(np.float64)[..., None]


def oracle_volume(blocks, vl, trunc):
    ov = oracle.Volume(vl, trunc)
    ov.import_blocks(*export_arrays(blocks))
    return ov


def records(blocks):
    """u8 [n][65536]: the device records (tsdf bits; colour sums with the 16-bit count in the high bytes of .y / .z) in pool
    order z*256 + x*16 + y"""
    keys, tsdf, weight, sums = blocks
    n = len(keys)
    w = weight.astype(np.uint32)
    r = np.empty((n, 4096, 4), np.uint32)
    r[..., 0] = tsdf.view(np.uint32)
    r[..., 1] = sums[..., 0] | ((w & 0xFF) << 24)
    r[..., 2] = sums[..., 1] | ((w >> 8) << 24)
    r[..., 3] = sums[..., 2]
    r = r.reshape(n, 16, 16, 16, 4).transpose(0, 3, 1, 2, 4)                      # [x][y][z] -> [z][x][y]
    return np.ascontiguousarray(r).view(np.uint8).reshape(n, fmt.BLOCK_BYTES)


def write_checkpoint(path, blocks, vl, trunc):
    fmt.write(path, blocks[0], records(blocks), voxel_length=vl, sdf_trunc=trunc, color_type=1, frames=COUNT)


def corner_keys(lo, side=2):
    """the side^3 keys of a cube of blocks whose lowest key is (lo, lo, lo)"""
    r = np.arange(lo, lo + side)
    return np.stack(np.meshgrid(r, r, r, indexing="ij"), -1).reshape(-1, 3)


VL, TRUNC = 0.005, 0.02
N_CORNER = unit([1.0, 2.0, 3.0])


def corner_plane(lo):
    """the oblique plane through the centre of the 2x2x2 blocks whose lowest key is (lo, lo, lo)"""
    return plane_blocks(corner_keys(lo), VL, TRUNC, (16 * lo + 16,) * 3, (0.3, -0.2, 0.1), N_CORNER)


def test_import_export_bit_exact():
    """blocks at the key limits, the arena seam keys and the origin come back from export_blocks bit for bit; importing a
    key again replaces its block"""
    keys = [(-KEY_LIMIT, 0, KEY_LIMIT - 1), (OBJ_HALF - 1, 3, -2), (-OBJ_HALF, 3, -2), (0, 0, 0), (KEY_LIMIT - 1, -KEY_LIMIT, 5)]
    blocks = plane_blocks(keys, VL, TRUNC, (0, 0, 0), (0.25, 0.5, 0.75), unit([1.0, -1.0, 0.5]))
    rng = np.random.default_rng(7)
    t = blocks[1].copy()
    t[:, ::3] = rng.random((len(keys), t[:, ::3].shape[1]), np.float32) * 2 - 1    # arbitrary values, not just a plane
    blocks = (blocks[0], t, blocks[2], blocks[3])
    want = export_arrays(blocks)
    ov = oracle.Volume(VL, TRUNC)
    ov.import_blocks(*[a[::-1] for a in want])                                       # any order in, sorted out
    got = ov.export_blocks()
    assert ov.num_blocks() == len(keys)
    assert (got[0] == want[0]).all() and (got[1].view(np.uint32) == want[1].view(np.uint32)).all()
    assert (got[2] == want[2]).all() and (got[3].view(np.uint64) == want[3].view(np.uint64)).all()
    assert (want[2] > 0).any() and (want[3][want[2] > 0] > 0).all()
    ov.import_blocks(want[0][:1], np.zeros((1, 4096), np.float32), np.zeros((1, 4096), np.float32), np.zeros((1, 4096, 3)))
    again = ov.export_blocks()
    assert ov.num_blocks() == len(keys) and not again[2][0].any() and (again[2][1:] == want[2][1:]).all()


def test_checkpoint_form_decodes_to_the_same_blocks(tmp_path):
    """the file the helper writes is a valid checkpoint (header checked without a GPU) whose records decode, in pool order,
    to the tsdf, counts and colour sums of the export form"""
    blocks = corner_plane(-KEY_LIMIT)
    p = tmp_path / "corner.otslam"
    write_checkpoint(p, blocks, VL, TRUNC)
    assert fmt.info(p) == (0, (VL, TRUNC, 1, COUNT, 8))
    hdr, keys, cks, rec = fmt.parse(p.read_bytes())
    assert (keys == blocks[0]).all()
    r = rec.view(np.uint32).reshape(8, 16, 16, 16, 4).transpose(0, 2, 3, 1, 4).reshape(8, 4096, 4)   # [z][x][y] -> x*256+y*16+z
    assert (r[..., 0] == blocks[1].view(np.uint32)).all()
    assert (((r[..., 1] >> 24) | ((r[..., 2] >> 24) << 8)) == blocks[2]).all()
    assert (np.stack([r[..., k] & 0xFFFFFF for k in (1, 2, 3)], -1) == blocks[3]).all()
    for i in range(8):
        assert fmt.block_checksum(rec[i].tobytes(), keys[i]) == int(cks[i])


def on_plane(p, anchor, frac, n):
    """signed distance of world points to the plane, in voxels, from the integer part of the anchor first"""
    g = np.asarray(p, np.float64) / VL - np.asarray(anchor, np.float64)
    return (g - np.asarray(frac)) @ n


def test_planes_at_the_key_corners_extract_onto_the_plane():
    """the oblique plane at the lowest and the highest corner of the key range: mesh vertices and points lie on it"""
    for lo in (-KEY_LIMIT, KEY_LIMIT - 2):
        ov = oracle_volume(corner_plane(lo), VL, TRUNC)
        verts, cols, faces, ek = ov.extract_triangle_mesh()
        pts, pcols, pek = ov.extract_point_cloud()
        assert len(verts) > 1000 and len(faces) > 1000 and len(pts) > 1000
        anchor = (16 * lo + 16,) * 3
        assert np.abs(on_plane(verts, anchor, (0.3, -0.2, 0.1), N_CORNER)).max() < 1e-4
        # points: Open3D divides by the FP32 sum |f0| + |f1|, whose rounding (2^-24 relative) moves a point 2^24 voxels out
        # by up to about one voxel along its edge
        assert np.abs(on_plane(pts, anchor, (0.3, -0.2, 0.1), N_CORNER)).max() < 1.0
        assert ek[:, :3].min() >= 16 * lo and ek[:, :3].max() < 16 * (lo + 2)


def test_corner_planes_are_the_origin_plane_shifted():
    """the same plane at the origin and at either corner: the same voxels, and mesh edge keys and point edge keys moved by
    16 * (the key shift), the same faces and vertex colours"""
    origin = oracle_volume(corner_plane(0), VL, TRUNC)
    m0 = origin.extract_triangle_mesh()
    p0 = origin.extract_point_cloud()
    b0 = corner_plane(0)
    for lo in (-KEY_LIMIT, KEY_LIMIT - 2):
        b = corner_plane(lo)
        assert (b[0] == b0[0] + lo).all() and (b[1].view(np.uint32) == b0[1].view(np.uint32)).all()
        assert (b[2] == b0[2]).all() and (b[3] == b0[3]).all()
        ov = oracle_volume(b, VL, TRUNC)
        m = ov.extract_triangle_mesh()
        assert len(m[0]) == len(m0[0]) and (m[3][:, :3] == m0[3][:, :3] + 16 * lo).all() and (m[3][:, 3] == m0[3][:, 3]).all()
        assert (m[2] == m0[2]).all() and (m[1] == m0[1]).all()
        p = ov.extract_point_cloud()
        assert len(p[0]) == len(p0[0]) and (p[2][:, :3] == p0[2][:, :3] + 16 * lo).all() and (p[2][:, 3] == p0[2][:, 3]).all()
