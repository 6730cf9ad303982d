"""Volume checkpoints on the GPU: save, load, resume.  "Integrate A, save, load, integrate B" must give the same bits as
"integrate A then B" -- for plain volumes, slab ranks resharded N -> M, and arena objects -- and a file that fails any
check must leave the volume exactly as it was."""
import os

import numpy as np
import pytest

import test_checkpoint_format as fmt
from conftest import canon_mesh, lexorder

pytestmark = pytest.mark.gpu

VL = 0.005


@pytest.fixture(scope="module")
def window():
    """64 contiguous frames of configs[1] (frames 468..531 of the 1000-frame chair+table sequence)."""
    from otslam_b200 import synth
    seq = synth.make_sequence("chair_table", 1000, poses=synth.trajectory("chair_table", 1000)[468:532], device="cuda")
    d, c = seq.numpy()
    return seq, d, c


def assert_same_volume(a, b, color=True):
    """export_blocks bit for bit, stats, canonical mesh and point cloud bit for bit"""
    ea, eb = a.export_blocks(color=color), b.export_blocks(color=color)
    assert ea[0].shape == eb[0].shape and (ea[0] == eb[0]).all()
    assert (ea[1].view(np.uint32) == eb[1].view(np.uint32)).all() and (ea[2] == eb[2]).all()
    if color:
        assert (ea[3] == eb[3]).all()
    assert a.stats() == b.stats()
    ma, mb = a.extract_triangle_mesh(normals=False), b.extract_triangle_mesh(normals=False)
    A, B = canon_mesh(ma[0], ma[1], ma[3], ma[4]), canon_mesh(mb[0], mb[1], mb[3], mb[4])
    assert len(A[0]) == len(B[0]) > 0 and all((x == y).all() for x, y in zip(A, B))
    pa, pb = a.extract_point_cloud(), b.extract_point_cloud()
    ia, ib = lexorder(pa[2]), lexorder(pb[2])
    assert len(ia) == len(ib) and (pa[2][ia] == pb[2][ib]).all() and (pa[0][ia] == pb[0][ib]).all() and (pa[1][ia] == pb[1][ib]).all()


def assert_same_merged(full, parts):
    """merged per-rank extraction == the full volume's (as tests/test_gpu_extract_cloud.py checks slab runs)"""
    from otslam_b200 import slab as slabmod
    fv = full.extract_triangle_mesh(normals=False)
    merged = slabmod.merge_mesh_parts([(p[0], p[1], p[3], p[4]) for p in (v.extract_triangle_mesh(normals=False) for v in parts)])
    A, B = canon_mesh(fv[0], fv[1], fv[3], fv[4]), canon_mesh(*merged)
    assert len(A[0]) == len(B[0]) > 0 and (A[3] == B[3]).all() and (A[0] == B[0]).all() and (A[2] == B[2]).all()
    assert (A[1] == B[1]).all()
    fp, _, fe = full.extract_point_cloud()
    pp = [v.extract_point_cloud() for v in parts]
    pe = np.concatenate([p[2] for p in pp])
    a, b = lexorder(fe), lexorder(pe)
    assert len(fe) == len(pe) and (fe[a] == pe[b]).all() and (fp[a] == np.concatenate([p[0] for p in pp])[b]).all()


def exchange(parts):
    exports = [v.halo_export() for v in parts]
    for r, v in enumerate(parts):
        for keys, dest, planes in exports:
            if (dest == r).any():
                v.halo_import(keys[dest == r], planes[dest == r])


@pytest.mark.parametrize("color", [True, False])
def test_resume_equals_uninterrupted(window, tmp_path, color):
    """split at frame 37 (not a batch boundary): integrate, save, load into a fresh volume, integrate the rest"""
    from otslam_b200.volume import TSDFVolume
    seq, d, c = window
    c = c if color else None
    full = TSDFVolume(VL, 4 * VL, color=color)
    full.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    first = TSDFVolume(VL, 4 * VL, color=color)
    first.integrate_batch(d[:37], None if c is None else c[:37], seq.fxfycxcy, seq.extrinsic[:37])
    p = tmp_path / "first.otslam"
    first.save(p)
    assert not [f for f in os.listdir(tmp_path) if ".tmp" in f]
    resumed = TSDFVolume(VL, 4 * VL, color=color)
    assert resumed.load(p) == first.num_blocks()
    resumed.integrate_batch(d[37:], None if c is None else c[37:], seq.fxfycxcy, seq.extrinsic[37:])
    assert_same_volume(full, resumed, color)
    for v in (full, first, resumed):
        v.close()


def test_round_trip_and_file_checksums(window, tmp_path):
    from otslam_b200.volume import TSDFVolume, checkpoint_info, checkpoint_profile
    seq, d, c = window
    v = TSDFVolume(VL, 4 * VL)
    v.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    assert v.num_blocks() > 512, "the volume must span more than one pool chunk"
    a, b = tmp_path / "a.otslam", tmp_path / "b.otslam"
    v.save(a)
    prof = checkpoint_profile()
    assert prof["kernel_ms"] > 0 and prof["copy_ms"] > 0 and prof["wall_ms"] > 0
    assert checkpoint_info(a) == {"voxel_length": VL, "sdf_trunc": 4 * VL, "color": True, "frames": 64, "n_blocks": v.num_blocks()}
    w = TSDFVolume(VL, 4 * VL)
    assert w.load(a) == v.num_blocks()
    ev, ew = v.export_blocks(), w.export_blocks()
    assert all((x == y).all() for x, y in zip(ev, ew))
    assert v.stats() == w.stats()
    w.save(b)
    blob = a.read_bytes()
    assert blob == b.read_bytes(), "saving the loaded volume must give the same file"
    hdr, keys, cks, rec = fmt.parse(blob)
    assert (keys == ev[0]).all() and hdr["frames"] == 64
    for i in range(len(keys)):
        assert fmt.block_checksum(rec[i].tobytes(), keys[i]) == int(cks[i]), i
    # the records are the device layout: weight of voxel (x, y, z) = count in .y/.z high bytes at rec_index z*256 + x*16 + y
    r = rec.view(np.uint32).reshape(len(keys), 16, 16, 16, 4)              # [block][z][x][y][word]
    wgt = (r[..., 1] >> 24) | ((r[..., 2] >> 24) << 8)
    assert (wgt.transpose(0, 2, 3, 1).reshape(len(keys), 4096) == ev[2]).all()
    v.close(); w.close()


def test_reshard_three_axis_ranks_to_diagonal_axis_and_single(table_seq, tmp_path):
    """3 axis ranks (halo = 0, after a halo exchange) save their owned blocks; the parts load into 2 diagonal ranks,
    2 axis ranks with halo = 1 and one full volume, which all continue integrating and must equal the full volume."""
    from otslam_b200.volume import TSDFVolume, checkpoint_info
    seq, d, c = table_seq
    intr, ext = seq.fxfycxcy, seq.extrinsic
    full = TSDFVolume(0.01, 0.04)
    full.integrate_batch(d, c, intr, ext)
    first = TSDFVolume(0.01, 0.04)
    first.integrate_batch(d[:4], c[:4], intr, ext[:4])
    src = [TSDFVolume(0.01, 0.04, slab=(0, 2, 3, r, 0)) for r in range(3)]
    for v in src:
        v.integrate_batch(d[:4], c[:4], intr, ext[:4])
    owned = [v.num_blocks() for v in src]
    exchange(src)
    assert sum(v.num_blocks() for v in src) > sum(owned)
    parts = [str(tmp_path / f"vol.rank{r}of3.otslam") for r in range(3)]
    for v, p in zip(src, parts):
        v.save(p)
    assert [checkpoint_info(p)["n_blocks"] for p in parts] == owned, "halo pieces are not saved"
    assert sum(owned) == first.num_blocks()

    single = TSDFVolume(0.01, 0.04)
    assert single.load(parts) == first.num_blocks()
    single.integrate_batch(d[4:], c[4:], intr, ext[4:])
    assert_same_volume(full, single)

    for specs, halo in (([(3, 1, 2, r, 0) for r in range(2)], 0), ([(1, 2, 2, r, 1) for r in range(2)], 1)):
        ranks = [TSDFVolume(0.01, 0.04, slab=s) for s in specs]
        for v in ranks:
            v.load(parts)
            v.integrate_batch(d[4:], c[4:], intr, ext[4:])
        if halo == 0:
            assert sum(v.num_blocks() for v in ranks) == full.num_blocks()
            exchange(ranks)
        assert sum(v.stats()["weight_sum"] for v in ranks) >= full.stats()["weight_sum"]
        assert_same_merged(full, ranks)
        for v in ranks:
            v.close()
    for v in src + [full, first, single]:
        v.close()


def test_arena_object_checkpoint(tmp_path):
    """object 2 of a four-object arena -> a plain volume and object 1 of a new arena; both resume bit-identically"""
    from otslam_b200 import _lib, pipeline, synth
    from otslam_b200.volume import ArenaView, TSDFVolume
    scenes, n_per = ("table", "chair", "cone", "cardboard"), (14, 11, 9, 12)
    seqs = [synth.make_sequence(s, 48, subsample=(i, 48 // n), device="cuda") for i, (s, n) in enumerate(zip(scenes, n_per))]
    data = [s.numpy() for s in seqs]
    split = 5                                                   # object 2's frames [0, 5) before the checkpoint
    counts = [len(s) for s in seqs]
    counts[2] = split
    order = pipeline.interleave_plan(counts)
    arena = TSDFVolume(0.01, 0.04)
    arena.set_objects(4)
    arena.integrate_batch(np.stack([data[o][0][k] for o, k in order]), np.stack([data[o][1][k] for o, k in order]), seqs[0].fxfycxcy,
                          np.stack([seqs[o].extrinsic[k] for o, k in order]), object_ids=np.array([o for o, _ in order], np.int32))
    p = tmp_path / "object2.otslam"
    ArenaView(arena, 2).save(p)
    d2, c2, e2, intr = data[2][0], data[2][1], seqs[2].extrinsic, seqs[2].fxfycxcy
    own = TSDFVolume(0.01, 0.04)                                # object 2 as a volume of its own, all frames
    own.integrate_batch(d2, c2, intr, e2)

    plain = TSDFVolume(0.01, 0.04)
    plain.load(p)
    plain.integrate_batch(d2[split:], c2[split:], intr, e2[split:])
    assert_same_volume(own, plain)

    other = TSDFVolume(0.01, 0.04)
    other.set_objects(2)
    view = ArenaView(other, 1)
    assert view.load(p) == ArenaView(arena, 2).num_blocks()
    n0 = 4                                                      # object 0 of the new arena gets frames too (one shared launch)
    other.integrate_batch(np.concatenate([data[0][0][:n0], d2[split:]]), np.concatenate([data[0][1][:n0], c2[split:]]), intr,
                          np.concatenate([seqs[0].extrinsic[:n0], e2[split:]]),
                          object_ids=np.array([0] * n0 + [1] * (len(d2) - split), np.int32))
    assert_same_volume(own, view)

    # a key outside an arena object's x window: refused with OTSLAM_ERR_OVERFLOW, object unchanged
    before = view.stats()
    for kx in (1 << 17, -(1 << 17) - 1):
        q = tmp_path / f"far{kx}.otslam"
        fmt.write(q, np.array([[kx, 0, 0]], np.int32), np.zeros((1, fmt.BLOCK_BYTES), np.uint8), voxel_length=0.01, sdf_trunc=0.04)
        with pytest.raises(RuntimeError, match="key range"):
            view.load(q)
        assert _lib.lib.otslam_volume_load(other._h, str(q).encode(), None) == _lib.ERR_OVERFLOW
        assert view.stats() == before
    other.select_object(-1)
    with pytest.raises(RuntimeError, match="select_object"):
        other.save(tmp_path / "none.otslam")
    for v in (arena, own, plain, other):
        v.close()


def test_errors_leave_the_volume_unchanged(window, tmp_path):
    """every refused file: stats, num_blocks and the blocks themselves as before; the pool slots a refused load wrote are
    zero again (later integration into fresh blocks is unaffected); the clean file then loads"""
    from otslam_b200 import _lib
    from otslam_b200.volume import TSDFVolume
    seq, d, c = window
    intr, ext = seq.fxfycxcy, seq.extrinsic
    halves = []
    for r in range(2):
        v = TSDFVolume(VL, 4 * VL, slab=(0, 4, 2, r, 0))
        v.integrate_batch(d[:37], c[:37], intr, ext[:37])
        halves.append(str(tmp_path / f"h{r}.otslam"))
        v.save(halves[-1])
        v.close()
    blob = open(halves[1], "rb").read()
    hdr, keys, cks, rec = fmt.parse(blob)
    keys_off, cks_off, rec_off, _ = fmt.layout(hdr["n_blocks"])
    flipped = bytearray(blob)
    flipped[rec_off + 37 * fmt.BLOCK_BYTES + 1001] ^= 0x10
    dup = bytearray(blob)
    dup[keys_off + 12:keys_off + 24] = dup[keys_off:keys_off + 12]
    cases = {
        "voxel_length": (fmt.with_header(blob, voxel_length=0.006), _lib.ERR_INVALID),
        "color_type": (fmt.with_header(blob, color_type=0), _lib.ERR_INVALID),
        "flipped record byte": (bytes(flipped), _lib.ERR_FORMAT),
        "duplicate key": (bytes(dup), _lib.ERR_FORMAT),
        "frames > 65535": (fmt.with_header(blob, frames=70000), _lib.ERR_FORMAT),
        "count > frames": (fmt.with_header(blob, frames=1), _lib.ERR_FORMAT),
    }
    t = TSDFVolume(VL, 4 * VL)
    t.load(halves[0])
    ref = TSDFVolume(VL, 4 * VL)
    ref.load(halves[0])
    before, nb, blocks = t.stats(), t.num_blocks(), t.export_blocks()
    for name, (b, code) in list(cases.items()) + [("already present", (open(halves[0], "rb").read(), _lib.ERR_INVALID))]:
        p = tmp_path / "bad.otslam"
        p.write_bytes(b)
        assert _lib.lib.otslam_volume_load(t._h, str(p).encode(), None) == code, (name, _lib.last_error())
        assert t.stats() == before and t.num_blocks() == nb, name
    assert all((x == y).all() for x, y in zip(blocks, t.export_blocks()))
    t.integrate_batch(d[37:], c[37:], intr, ext[37:])          # new blocks take the slots the refused loads had written
    ref.integrate_batch(d[37:], c[37:], intr, ext[37:])
    assert_same_volume(ref, t)
    good = TSDFVolume(VL, 4 * VL)
    assert good.load(halves) == good.num_blocks() > 0
    for v in (t, ref, good):
        v.close()


def test_frame_guard_carries_over(table_seq, tmp_path):
    from otslam_b200.volume import TSDFVolume
    seq, d, c = table_seq
    v = TSDFVolume(0.01, 0.04)
    v.integrate_batch(d[:2], c[:2], seq.fxfycxcy, seq.extrinsic[:2])
    p = tmp_path / "a.otslam"
    v.save(p)
    p.write_bytes(fmt.with_header(p.read_bytes(), frames=65532))
    w = TSDFVolume(0.01, 0.04)
    w.load(p)
    w.integrate_batch(d[2:5], c[2:5], seq.fxfycxcy, seq.extrinsic[2:5])          # 65535 frames
    with pytest.raises(RuntimeError, match="65535"):
        w.integrate_batch(d[5:6], c[5:6], seq.fxfycxcy, seq.extrinsic[5:6])
    v.close(); w.close()


def test_compat_save_load(table_seq, tmp_path):
    """ScalableTSDFVolume.load(save(...)) extracts the same mesh, also for config-3 volumes after pipeline.integrate_many"""
    import otslam_b200.o3d_compat as o3d
    from otslam_b200 import pipeline, synth
    seq, d, c = table_seq
    I = o3d.pipelines.integration
    intr = o3d.camera.PinholeCameraIntrinsic(*seq.intr)

    def same_mesh(a, b):
        ma, mb = a.extract_triangle_mesh(), b.extract_triangle_mesh()
        for attr in ("vertices", "vertex_colors", "triangles"):
            x, y = np.asarray(getattr(ma, attr)), np.asarray(getattr(mb, attr))
            assert x.shape == y.shape and len(x) > 0 and (x == y).all(), attr

    vol = I.ScalableTSDFVolume(0.01, 0.04, I.TSDFVolumeColorType.RGB8)
    vol.integrate_sequence(d, c, intr, seq.extrinsic)
    vol.save(str(tmp_path / "v.otslam"))
    same_mesh(vol, I.ScalableTSDFVolume.load(str(tmp_path / "v.otslam")))

    base = str(tmp_path / "scan")
    jobs = []
    for label, scene in (("Object_0", "table"), ("Object_1", "cone")):
        s = synth.make_sequence(scene, 12, subsample=(0, 2))
        synth.write_capture_tree(s, base, label=label)
        P = lambda sub, k, ext, label=label: os.path.join(base, sub, f"{label}_{k}.{ext}")
        triples = [(P("color", k, "jpg"), P("depth", k, "png"), P("poses", k, "txt"), k) for k in range(1, len(s) + 1)]
        jobs.append((I.ScalableTSDFVolume(0.01, 0.04, I.TSDFVolumeColorType.RGB8), triples, dict(intrinsics=intr, T_fix=synth.T_FIX)))
    assert pipeline.integrate_many(jobs) == [6, 6]
    for k, (v, _, _) in enumerate(jobs):
        p = str(tmp_path / f"obj{k}.otslam")
        v.save(p)
        same_mesh(v, I.ScalableTSDFVolume.load(p))
