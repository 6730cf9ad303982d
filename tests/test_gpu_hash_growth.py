"""Growth of the block hash (csrc/hash_table.cuh, volume.cu: grow_hash / reserve_hash).  The table starts at 2^18 entries
and holds at most half of them, so a volume grows it when it passes 131 072 blocks: in the middle of an integrate_batch
call (the batches already allocated in the old table are allocated again), and up front in a checkpoint load.  A grown
volume must hold exactly what a volume that never grew holds."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

VL = 0.0015                 # room sequence below: ~124 k blocks after 20 frames, ~240 k after 64
GROWTH_BLOCKS = 1 << 17     # the initial 2^18-entry table holds at most this many keys


@pytest.fixture(scope="module")
def room():
    """64 frames of a 96-frame room trajectory, 640x480."""
    from otslam_b200 import synth
    seq = synth.make_sequence("room", 96, poses=synth.trajectory("room", 96)[:64], device="cuda")
    d, c = seq.numpy()
    return seq, d, c


def block_keys(v):
    """the sorted block keys alone (export_blocks without the voxel arrays, which would take gigabytes here)"""
    from otslam_b200 import _lib
    keys = np.empty((v.num_blocks(), 3), np.int32)
    _lib.check(_lib.lib.otslam_volume_export_blocks(v._h, _lib.ptr(keys), None, None, None))
    return keys


def digest(v, seq, views):
    """block count, weight sums, sorted keys and ray-cast depth / normal / colour maps from a few poses"""
    out = v.ray_cast(seq.fxfycxcy, seq.extrinsic[views], 640, 480, attributes=("depth", "normal", "color"))
    assert (out["depth"] > 0).mean() > 0.25
    return v.stats(), block_keys(v), out


def assert_same(a, b):
    assert a[0] == b[0]
    assert a[1].shape == b[1].shape and (a[1] == b[1]).all()
    for k in a[2]:
        assert a[2][k].tobytes() == b[2][k].tobytes(), k


@pytest.mark.parametrize("batch", [32, 7])
def test_growth_during_integration(room, batch):
    """The table grows while the call's batches are in flight (batch 32: after batch 0, batch 1 already allocated; batch
    7: after batch 3); after reset() the capacity stays, so the second pass never grows and must give the same volume."""
    from otslam_b200.volume import TSDFVolume
    seq, d, c = room
    v = TSDFVolume(VL, 4 * VL)
    if batch != 32:
        v.set_batch(batch)
    v.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    assert v.num_blocks() > GROWTH_BLOCKS, "the workload no longer grows the table"
    views = [0, 21, 42, 63]
    grown = digest(v, seq, views)
    assert grown[0]["n_blocks"] == v.num_blocks()
    v.reset()
    v.integrate_batch(d, c, seq.fxfycxcy, seq.extrinsic)
    assert_same(grown, digest(v, seq, views))
    v.close()


def test_growth_during_checkpoint_load(room, tmp_path):
    """Object 0 of a two-object arena sits just below the threshold; loading a checkpoint into object 1 grows the table.
    Object 1 then equals the saved volume bit for bit, and object 0 is unchanged."""
    from otslam_b200.volume import ArenaView, TSDFVolume
    seq, d, c = room
    intr, ext = seq.fxfycxcy, seq.extrinsic
    src = TSDFVolume(VL, 4 * VL)
    src.integrate_batch(d[20:24], c[20:24], intr, ext[20:24])
    p = tmp_path / "src.otslam"
    src.save(p)

    arena = TSDFVolume(VL, 4 * VL)
    arena.set_objects(2)
    obj0, obj1 = ArenaView(arena, 0), ArenaView(arena, 1)
    obj0.integrate_batch(d[:20], c[:20], intr, ext[:20])
    n0 = obj0.num_blocks()
    assert n0 <= GROWTH_BLOCKS < n0 + src.num_blocks(), "the load no longer grows the table"
    before = digest(obj0, seq, [0, 10, 19])
    assert obj1.load(p) == src.num_blocks()
    assert_same(before, digest(obj0, seq, [0, 10, 19]))
    assert_same(digest(src, seq, [20, 23]), digest(obj1, seq, [20, 23]))
    es, e1 = src.export_blocks(color=False), obj1.export_blocks(color=False)
    assert (es[1].view(np.uint32) == e1[1].view(np.uint32)).all() and (es[2] == e1[2]).all()
    src.close(); arena.close()
