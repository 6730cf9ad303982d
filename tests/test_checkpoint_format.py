"""Checkpoint file format version 1 (DESIGN.md §4), restated in NumPy: a file written here to the documented layout is
accepted by otslam_checkpoint_info (host only, no GPU), and damaged headers / sizes are refused.  The helpers are also
used by tests/test_gpu_checkpoint.py to read, check and alter files the library wrote."""
import ctypes as C
import struct

import numpy as np
import pytest

MAGIC = b"OTSLAMCK"
PAGE = 4096
BLOCK_BYTES = 65536
GOLDEN = np.uint64(0x9E3779B97F4A7C15)
HEADER = struct.Struct("<8sIIIiddqq")          # magic, version, record bytes, voxels per block, colour, vl, trunc, frames, n


def mix(x):
    """splitmix64 of every element (uint64, wrapping arithmetic)."""
    with np.errstate(over="ignore"):
        x = np.asarray(x, np.uint64) + GOLDEN
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return x ^ (x >> np.uint64(31))


def word_sum(words):
    """sum_i mix(w[i] ^ (i * golden)) mod 2^64"""
    w = np.frombuffer(bytes(words), "<u8") if not isinstance(words, np.ndarray) else words.view("<u8").ravel()
    return int(np.sum(mix(w ^ (np.arange(len(w), dtype=np.uint64) * GOLDEN)), dtype=np.uint64))


def pack_key(x, y, z):
    """the library's pack_key, also for keys outside the range (each biased field taken as uint32, shifted, mod 2^64)"""
    b, m = 1 << 20, (1 << 32) - 1
    return ((((x + b) & m) << 42) | (((y + b) & m) << 21) | ((z + b) & m)) & ((1 << 64) - 1)


def block_checksum(records, key):
    """records: 65536 bytes of one block; key: (x, y, z) as stored in the file"""
    return (int(mix(np.uint64(pack_key(*(int(k) for k in key))))) + word_sum(records)) % (1 << 64)


def pad(n):
    return (n + PAGE - 1) // PAGE * PAGE


def layout(n):
    keys_off = PAGE
    cks_off = keys_off + pad(12 * n)
    rec_off = cks_off + pad(8 * n)
    return keys_off, cks_off, rec_off, rec_off + n * BLOCK_BYTES


def header(voxel_length, sdf_trunc, color_type, frames, n_blocks, version=1, magic=MAGIC):
    h = bytearray(PAGE)
    HEADER.pack_into(h, 0, magic, version, 16, 4096, color_type, voxel_length, sdf_trunc, frames, n_blocks)
    h[4088:] = struct.pack("<Q", word_sum(h[:4088]))
    return h


def write(path, keys, records, voxel_length=0.005, sdf_trunc=0.02, color_type=1, frames=1):
    """keys i32 [n][3] ascending, records u8 [n][65536]"""
    keys = np.ascontiguousarray(keys, np.int32).reshape(-1, 3)
    records = np.ascontiguousarray(records, np.uint8).reshape(len(keys), BLOCK_BYTES)
    n = len(keys)
    keys_off, cks_off, rec_off, total = layout(n)
    buf = bytearray(total)
    buf[:PAGE] = header(voxel_length, sdf_trunc, color_type, frames, n)
    buf[keys_off:keys_off + 12 * n] = keys.tobytes()
    cks = np.array([block_checksum(records[i].tobytes(), keys[i]) for i in range(n)], np.uint64)
    buf[cks_off:cks_off + 8 * n] = cks.tobytes()
    buf[rec_off:] = records.tobytes()
    open(path, "wb").write(bytes(buf))


def parse(blob):
    """(header fields dict, keys [n][3], checksums [n], records [n][65536] u8) of a file's bytes"""
    magic, version, rb, vpb, color, vl, tr, frames, n = HEADER.unpack_from(blob, 0)
    keys_off, cks_off, rec_off, total = layout(n)
    assert len(blob) == total
    keys = np.frombuffer(blob, np.int32, 3 * n, keys_off).reshape(n, 3)
    cks = np.frombuffer(blob, np.uint64, n, cks_off)
    rec = np.frombuffer(blob, np.uint8, n * BLOCK_BYTES, rec_off).reshape(n, BLOCK_BYTES)
    hdr = dict(magic=magic, version=version, record_bytes=rb, voxels_per_block=vpb, color_type=color, voxel_length=vl,
               sdf_trunc=tr, frames=frames, n_blocks=n, checksum=struct.unpack_from("<Q", blob, 4088)[0])
    return hdr, keys, cks, rec


def with_header(blob, **fields):
    """The same file with header fields replaced and the header checksum recomputed."""
    h, *_ = parse(blob)
    h.update(fields)
    out = bytearray(blob)
    out[:PAGE] = header(h["voxel_length"], h["sdf_trunc"], h["color_type"], h["frames"], h["n_blocks"], h["version"], h["magic"])
    return bytes(out)


def sample_records(n, seed=0):
    """n blocks of valid-looking records: count <= 40, colour sums <= 255 * count"""
    rng = np.random.default_rng(seed)
    w = rng.integers(0, 41, (n, 4096)).astype(np.uint32)
    r = np.zeros((n, 4096, 4), np.uint32)
    r[..., 0] = rng.random((n, 4096), np.float32).view(np.uint32)
    for c in range(3):
        r[..., 1 + c] = (rng.random((n, 4096)) * 255 * w).astype(np.uint32)
    r[..., 1] |= (w & 0xFF) << 24
    r[..., 2] |= (w >> 8) << 24
    return r.view(np.uint8).reshape(n, BLOCK_BYTES)


def info(path):
    from otslam_b200 import _lib
    vl, tr, ct, fr, nb = C.c_double(), C.c_double(), C.c_int32(), C.c_int64(), C.c_int64()
    st = _lib.lib.otslam_checkpoint_info(str(path).encode(), C.byref(vl), C.byref(tr), C.byref(ct), C.byref(fr), C.byref(nb))
    return st, (vl.value, tr.value, ct.value, fr.value, nb.value)


def test_numpy_written_file_is_accepted(tmp_path):
    from otslam_b200.volume import checkpoint_info
    keys = np.array([[-3, 0, 5], [-3, 1, -2], [0, 0, 0], [7, -1, 2]], np.int32)
    p = tmp_path / "a.otslam"
    write(p, keys, sample_records(4), voxel_length=0.005, sdf_trunc=0.02, color_type=1, frames=40)
    assert info(p) == (0, (0.005, 0.02, 1, 40, 4))
    assert checkpoint_info(p) == {"voxel_length": 0.005, "sdf_trunc": 0.02, "color": True, "frames": 40, "n_blocks": 4}
    assert p.stat().st_size == 4096 + 4096 + 4096 + 4 * 65536
    e = tmp_path / "empty.otslam"
    write(e, np.zeros((0, 3), np.int32), np.zeros((0, BLOCK_BYTES), np.uint8), color_type=0, frames=0)
    assert info(e) == (0, (0.005, 0.02, 0, 0, 0)) and e.stat().st_size == 4096


def test_checksum_restatement_matches_the_definition():
    """c = mix(pack_key) + sum_i mix(w[i] ^ (i * golden)), one word at a time in plain Python integers"""
    M = (1 << 64) - 1

    def mix1(x):
        x = (x + 0x9E3779B97F4A7C15) & M
        x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M
        x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & M
        return x ^ (x >> 31)
    rec = sample_records(1, seed=3)[0].tobytes()
    words = struct.unpack("<8192Q", rec)
    want = (mix1(pack_key(-5, 2, 1)) + sum(mix1(w ^ ((i * 0x9E3779B97F4A7C15) & M)) for i, w in enumerate(words))) & M
    assert block_checksum(rec, (-5, 2, 1)) == want


def test_damaged_headers_and_sizes_are_refused(tmp_path):
    from otslam_b200 import _lib
    keys = np.array([[0, 0, 0], [0, 0, 1]], np.int32)
    good = tmp_path / "good.otslam"
    write(good, keys, sample_records(2), frames=40)
    blob = good.read_bytes()
    cases = {
        "magic": with_header(blob, magic=b"OTSLAMXX"),
        "version": with_header(blob, version=2),
        "corrupt": blob[:30] + bytes([blob[30] ^ 1]) + blob[31:],          # header byte flipped, checksum kept
        "truncated": blob[:-1],
        "short": blob[:100],
        "n_blocks": with_header(blob, n_blocks=3),
        "frames": with_header(blob, frames=70000),
    }
    for name, b in cases.items():
        p = tmp_path / f"{name}.otslam"
        p.write_bytes(b)
        st, _ = info(p)
        assert st == _lib.ERR_FORMAT, name
    assert info(tmp_path / "missing.otslam")[0] == _lib.ERR_INVALID
    assert _lib.lib.otslam_checkpoint_info(None, None, None, None, None, None) == _lib.ERR_INVALID
    assert info(good)[0] == _lib.OK


def test_save_and_load_validate_arguments_before_cuda(tmp_path):
    from otslam_b200 import _lib
    n = C.c_int64(7)
    assert _lib.lib.otslam_volume_save(None, str(tmp_path / "x").encode()) == _lib.ERR_INVALID
    assert _lib.lib.otslam_volume_load(None, str(tmp_path / "x").encode(), C.byref(n)) == _lib.ERR_INVALID
    assert _lib.lib.otslam_volume_load(None, None, None) == _lib.ERR_INVALID
    assert not (tmp_path / "x").exists()
    out = np.zeros(4, np.float64)
    assert _lib.lib.otslam_checkpoint_profile(_lib.ptr(out)) == _lib.OK
    assert _lib.lib.otslam_checkpoint_profile(None) == _lib.ERR_INVALID
    with pytest.raises(RuntimeError):
        from otslam_b200.volume import checkpoint_info
        checkpoint_info(tmp_path / "x")
