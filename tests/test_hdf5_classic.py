"""host/hdf5_classic.py: the reader against a libhdf5-written file, the writer against the reader and against a
byte-level walk of what libhdf5 checks when it opens a classic-format file (seam B5: reference
run/dino_features.py:109-153 writes, datasets/vit_dataset.py:83-84 / tomo_dataset.py:110-123 read)."""
import os
import struct
import zlib
from pathlib import Path

import numpy as np
import pytest

from cryovit_b200.host import hdf, hdf5_classic as h5c


def _libhdf5_file():
    """A file written by libhdf5 itself (MATLAB 7.3 = HDF5 behind a 512-byte user block): scipy's test file
    scipy/io/matlab/tests/data/testhdf5_7.4_GLNX86.mat (BSD-3-Clause), stored byte for byte."""
    return Path(__file__).resolve().parent / "golden" / "testhdf5_7.4_GLNX86.mat"


def test_reader_parses_a_libhdf5_written_file():
    with h5c.File(_libhdf5_file()) as fh:
        assert fh.base == 512 and fh.leaf_k == 4 and fh.internal_k == 16
        assert fh.eof == os.path.getsize(_libhdf5_file())  # absolute end-of-file address
        assert fh.keys() == ["testdouble"]
        info = fh.info("testdouble")
        assert info.layout == "contiguous" and info.dtype == np.dtype("<f8") and info.shape == (9, 1)
        np.testing.assert_allclose(fh.read("testdouble")[:, 0], np.arange(9) * np.pi / 4, rtol=0, atol=1e-15)


def _walk(path):
    """What libhdf5 validates on open / traversal: signature and version bytes, every structure inside the end-of-file
    address, node fill <= 2K, group names strictly increasing with B-tree keys naming each node's last entry, chunk
    keys strictly increasing (lexicographic) and below the node's right key, chunk payloads inflating to a whole
    chunk. Returns (datasets, chunk count)."""
    raw = Path(path).read_bytes()
    assert raw[:8] == h5c.SIGNATURE
    sb_ver, fs_ver, rg_ver, _, sh_ver, so, sl, _, leaf_k, int_k, flags = struct.unpack_from("<BBBBBBBBHHI", raw, 8)
    assert (sb_ver, fs_ver, rg_ver, sh_ver, so, sl, flags) == (0, 0, 0, 0, 8, 8, 0)
    base, free, eof, drv = struct.unpack_from("<QQQQ", raw, 24)
    assert base == 0 and free == h5c.UNDEF and drv == h5c.UNDEF and eof == len(raw)
    seen = {"datasets": 0, "chunks": 0}

    def inside(addr, size):
        assert addr % 8 == 0 and addr + size <= eof, (addr, size, eof)

    def messages(addr):
        ver, _, n, ref, size = struct.unpack_from("<BBHII", raw, addr)
        assert ver == 1 and ref == 1
        inside(addr, 16 + size)
        pos, out = addr + 16, []
        for _ in range(n):
            t, s, f = struct.unpack_from("<HHB", raw, pos)
            assert s % 8 == 0
            out.append((t, raw[pos + 8:pos + 8 + s]))
            pos += 8 + s
        assert pos == addr + 16 + size
        return out

    def heap_name(heap, off):
        sig, ver, size, free_head, data = struct.unpack_from("<4sB3xQQQ", raw, heap)
        assert sig == b"HEAP" and ver == 0 and size % 8 == 0 and free_head == h5c.FREE_NULL
        inside(heap, 32)
        inside(data, size)
        assert raw[data:data + 8] == b"\x00" * 8 and off % 8 == 0 and off < size
        return raw[data + off:raw.index(b"\x00", data + off)]

    def group(header, cached):
        msgs = messages(header)
        assert [t for t, _ in msgs] == [h5c.MSG_SYMBOL_TABLE]
        btree, heap = struct.unpack("<QQ", msgs[0][1])
        assert cached is None or cached == (btree, heap)
        node_size = 24 + (2 * int_k + 1) * 8 + 2 * int_k * 8
        inside(btree, node_size)
        sig, ntype, level, used, left, right = struct.unpack_from("<4sBBHQQ", raw, btree)
        assert (sig, ntype, level, left, right) == (b"TREE", 0, 0, h5c.UNDEF, h5c.UNDEF) and used <= 2 * int_k
        keys = [struct.unpack_from("<Q", raw, btree + 24 + 16 * i)[0] for i in range(used + 1)]
        assert keys[0] == 0
        prev = b""
        for i in range(used):
            snod = struct.unpack_from("<Q", raw, btree + 32 + 16 * i)[0]
            inside(snod, 8 + 2 * leaf_k * 40)
            sig, ver, _, n = struct.unpack_from("<4sBBH", raw, snod)
            assert sig == b"SNOD" and ver == 1 and 1 <= n <= 2 * leaf_k
            for j in range(n):
                off, obj, cache, _, bt, hp = struct.unpack_from("<QQIIQQ", raw, snod + 8 + 40 * j)
                name = heap_name(heap, off)
                assert name > prev, "links of a group are sorted by name"
                prev = name
                if cache == 1:
                    group(obj, (bt, hp))
                else:
                    assert cache == 0
                    dataset(obj)
            assert heap_name(heap, keys[i + 1]) == prev, "key i+1 names the last entry of node i"

    def dataset(header):
        msgs = dict(messages(header))
        seen["datasets"] += 1
        space, dtype, layout = msgs[h5c.MSG_DATASPACE], msgs[h5c.MSG_DATATYPE], msgs[h5c.MSG_LAYOUT]
        assert space[0] == 1 and h5c.MSG_FILL in msgs and msgs[h5c.MSG_FILL][:4] in (b"\x02\x02\x02\x01", b"\x02\x03\x02\x01")
        rank = space[1]
        shape = struct.unpack_from(f"<{rank}Q", space, 8)
        itemsize = struct.unpack_from("<I", dtype, 4)[0]
        assert layout[0] == 3
        if layout[1] == 1:
            addr, size = struct.unpack_from("<QQ", layout, 2)
            assert size == int(np.prod(shape, dtype=np.int64)) * itemsize
            if size:
                inside(addr, size)
            return
        assert layout[1] == 2 and layout[2] == rank + 1
        root = struct.unpack_from("<Q", layout, 3)[0]
        dims = struct.unpack_from(f"<{rank + 1}I", layout, 11)
        assert dims[-1] == itemsize
        pipeline = msgs[h5c.MSG_FILTERS]
        assert pipeline[:2] == b"\x01\x01" and struct.unpack_from("<HHHH", pipeline, 8) == (1, 8, 1, 1)
        assert pipeline[16:24] == b"deflate\x00"
        key_size = 8 + 8 * (rank + 1)
        node_size = 24 + (2 * h5c.CHUNK_K + 1) * key_size + 2 * h5c.CHUNK_K * 8
        chunk_bytes = int(np.prod(dims))

        def node(addr, want_level=None):
            inside(addr, node_size)
            sig, ntype, level, used, left, right = struct.unpack_from("<4sBBHQQ", raw, addr)
            assert sig == b"TREE" and ntype == 1 and 1 <= used <= 2 * h5c.CHUNK_K
            assert want_level is None or level == want_level
            keys, kids = [], []
            for i in range(used + 1):
                pos = addr + 24 + i * (key_size + 8)
                nbytes, mask = struct.unpack_from("<II", raw, pos)
                keys.append((struct.unpack_from(f"<{rank + 1}Q", raw, pos + 8), nbytes, mask))
                if i < used:
                    kids.append(struct.unpack_from("<Q", raw, pos + key_size)[0])
            assert all(a[0] < b[0] for a, b in zip(keys, keys[1:])), "chunk keys increase lexicographically"
            first_last = []
            for i, kid in enumerate(kids):
                if level == 0:
                    origin, nbytes, mask = keys[i]
                    assert mask == 0 and origin[-1] == 0 and all(o % d == 0 and o < s for o, d, s in zip(origin, dims, shape))
                    inside(kid, nbytes)
                    assert len(zlib.decompress(raw[kid:kid + nbytes])) == chunk_bytes
                    seen["chunks"] += 1
                else:
                    lo, hi = node(kid, level - 1)
                    assert lo == keys[i][0] and hi == keys[i + 1][0], "parent keys bracket the child"
            return keys[0][0], keys[-1][0]

        lo, hi = node(root)
        assert all(h >= s for h, s in zip(hi[:-1], shape)), "the last key lies beyond every chunk"

    _, root_header, cache, _, bt, hp = struct.unpack_from("<QQIIQQ", raw, 56)
    assert cache == 1
    group(root_header, (bt, hp))
    return seen


def test_tomogram_layout_round_trip_and_structure(tmp_path):
    rng = np.random.default_rng(0)
    sets = {
        "data": rng.integers(0, 255, (20, 70, 50), dtype=np.uint8),
        "labels/mito": rng.integers(-1, 2, (20, 70, 50)).astype(np.int8),
        "labels/granule": rng.integers(-1, 2, (20, 70, 50)).astype(np.int8),
        "dino_features": rng.standard_normal((16, 20, 5, 4)).astype(np.float16),
        "data_f32": rng.random((4, 9, 7), dtype=np.float32),
        "scalar": np.float64(3.5),
    }
    path = tmp_path / "t.hdf"
    h5c.write_file(path, sets, gzip={"data": 4, "labels/mito": 4, "labels/granule": 4, "data_f32": 4},
                   chunks={"data": (3, 32, 32)})  # ragged edge chunks on every axis
    with h5c.File(path) as fh:
        assert sorted(fh.keys()) == sorted(sets)
        assert fh.info("dino_features").layout == "contiguous" and fh.info("dino_features").filters == []
        assert fh.info("data").layout == "chunked" and fh.info("data").filters == [(h5c.FILTER_DEFLATE, (4,))]
        for k, v in sets.items():
            got = fh.read(k)
            assert got.dtype == np.asarray(v).dtype and got.shape == np.shape(v) and np.array_equal(got, v), k
        # the raw features sit in one piece at their address: a reader may map them
        info = fh.info("dino_features")
        mapped = np.memmap(path, np.float16, "r", offset=info.address, shape=info.shape)
        assert np.array_equal(mapped, sets["dino_features"])
    seen = _walk(path)
    assert seen["datasets"] == 6 and seen["chunks"] == 7 * 3 * 2 + 3  # data 7x3x2 ragged chunks; the labels and data_f32 fit one chunk each
    assert h5c.read_file(path, keys=["labels/mito"]).keys() == {"labels/mito"}


def test_multi_level_chunk_tree_and_wide_groups(tmp_path):
    rng = np.random.default_rng(1)
    x = rng.integers(0, 255, (300, 64, 64), dtype=np.uint8)
    many = {f"g/d{i:03d}": np.arange(i + 1, dtype=np.int32) for i in range(200)}  # 25 symbol-table nodes in one group
    path = tmp_path / "m.hdf"
    h5c.write_file(path, {"x": x, **many}, gzip={"x": 1}, chunks={"x": (1, 32, 32)}, threads=2)  # 1200 chunks: a two-level chunk B-tree
    got = h5c.read_file(path)
    assert np.array_equal(got["x"], x) and all(np.array_equal(got[k], v) for k, v in many.items())
    seen = _walk(path)
    assert seen == {"datasets": 201, "chunks": 1200}
    with pytest.raises(h5c.Hdf5FormatError):
        h5c.write_file(tmp_path / "bad.hdf", {"a": x, "a/b": x})


def test_reader_rejects_what_it_does_not_cover(tmp_path):
    p = tmp_path / "v2.hdf"
    p.write_bytes(h5c.SIGNATURE + bytes([2]) + b"\x00" * 87)
    with pytest.raises(h5c.Hdf5FormatError, match="superblock version 2"):
        h5c.File(p)
    q = tmp_path / "none.hdf"
    q.write_bytes(b"not an hdf5 file" * 8)
    assert not h5c.is_hdf5(q)
    with pytest.raises(ValueError):
        hdf.read_tomogram(q)
    good = tmp_path / "ok.hdf"
    h5c.write_file(good, {"data": np.zeros((4, 4, 4), np.uint8)}, gzip={"data": 4})
    cut = tmp_path / "cut.hdf"
    cut.write_bytes(good.read_bytes()[:200])
    with pytest.raises(h5c.Hdf5FormatError):
        h5c.read_file(cut)


def test_hdf_module_writes_real_hdf5_and_still_reads_the_zip_container(tmp_path, monkeypatch):
    sets = {"data": np.arange(2 * 16 * 16, dtype=np.uint8).reshape(2, 16, 16), "labels/mito": np.ones((2, 16, 16), np.int8),
            "dino_features": np.ones((8, 2, 1, 1), np.float16)}
    monkeypatch.delenv("CRYOVIT_HDF_BACKEND", raising=False)
    a = tmp_path / "a.hdf"
    hdf.write_tomogram(a, sets)
    if hdf.backend() == "hdf5-classic":
        assert a.read_bytes()[:8] == h5c.SIGNATURE
        with h5c.File(a) as fh:
            assert fh.info("data").layout == "chunked" and fh.info("dino_features").layout == "contiguous"
    assert sorted(hdf.list_keys(a)) == sorted(sets)
    monkeypatch.setenv("CRYOVIT_HDF_BACKEND", "npz")
    b = tmp_path / "b.hdf"
    hdf.write_tomogram(b, sets)
    assert b.read_bytes()[:2] == b"PK"
    monkeypatch.delenv("CRYOVIT_HDF_BACKEND")
    for f in (a, b):  # either container is read back whatever the write back end is now
        got = hdf.read_tomogram(f)
        assert all(np.array_equal(got[k], v) for k, v in sets.items())


def test_uncompressed_chunked_features(tmp_path):
    """dino_features in depth slabs (SURVEY.md 8f row f2's chunked option): chunk B-tree, no filter pipeline."""
    feats = np.random.default_rng(2).standard_normal((24, 10, 3, 5)).astype(np.float16)
    path = tmp_path / "f.hdf"
    h5c.write_file(path, {"dino_features": feats}, chunks={"dino_features": (24, 4, 3, 5)})
    with h5c.File(path) as fh:
        info = fh.info("dino_features")
        assert info.layout == "chunked" and info.chunks == (24, 4, 3, 5) and info.filters == []
        assert np.array_equal(fh.read("dino_features"), feats)


def test_round_trip_property():
    """Random shapes / dtypes / chunkings / compression levels survive the write -> read round trip bit for bit."""
    import tempfile

    from hypothesis import given, settings, strategies as st

    dtypes = [np.uint8, np.int8, np.int16, np.uint16, np.int32, np.int64, np.float16, np.float32, np.float64]

    @settings(max_examples=40, deadline=None)
    @given(st.data())
    def run(data):
        rank = data.draw(st.integers(1, 4))
        shape = tuple(data.draw(st.integers(1, 9)) for _ in range(rank))
        dtype = data.draw(st.sampled_from(dtypes))
        chunk = tuple(data.draw(st.integers(1, s + 2)) for s in shape)
        level = data.draw(st.sampled_from([None, 1, 4, 9]))
        chunked = level is not None or data.draw(st.booleans())
        arr = np.random.default_rng(data.draw(st.integers(0, 1 << 30))).integers(0, 120, shape).astype(dtype)
        with tempfile.TemporaryDirectory() as d:
            path = Path(d) / "p.hdf"
            h5c.write_file(path, {"grp/x": arr, "y": arr.T.copy()}, gzip={"grp/x": level} if level is not None else None,
                           chunks={"grp/x": chunk} if chunked else None, threads=1)
            got = h5c.read_file(path)
            assert got["grp/x"].dtype == arr.dtype and np.array_equal(got["grp/x"], arr) and np.array_equal(got["y"], arr.T)
            if chunked:
                _walk_if_deflate(path, level)

    def _walk_if_deflate(path, level):
        if level is not None:
            _walk(path)

    run()


def test_filter_pipeline_is_undone_in_reverse_order():
    """shuffle -> deflate -> fletcher32, as h5py applies them with shuffle=True, compression="gzip", fletcher32=True; a
    chunk whose filter mask skipped deflate (libhdf5 does that when a chunk does not shrink); unknown filters refuse."""
    raw = np.arange(600, dtype=np.int32)
    shuffled = raw.view(np.uint8).reshape(-1, 4).T.tobytes()
    stored = zlib.compress(shuffled, 4) + b"\x12\x34\x56\x78"
    filters = [(h5c.FILTER_SHUFFLE, (4,)), (h5c.FILTER_DEFLATE, (4,)), (h5c.FILTER_FLETCHER32, ())]
    assert h5c.undo_filters(stored, filters, 0, 4) == raw.tobytes()
    assert h5c.undo_filters(shuffled + b"\x00" * 4, filters, 0b010, 4) == raw.tobytes()
    with pytest.raises(h5c.Hdf5FormatError, match="filter 32015"):
        h5c.undo_filters(stored, [(32015, (3,))], 0, 4)


def test_an_unreadable_dataset_does_not_hide_the_others(tmp_path):
    """A dataset of a type outside the subset (here: the datatype class byte patched to 'string') is listed, refuses to
    be read with the reason, and leaves the tomogram's own datasets readable."""
    path = tmp_path / "s.hdf"
    data = np.arange(24, dtype=np.uint8).reshape(2, 3, 4)
    h5c.write_file(path, {"data": data, "note": np.zeros(5, np.int16)})
    raw = bytearray(path.read_bytes())
    i16 = struct.pack("<BBBBI", 0x10, 0x08, 0, 0, 2)  # the int16 datatype message body as the writer emits it
    at = raw.index(i16)
    raw[at] = 0x13  # class 3 = string
    path.write_bytes(bytes(raw))
    with h5c.File(path) as fh:
        assert sorted(fh.keys()) == ["data", "note"] and "class 3" in fh.info("note").error
        assert np.array_equal(fh.read("data"), data)
        with pytest.raises(h5c.Hdf5FormatError, match="note"):
            fh.read("note")
    assert np.array_equal(hdf.read_tomogram(path, keys=["data"])["data"], data)
