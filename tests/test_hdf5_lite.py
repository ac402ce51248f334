"""hdf5_lite — the dependency-free HDF5 behind the result files (Data_prepare.py:243-246, Shared_extraction.py:32-40,
Tools/DNN_tools.py:286-287) where h5py is not installed.

Anchor: a file written by the HDF5 library itself — tests/golden/testhdf5_7.4_GLNX86.mat, MATLAB 7.3 test data from
scipy's test suite (scipy/io/matlab/tests/data, BSD-licensed), which is HDF5 behind a 512-byte user block.  The reader
must decode it; the writer's structures are compared with that file's bytes one by one, checked against the consistency
rules the library applies when it opens a file, and round-tripped through the reader."""
import os
import struct
import sys
import zlib

import numpy as np
import pytest

import saa_b200  # noqa: F401
from saa_b200 import hdf5_lite as h5
from util import GOLDEN, ROOT, bits_equal

PKG = os.path.join(ROOT, "synchronization-avoiding-algorithms_b200")


def _genuine():
    return os.path.join(GOLDEN, "testhdf5_7.4_GLNX86.mat")


def _messages(buf, addr):
    ver, _, n, ref, size = struct.unpack_from("<BBHII", buf, addr)
    out, p = [], addr + 16
    while p < addr + 16 + size:
        t, s, fl = struct.unpack_from("<HHB", buf, p)
        out.append((t, fl, buf[p + 8:p + 8 + s]))
        p += 8 + s
    assert ver == 1 and ref == 1 and len(out) == n and p == addr + 16 + size      # NIL messages count (library rule)
    return out


def test_reader_decodes_a_file_written_by_the_hdf5_library():
    d = h5.read_file(_genuine())
    assert list(d) == ["testdouble"] and d["testdouble"].shape == (9, 1) and d["testdouble"].dtype == np.float64
    assert bits_equal(d["testdouble"].ravel(), np.arange(9) * (np.pi / 4))      # MATLAB's 0:pi/4:2*pi
    with h5.File(_genuine(), "r") as f:
        assert f.keys() == ["testdouble"] and "testdouble" in f and f.get("nope") is None
        assert np.array(f["testdouble"]).shape == (9, 1)
        with pytest.raises(KeyError):
            f["nope"]


def test_writer_structures_equal_the_library_bytes(tmp_path):
    """Same array, same name as in the library-written file: datatype, dataspace and fill-value messages, the heap's
    name segment (empty string, name, free block with next = 1), the B-tree node header and keys, the symbol-table
    node entry and the superblock's format fields come out byte for byte as the library wrote them."""
    g = open(_genuine(), "rb").read()
    B = 512                                                         # user block: addresses in the file are relative to it
    path = str(tmp_path / "t.hdf5")
    h5.write_file(path, {"testdouble": (np.arange(9) * (np.pi / 4)).reshape(9, 1)})
    w = open(path, "rb").read()
    # superblock: signature, versions, sizes, K values (consistency flags / addresses differ by construction)
    assert w[:20] == g[B:B + 20] and w[8:16] == bytes([0, 0, 0, 0, 0, 8, 8, 0])
    g_root, w_root = struct.unpack_from("<Q", g, B + 64)[0] + B, struct.unpack_from("<Q", w, 64)[0]
    (gt, gf, gd), (wt, wf, wd) = _messages(g, g_root)[0], _messages(w, w_root)[0]
    assert (gt, gf, len(gd)) == (wt, wf, len(wd)) == (0x11, 1, 16)
    assert [m[0] for m in _messages(g, g_root)] == [m[0] for m in _messages(w, w_root)] == [0x11, 0]
    g_tree, g_heap = (x + B for x in struct.unpack("<QQ", gd))
    w_tree, w_heap = struct.unpack("<QQ", wd)
    assert struct.unpack_from("<QQ", w, 80) == (w_tree, w_heap)     # cached in the root entry's scratch pad, as the library does
    # local heap header + the whole 256-byte data segment
    assert g[g_heap:g_heap + 24] == w[w_heap:w_heap + 24]
    g_seg, w_seg = struct.unpack_from("<Q", g, g_heap + 24)[0] + B, struct.unpack_from("<Q", w, w_heap + 24)[0]
    assert g[g_seg:g_seg + 256] == w[w_seg:w_seg + 256]
    # B-tree node: signature, type, level, entries, siblings, key 0, (child), key 1
    assert g[g_tree:g_tree + 32] == w[w_tree:w_tree + 32] and g[g_tree + 40:g_tree + 48] == w[w_tree + 40:w_tree + 48]
    g_snod, w_snod = struct.unpack_from("<Q", g, g_tree + 32)[0] + B, struct.unpack_from("<Q", w, w_tree + 32)[0]
    assert g[g_snod:g_snod + 16] == w[w_snod:w_snod + 16]           # "SNOD", version, count, name offset of entry 0
    assert g[g_snod + 24:g_snod + 48] == w[w_snod + 24:w_snod + 48]  # cache type 0, reserved, empty scratch pad
    g_ds, w_ds = struct.unpack_from("<Q", g, g_snod + 16)[0] + B, struct.unpack_from("<Q", w, w_snod + 16)[0]
    gm = {t: (fl, d) for t, fl, d in _messages(g, g_ds)}
    wm = {t: (fl, d) for t, fl, d in _messages(w, w_ds)}
    for t in (0x01, 0x03, 0x05):                                    # dataspace, datatype, fill value: flags and bytes
        assert gm[t] == wm[t], hex(t)
    # data layout: the library of 2008 wrote version 2, the writer writes version 3 (contiguous: address, size)
    ver, cls, addr, size = struct.unpack_from("<BBQQ", wm[0x08][1])
    assert (ver, cls, size) == (3, 1, 72) and w[addr:addr + 72] == g[-72:] and addr + 72 == len(w)


def _check_like_the_library(buf):
    """The consistency rules the HDF5 library applies on open (H5F superblock, H5HL, H5B, H5G node, H5O version 1)."""
    assert buf[:8] == h5.SIGNATURE and buf[8] == 0 and buf[13] == 8 and buf[14] == 8
    leaf_k, int_k = struct.unpack_from("<HH", buf, 16)
    base, free, eof, drv = struct.unpack_from("<QQQQ", buf, 24)
    assert base == 0 and free == h5.UNDEF and drv == h5.UNDEF and eof == len(buf)             # "truncated file" otherwise
    name0, root, cache, _ = struct.unpack_from("<QQII", buf, 56)
    tree, heap = struct.unpack_from("<QQ", buf, 80)
    assert root % 8 == 0 and cache == 1
    msgs = _messages(buf, root)
    assert msgs[0][0] == 0x11 and struct.unpack("<QQ", msgs[0][2]) == (tree, heap)
    assert buf[heap:heap + 4] == b"HEAP" and buf[heap + 4] == 0
    seg_size, free_off, seg = struct.unpack_from("<QQQ", buf, heap + 8)
    assert seg_size % 8 == 0 and seg + seg_size <= len(buf)
    assert free_off == 1 or (free_off % 8 == 0 and free_off + 16 <= seg_size)                 # H5HL_FREE_NULL == 1
    if free_off != 1:
        nxt, fsz = struct.unpack_from("<QQ", buf, seg + free_off)
        assert nxt == 1 and free_off + fsz == seg_size
    assert buf[tree:tree + 4] == b"TREE" and buf[tree + 4] == 0 and buf[tree + 5] == 0
    used = struct.unpack_from("<H", buf, tree + 6)[0]
    assert used <= 2 * int_k and tree + 24 + (2 * int_k + 1) * 8 + 2 * int_k * 8 <= len(buf)  # nodes are read at full size
    assert struct.unpack_from("<QQ", buf, tree + 8) == (h5.UNDEF, h5.UNDEF)

    def name_at(off):
        return buf[seg + off:buf.index(b"\0", seg + off)]

    names, prev_key = [], name_at(struct.unpack_from("<Q", buf, tree + 24)[0])
    assert prev_key == b""
    for i in range(used):
        child, key = struct.unpack_from("<QQ", buf, tree + 32 + 16 * i)
        assert buf[child:child + 4] == b"SNOD" and buf[child + 4] == 1 and child + 8 + 2 * leaf_k * 40 <= len(buf)
        n = struct.unpack_from("<H", buf, child + 6)[0]
        assert 1 <= n <= 2 * leaf_k
        here = []
        for j in range(n):
            off, hdr, ctype, _ = struct.unpack_from("<QQII", buf, child + 8 + 40 * j)
            assert off % 8 == 0 and off < free_off and ctype == 0 and hdr % 8 == 0
            here.append(name_at(off))
            ds = {t: d for t, fl, d in _messages(buf, hdr)}
            assert {0x01, 0x03, 0x08} <= set(ds)
            ver, cls, addr, size = struct.unpack_from("<BBQQ", ds[0x08])
            assert (ver, cls) == (3, 1) and (size == 0 or addr + size <= eof)
            rank = ds[0x01][1]
            dims = struct.unpack_from(f"<{rank}Q", ds[0x01], 8)
            assert size == int(np.prod(dims, dtype=np.int64)) * struct.unpack_from("<I", ds[0x03], 4)[0]
        assert here == sorted(here) and prev_key < here[0] and here[-1] == name_at(key)       # keys bound the children
        prev_key = name_at(key)
        names += here
    assert names == sorted(names) and len(set(names)) == len(names)
    return [n.decode() for n in names]


@pytest.mark.parametrize("n_sets", [0, 1, 8, 9, 40])
def test_files_pass_the_library_checks_and_round_trip(tmp_path, n_sets):
    rng = np.random.default_rng(n_sets)
    dts = [np.float64, np.float32, np.int64, np.int32, np.uint8, np.float16, np.int16, np.uint64, np.bool_]
    data = {}
    for i in range(n_sets):
        shape = tuple(int(x) for x in rng.integers(0 if i % 7 == 6 else 1, 9, size=i % 4))
        a = (rng.standard_normal(shape) * 100)
        data[f"set_{(i * 37) % 101:03d}_{'x' * (i % 11)}"] = a.astype(dts[i % len(dts)])
    if n_sets:
        data["Displacement"] = rng.standard_normal((330, 25))
    path = str(tmp_path / "r.hdf5")
    h5.write_file(path, data)
    assert _check_like_the_library(open(path, "rb").read()) == sorted(data)
    back = h5.read_file(path)
    assert sorted(back) == sorted(data)
    for k, a in data.items():
        want = a.astype(np.int8) if a.dtype == np.bool_ else a
        assert back[k].shape == want.shape and back[k].dtype == want.dtype and bits_equal(back[k], want), k


def test_file_object_follows_the_reference_usage(tmp_path):
    """Data_prepare.py:243-246 / Shared_extraction.py:32-40 / DNN_tools.py:286-287, statement by statement."""
    d1_save = np.random.default_rng(3).standard_normal((330, 40))
    save_name = str(tmp_path / "Results" / "Dynamics" / "Local-rank-0.hdf5")
    hf = h5.File(save_name, "w")
    hf.create_dataset("Displacement", data=d1_save, compression="gzip")
    hf.close()
    assert open(save_name, "rb").read(8) == h5.SIGNATURE and not os.path.exists(save_name + ".npz")
    with h5.File(save_name, "r") as f:
        Data_numpy = f["Displacement"]
        Data_numpy = np.array(Data_numpy)
        d = Data_numpy[[3, 4, 5, 30, 31, 32], :]
    assert bits_equal(Data_numpy, d1_save)
    hf = h5.File(str(tmp_path / "shared.hdf5"), "w")
    hf.create_dataset("Displacement", data=d)
    hf.close()
    with h5.File(str(tmp_path / "shared.hdf5"), "r") as f:
        assert bits_equal(np.array(f["Displacement"]).transpose(), d.T)
    with pytest.raises(OSError):
        h5.File(save_name, "r").create_dataset("x", data=d)
    with pytest.raises(h5.Hdf5Error):
        h5.write_file(str(tmp_path / "bad.hdf5"), {"s": np.array(["a", "b"])})
    with pytest.raises(h5.Hdf5Error):
        h5.read_file(__file__)


def _chunked_file(path, a, chunk, gzip=True, shuffle=True, big_endian=False):
    """What h5py writes for create_dataset(..., chunks=chunk, compression='gzip', shuffle=True): filter pipeline message,
    version-3 chunked layout, one version-1 chunk B-tree node (type 1) with a key per chunk."""
    a = np.asarray(a)
    dt = a.dtype.newbyteorder(">" if big_endian else "<")
    rank, es = a.ndim, a.dtype.itemsize
    grid = [range(0, s, c) for s, c in zip(a.shape, chunk)]
    offs = np.stack(np.meshgrid(*grid, indexing="ij"), -1).reshape(-1, rank)
    blobs = []
    for o in offs:
        block = np.zeros(chunk, dtype=dt)
        sl = tuple(slice(x, min(x + c, s)) for x, c, s in zip(o, chunk, a.shape))
        block[tuple(slice(0, s.stop - s.start) for s in sl)] = a[sl]
        raw = block.tobytes()
        if shuffle:
            raw = np.frombuffer(raw, dtype=np.uint8).reshape(-1, es).T.tobytes()
        if gzip:
            raw = zlib.compress(raw, 4)
        blobs.append(raw)
    # a contiguous file with a placeholder gives every structure but the dataset header; rebuild that header
    h5.write_file(path, {"Displacement": np.zeros(1)})
    base = bytearray(open(path, "rb").read())
    snod = struct.unpack_from("<Q", base, struct.unpack_from("<Q", base, 80)[0] + 32)[0]
    hdr = struct.unpack_from("<Q", base, snod + 16)[0]
    del base[hdr:]
    filt = struct.pack("<BB6x", 1, int(shuffle) + int(gzip))
    if shuffle:
        filt += struct.pack("<HHHH", 2, 0, 1, 1) + struct.pack("<II", es, 0)
    if gzip:
        filt += struct.pack("<HHHH", 1, 0, 1, 1) + struct.pack("<II", 4, 0)
    tdt = bytearray(h5._datatype_message(a.dtype))
    tdt[1] |= 1 if big_endian else 0
    space = struct.pack("<BBB5x", 1, rank, 0) + b"".join(struct.pack("<Q", s) for s in a.shape)
    key = 8 + 8 * (rank + 1)
    tree_size = 24 + 2 * h5.CHUNK_K * 8 + (2 * h5.CHUNK_K + 1) * key
    msgs_wo_layout = h5._message(1, space) + h5._message(3, bytes(tdt), 1) + h5._message(0x0B, filt)
    layout_len = len(h5._message(8, struct.pack("<BBBQ", 3, 2, rank + 1, 0) + struct.pack(f"<{rank + 1}I", *chunk, es)))
    tree_at = hdr + 16 + len(msgs_wo_layout) + layout_len
    data_at = tree_at + tree_size
    tree = bytearray(b"TREE" + struct.pack("<BBHQQ", 1, 0, len(blobs), h5.UNDEF, h5.UNDEF))
    pos = data_at
    for o, raw in zip(offs, blobs):
        tree += struct.pack("<II", len(raw), 0) + struct.pack(f"<{rank + 1}Q", *o, 0) + struct.pack("<Q", pos)
        pos += len(raw)
    tree += struct.pack("<II", 0, 0) + struct.pack(f"<{rank + 1}Q", *a.shape, 0)        # final key: one past the last chunk
    tree += b"\0" * (tree_size - len(tree))
    layout = h5._message(8, struct.pack("<BBBQ", 3, 2, rank + 1, tree_at) + struct.pack(f"<{rank + 1}I", *chunk, es))
    body = msgs_wo_layout + layout
    base += struct.pack("<BBHII4x", 1, 0, 4, 1, len(body)) + body + tree + b"".join(blobs)
    struct.pack_into("<Q", base, 40, len(base))
    open(path, "wb").write(bytes(base))


@pytest.mark.parametrize("gzip,shuffle,big", [(True, True, False), (True, False, False), (False, False, True), (False, True, False)])
def test_reader_handles_chunked_filtered_datasets(tmp_path, gzip, shuffle, big):
    """`compression='gzip'` files of real h5py (Data_prepare.py:245) are chunked + deflate (+ shuffle): partial edge
    chunks, several chunks per axis, big-endian storage."""
    a = np.random.default_rng(5).standard_normal((330, 41))
    path = str(tmp_path / "c.hdf5")
    _chunked_file(path, a, (64, 16), gzip, shuffle, big)
    got = h5.read_file(path)["Displacement"]
    assert got.dtype == np.float64 and bits_equal(got, a)


def test_compat_h5py_writes_genuine_hdf5(tmp_path):
    """With no h5py installed, `import h5py` from compat/ writes real HDF5 at the path the caller names (no .npz);
    archives written by earlier versions of the stand-in are still readable."""
    import subprocess
    code = ("import h5py, numpy as np, sys\n"
            "a = np.arange(12.0).reshape(3, 4)\n"
            "hf = h5py.File('x.hdf5', 'w'); hf.create_dataset('Displacement', data=a, compression='gzip'); hf.close()\n"
            "assert open('x.hdf5', 'rb').read(8) == b'\\x89HDF\\r\\n\\x1a\\n'\n"
            "with h5py.File('x.hdf5', 'r') as f: assert np.array_equal(np.array(f['Displacement']), a)\n"
            "np.savez_compressed('old.hdf5.npz', Displacement=a + 1)\n"
            "with h5py.File('old.hdf5', 'r') as f: assert np.array_equal(f['Displacement'][:], a + 1)\n"
            "print('stand-in' if getattr(h5py, 'IS_STAND_IN', False) else 'real')\n")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([PKG, os.path.join(PKG, "compat")]))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() in ("stand-in", "real")
