"""Labeling gzip HDF5 datasets of any chunk shape from their compressed chunks (device inflate + frame gather).

h5py is not installed here, so _ChunkedGzip stands in for an h5py dataset with gzip chunks of any shape: it writes one
real zlib stream per chunk (edge chunks at the full chunk size, zero past the dataset's extent, as HDF5 stores them) to
a file in shuffled order and has the attributes _zchunk_table reads (shape, dtype, chunks, compression, shuffle,
fletcher32, scaleoffset, id.get_chunk_info_by_coord / get_create_plist, file.filename); id.get_num_chunks /
get_chunk_info give the whole chunk index, as h5py's do.
CPU: which datasets take the compressed-chunk path and which keep h5py; routing between label_zfile, label_zchunks and
the slab path; each shard's row_lo and chunk table; the C ABI refuses a null handle.
GPU (-m gpu): arp_label_zchunks gives arp_label_file's bits over chunk layouts, frame sizes, max_batch boundaries and
row_lo inside a chunk, with chunks that hold no scored frame filled with garbage; embed / tower records likewise; a
corrupt needed chunk is named by its logical origin and the handle stays usable; refusals; arp_gather_frames against
numpy indexing; the drop-in writes from each layout what it writes from an NpyStore."""
import ctypes as C
import itertools
import os
import zlib
from collections import namedtuple

import numpy as np
import pytest
import torch

from arp_b200.label_reward import _zchunk_table, _zfile_rows

StoreInfo = namedtuple("StoreInfo", "chunk_offset filter_mask byte_offset size")


def _chunk_grid(shape, chunks):
    return list(itertools.product(*[range(0, s, c) for s, c in zip(shape, chunks)]))


def _chunk_of(arr, origin, chunks):
    """the full-size chunk at `origin`, zero past the dataset's extent"""
    out = np.zeros(chunks, np.uint8)
    src = arr[tuple(slice(o, o + c) for o, c in zip(origin, chunks))]
    out[tuple(slice(0, n) for n in src.shape)] = src
    return out


class _ChunkedGzip:
    """uint8 array `arr` as gzip chunks of shape `chunks` in `path`, with h5py's attributes and chunk index.
    garbage(origin) -> True: that chunk's stored bytes are random (it must never be read); streams: origin -> bytes
    overrides a chunk's stream; missing: origins left unallocated; filter_mask: origin -> mask."""

    def __init__(self, path, arr, chunks, level=4, compression="gzip", shuffle=False, fletcher32=False,
                 scaleoffset=None, nfilters=None, filter_mask=None, missing=(), garbage=None, streams=None, seed=0):
        arr = np.ascontiguousarray(arr)
        self.shape, self.dtype, self.chunks = arr.shape, arr.dtype, tuple(chunks)
        self.compression, self.compression_opts = compression, level
        self.shuffle, self.fletcher32, self.scaleoffset = shuffle, fletcher32, scaleoffset
        self._arr = arr
        rng = np.random.default_rng(seed)
        origins = _chunk_grid(arr.shape, self.chunks)
        data = {}
        for o in origins:
            if garbage is not None and garbage(o):
                data[o] = rng.integers(0, 256, int(rng.integers(1, 64)), dtype=np.uint8).tobytes()
            else:
                data[o] = zlib.compress(_chunk_of(arr, o, self.chunks).tobytes(), level)
        data.update(streams or {})
        place = {}
        with open(path, "wb") as f:
            f.write(b"\x89HDF-like header\n")
            for i in rng.permutation(len(origins)):
                place[origins[i]] = (f.tell(), len(data[origins[i]]))
                f.write(data[origins[i]])
        self._infos = [StoreInfo(o, (filter_mask or {}).get(o, 0), *place[o]) for o in origins if o not in missing]
        self._infos = [self._infos[i] for i in rng.permutation(len(self._infos))]
        self._by_origin = {info.chunk_offset: info for info in self._infos}
        self.lookups = []                              # origins asked for through get_chunk_info_by_coord
        nf = (1 + bool(shuffle)) if nfilters is None else nfilters
        ds = self

        class _Plist:
            def get_nfilters(self):
                return nf

        class _Id:
            def get_num_chunks(self):
                return len(ds._infos)

            def get_chunk_info(self, i):
                return ds._infos[i]

            def get_chunk_info_by_coord(self, origin):
                origin = tuple(int(v) for v in origin)
                ds.lookups.append(origin)
                return ds._by_origin.get(origin, StoreInfo(origin, 0, None, 0))   # h5py: no address when unallocated

            def get_create_plist(self):
                return _Plist()

        class _File:
            filename = os.fspath(path)

        self.id, self.file = _Id(), _File()

    @property
    def ndim(self):
        return len(self.shape)

    def __len__(self):
        return self.shape[0]

    def __getitem__(self, idx):
        return self._arr[idx]


def _rows(T=20, size=64, F=4, seed=0, w=None):
    from arp_b200.synth import make_dataset
    d = make_dataset(n_episodes=T // 4 + 1, len_lo=4, len_hi=5, size=size, num_frames=F, seed=seed, kind="structured")
    ob = np.ascontiguousarray(d["ob"][:T])
    if w is not None:                       # a non-square frame: the rows cut to width w (or tiled past it)
        ob = np.ascontiguousarray(np.concatenate([ob] * (-(-w // size)), axis=-2)[..., :w, :])
    return ob


def _layouts(F, H, W):
    """name -> (chunks, 4-D?) over the shapes the tests cover"""
    return {
        "row": ((1, F, H, W, 3), False),
        "rows3": ((3, F, H, W, 3), False),
        "frames8": ((8, 1, H, W, 3), False),
        "tiles": ((5, 2, H // 2, W // 2, 3), False),
        "channels": ((4, 1, H // 2 + 3, W, 2), False),   # channel split, partial edge chunks along T, H and C
        "4d": ((3, H // 2, W // 3 + 1, 3), True),
    }


# ------------------------------------------------------------------------------------------------
# CPU: eligibility, routing, shard tables
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["row", "rows3", "frames8", "tiles", "channels", "4d"])
def test_eligible_layouts_give_the_needed_chunks(tmp_path, name):
    ob = _rows()
    T, F, H, W = ob.shape[:4]
    chunks, four = _layouts(F, H, W)[name]
    arr = np.ascontiguousarray(ob[:, -1]) if four else ob
    ds = _ChunkedGzip(tmp_path / "d.h5", arr, chunks)
    path, (shape, ch), origins, off, nb = _zchunk_table(ds, 5, 17)
    assert path == os.fspath(tmp_path / "d.h5") and shape == arr.shape and ch == chunks
    raw = (tmp_path / "d.h5").read_bytes()
    fc = 0 if four else (F - 1) // chunks[1]
    want = {o for o in _chunk_grid(arr.shape, chunks)
            if 5 // chunks[0] <= o[0] // chunks[0] <= 16 // chunks[0] and (four or o[1] // chunks[1] == fc)}
    assert {tuple(o) for o in origins} == want
    assert sorted(ds.lookups) == sorted(want)          # only the needed chunks are looked up
    for o, a, n in zip(origins, off, nb):
        assert zlib.decompress(raw[a:a + n]) == _chunk_of(arr, tuple(o), chunks).tobytes()


def test_shuffle_is_accepted_on_uint8(tmp_path):
    ob = _rows()
    assert _zchunk_table(_ChunkedGzip(tmp_path / "d.h5", ob, (2,) + ob.shape[1:], shuffle=True)) is not None
    # the recorder layout with shuffle is not a zfile dataset, but a zchunks one
    ds = _ChunkedGzip(tmp_path / "e.h5", ob, (1,) + ob.shape[1:], shuffle=True)
    assert _zfile_rows(ds) is None and _zchunk_table(ds) is not None


def _bad_kw(ob):
    T, F, H, W = ob.shape[:4]
    last = (0, F - 1, 0, 0, 0)                     # chunk (1, 1, H, W, 3) holding row 0's scored frame
    return {"lzf": dict(compression="lzf"), "none": dict(compression=None), "fletcher32": dict(fletcher32=True),
            "scaleoffset": dict(scaleoffset=0), "third-filter": dict(shuffle=True, nfilters=3),
            "unnamed-filter": dict(nfilters=2), "missing": dict(missing={last}),
            "filter-mask": dict(filter_mask={last: 1})}


@pytest.mark.parametrize("case", list(_bad_kw(np.zeros((1, 4, 1, 1, 3)))))
def test_ineligible_datasets_keep_the_h5py_path(tmp_path, case):
    ob = _rows()
    ds = _ChunkedGzip(tmp_path / "d.h5", ob, (1, 1) + ob.shape[2:], **_bad_kw(ob)[case])
    assert _zchunk_table(ds) is None


def test_a_missing_chunk_of_unscored_frames_is_accepted(tmp_path):
    ob = _rows()
    F = ob.shape[1]
    ds = _ChunkedGzip(tmp_path / "d.h5", ob, (1, 1) + ob.shape[2:], missing={(3, 0, 0, 0, 0), (7, F - 2, 0, 0, 0)},
                      filter_mask={(4, 1, 0, 0, 0): 1})
    assert _zchunk_table(ds) is not None


def test_the_scratch_bound_is_refused(tmp_path, monkeypatch):
    from arp_b200 import capi
    ob = _rows()
    ds = _ChunkedGzip(tmp_path / "d.h5", ob, (4, 1) + ob.shape[2:])
    vol = 4 * ob[0, 0].nbytes
    monkeypatch.setattr(capi, "ZCHUNK_SCRATCH_BYTES", 3 * vol)
    assert _zchunk_table(ds, max_batch=8) is not None            # 8 rows touch at most 3 chunks of 4 rows
    assert _zchunk_table(ds, max_batch=9) is not None            # so do 9
    assert _zchunk_table(ds, max_batch=10) is None               # 10 rows may touch 4


def test_a_needed_chunk_over_the_compressed_bound_keeps_the_h5py_path(tmp_path, monkeypatch):
    from arp_b200 import capi
    ob = _rows()
    ds = _ChunkedGzip(tmp_path / "d.h5", ob, (4, 1) + ob.shape[2:])
    largest = int(_zchunk_table(ds)[4].max())        # the largest needed chunk
    monkeypatch.setattr(capi, "ZCHUNK_MAX_COMPRESSED_BYTES", largest)
    assert _zchunk_table(ds) is not None
    monkeypatch.setattr(capi, "ZCHUNK_MAX_COMPRESSED_BYTES", largest - 1)
    assert _zchunk_table(ds) is None


def test_datasets_without_a_chunk_index_keep_their_path(tmp_path):
    from arp_b200.store import NpyStore
    s = NpyStore(tmp_path / "s", "w")
    s.create_dataset("ob", data=_rows())
    assert _zchunk_table(s["ob"]) is None
    s.close()


class _RecordingLabeler:
    """records which call _label_rows / _embed_rows chose and what it passed"""
    goal = False
    embedding_dim = 4
    max_batch = 8

    def __init__(self):
        self.calls = []

    def label_zfile(self, fd, offsets, sizes, row_bytes, rel, num_frames):
        self.calls.append(("zfile", len(offsets)))
        return self._out(len(offsets), num_frames)

    def embed_zfile(self, fd, offsets, sizes, row_bytes):
        self.calls.append(("zfile", len(offsets)))
        return np.zeros((len(offsets), 4), np.float32)

    def label_zchunks(self, fd, layout, origins, offsets, sizes, row_lo, T, rel, num_frames):
        self.calls.append(("zchunks", row_lo, T, {tuple(o) for o in origins}, layout))
        return self._out(T, num_frames)

    def embed_zchunks(self, fd, layout, origins, offsets, sizes, row_lo, T):
        self.calls.append(("zchunks", row_lo, T, {tuple(o) for o in origins}, layout))
        return np.zeros((T, 4), np.float32)

    def label_slab(self, ob, rel, num_frames):
        self.calls.append(("slab", len(ob)))
        return self._out(len(ob), num_frames)

    def embed_slab(self, ob):
        self.calls.append(("slab", len(ob)))
        return np.zeros((len(ob), 4), np.float32)

    @staticmethod
    def _out(T, F):
        return np.zeros(T, np.float32), None, np.zeros((T, F), np.float32), np.zeros((T, F), np.float32)


def test_routing_recorder_layout_other_layouts_and_sidecar(tmp_path):
    from arp_b200.label_reward import _embed_rows, _label_rows
    ob = _rows()
    off = np.array([0, 20], np.int64)
    lab = _RecordingLabeler()
    _label_rows(lab, _ChunkedGzip(tmp_path / "a.h5", ob, (1,) + ob.shape[1:]), None, off, 0, 1, 4, 1 << 14)
    _embed_rows(lab, _ChunkedGzip(tmp_path / "a.h5", ob, (1,) + ob.shape[1:]), None, off, 0, 1, 1 << 14)
    assert [c[0] for c in lab.calls] == ["zfile", "zfile"]
    lab.calls.clear()
    ds = _ChunkedGzip(tmp_path / "b.h5", ob, (3, 2) + ob.shape[2:])
    _label_rows(lab, ds, None, off, 0, 1, 4, 1 << 14)
    _embed_rows(lab, ds, None, off, 0, 1, 1 << 14)
    assert [c[0] for c in lab.calls] == ["zchunks", "zchunks"]
    lab.calls.clear()
    _label_rows(lab, ds, np.ascontiguousarray(ob[:, -1]), off, 0, 1, 4, 1 << 14)
    assert [c[0] for c in lab.calls] == ["slab"]


def test_each_shard_gets_its_row_lo_and_chunk_table(tmp_path):
    from arp_b200.label_reward import _embed_rows, _label_rows
    from arp_b200.sharding import partition_episodes
    ob = _rows(T=20)
    F = ob.shape[1]
    chunks = (3, 2) + ob.shape[2:]
    ds = _ChunkedGzip(tmp_path / "d.h5", ob, chunks)
    off = np.array([0, 4, 7, 11, 16, 20], np.int64)
    lab = _RecordingLabeler()
    for e_lo, e_hi in partition_episodes(off, 3):
        lo, hi = int(off[e_lo]), int(off[e_hi])
        _label_rows(lab, ds, None, off, e_lo, e_hi, 4, 1 << 14)
        _embed_rows(lab, ds, None, off, e_lo, e_hi, 1 << 14)
        want = {(r, (F - 1) // 2 * 2, 0, 0, 0) for r in range(lo // 3 * 3, hi, 3)}
        for kind, row_lo, T, origins, layout in lab.calls[-2:]:
            assert kind == "zchunks" and (row_lo, T) == (lo, hi - lo) and origins == want
            assert layout == (ob.shape, chunks)


def test_c_abi_refuses_a_null_handle(built_lib):
    from arp_b200 import capi
    lib = capi.load_library()
    tab = np.zeros(5, np.int64)
    hp = C.c_void_p(tab.ctypes.data)
    lay = capi.chunk_layout((2, 4, 64, 64, 3), (1, 4, 64, 64, 3))
    assert lib.arp_label_zchunks(None, 0, C.byref(lay), hp, hp, hp, 1, 0, 2, hp, 1, 4, None, None, None,
                                 None) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_zchunks(None, 0, C.byref(lay), hp, hp, hp, 1, 0, 2, hp) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_zchunks(None, 0, C.byref(lay), hp, hp, hp, 1, 0, 2, hp) == capi.ARP_ERR_INVALID
    assert lib.arp_gather_frames(None, C.byref(lay), 0, 1, hp, hp, None) == capi.ARP_ERR_INVALID


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def capi():
    from arp_b200 import capi as m
    from arp_b200.build import build
    build()
    return m


def _sds():
    from arp_b200.weights import random_adapter_state_dict, random_clip_state_dict
    clip_sd = random_clip_state_dict("ViT-B/32", 0, "cpu")
    return clip_sd, random_adapter_state_dict("ViT-B/32", seed=1, device="cpu", clip_sd=clip_sd)


_SDS = {}


def _engine(capi, model_type, H, W, groups=1, max_batch=8):
    from test_embeddings import _text
    from test_instruction_sets import COINRUN_TYPES
    from arp_b200.instructions import get_clip_instruct, get_clip_special_instruct
    from arp_b200.label_reward import _head_for
    if not _SDS:
        _SDS["clip"], _SDS["adapter"] = _sds()
    sd = _SDS["adapter" if "ft" in model_type else "clip"]
    head, pre = _head_for(model_type)
    e = capi.Engine(device=0, patch=32, in_h=H, in_w=W, preprocess=pre, head=head, max_batch=max_batch)
    assert not e.load_state_dict(sd)
    texts = [[get_clip_instruct("coinrun") if t == "none" else get_clip_special_instruct("coinrun", t)]
             for t in COINRUN_TYPES][:groups]
    _text(capi, e, sd, texts, groups > 1)
    return e


def _episodes(T_all, row_lo, T):
    """relative episode offsets over rows [row_lo, row_lo + T): episodes of 3-7 rows"""
    cuts = np.cumsum(np.random.default_rng(T_all + row_lo).integers(3, 8, T))
    return np.concatenate([[0], cuts[cuts < T], [T]]).astype(np.int64)


def _data(tmp_path, name, size, w=None, garbage=True):
    """(dataset array, chunks, stand-in, raw-file fd): 41 rows, F = 4; chunks without frame F-1 hold garbage"""
    ob = _rows(T=41, size=size, F=4, seed=size, w=w)
    T, F, H, W = ob.shape[:4]
    chunks, four = _layouts(F, H, W)[name]
    arr = np.ascontiguousarray(ob[:, -1]) if four else ob
    fc = None if four else (F - 1) // chunks[1]
    junk = (lambda o: o[1] // chunks[1] != fc) if garbage and not four else None
    ds = _ChunkedGzip(tmp_path / f"{name}.h5", arr, chunks, garbage=junk)
    (tmp_path / "raw.bin").write_bytes(arr.tobytes())
    return arr, chunks, ds


def _raw_args(arr, row_lo):
    frame = int(np.prod(arr.shape[-3:]))
    stride = frame * (arr.shape[1] if arr.ndim == 5 else 1)
    return row_lo * stride + stride - frame, stride


_CASES = [(name, size, None) for name in ("row", "rows3", "frames8", "tiles", "channels", "4d") for size in (64, 256)]
_CASES.append(("tiles", 64, 96))


@pytest.mark.gpu
@pytest.mark.parametrize("name,size,w", _CASES, ids=[f"{n}-{s}" + (f"x{w}" if w else "") for n, s, w in _CASES])
def test_label_zchunks_equals_label_file(capi, tmp_path, name, size, w):
    """clip head with 3 instruction sets, max_batch 8, row_lo = 5 inside a chunk of every multi-row layout"""
    arr, chunks, ds = _data(tmp_path, name, size, w)
    H, W = arr.shape[-3:-1]
    e = _engine(capi, "clip", H, W, groups=3)
    row_lo, T = 5, 33
    ep = _episodes(len(arr), row_lo, T)
    path, layout, origins, off, nb = _zchunk_table(ds, row_lo, row_lo + T, 8)
    fd_raw, fd_z = os.open(tmp_path / "raw.bin", os.O_RDONLY), os.open(path, os.O_RDONLY)
    try:
        base, stride = _raw_args(arr, row_lo)
        want = e.label_file(fd_raw, base, T, stride, ep, 4)
        got = e.label_zchunks(fd_z, layout, origins, off, nb, row_lo, T, ep, 4)
        for i, (a, b) in enumerate(zip(got, want)):
            assert a.shape == b.shape and np.array_equal(a, b), i
        if name == "row":                      # the recorder layout: also arp_label_zfile's bits on all rows
            full = _zfile_rows(_ChunkedGzip(tmp_path / "z.h5", arr, chunks))
            fd_f = os.open(full[0], os.O_RDONLY)
            try:
                ep_all = _episodes(len(arr), 0, len(arr))
                zf = e.label_zfile(fd_f, full[1], full[2], full[3], ep_all, 4)
            finally:
                os.close(fd_f)
            tab = _zchunk_table(ds)
            zc = e.label_zchunks(fd_z, tab[1], tab[2], tab[3], tab[4], 0, len(arr), ep_all, 4)
            for a, b in zip(zf, zc):
                assert np.array_equal(a, b)
    finally:
        os.close(fd_raw)
        os.close(fd_z)
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model_type", ["clip_ft", "clip_goal_conditioned"])
@pytest.mark.parametrize("name", ["tiles", "channels", "row"])
def test_label_zchunks_heads(capi, tmp_path, model_type, name):
    arr, chunks, ds = _data(tmp_path, name, 64)
    e = _engine(capi, model_type, 64, 64)
    row_lo, T = 7, 30
    ep = _episodes(len(arr), row_lo, T)
    path, layout, origins, off, nb = _zchunk_table(ds, row_lo, row_lo + T, 8)
    fd_raw, fd_z = os.open(tmp_path / "raw.bin", os.O_RDONLY), os.open(path, os.O_RDONLY)
    try:
        base, stride = _raw_args(arr, row_lo)
        want = e.label_file(fd_raw, base, T, stride, ep, 4)
        got = e.label_zchunks(fd_z, layout, origins, off, nb, row_lo, T, ep, 4)
    finally:
        os.close(fd_raw)
        os.close(fd_z)
    for i, (a, b) in enumerate(zip(got, want)):
        assert a.shape == b.shape and np.array_equal(a, b), i
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model_type,tower", [("clip", False), ("clip_ft", False), ("clip_ft", True)])
def test_embed_zchunks_equals_embed_file(capi, tmp_path, model_type, tower):
    arr, chunks, ds = _data(tmp_path, "tiles", 64)
    e = _engine(capi, model_type, 64, 64)
    row_lo, T = 3, 36
    path, layout, origins, off, nb = _zchunk_table(ds, row_lo, row_lo + T, 8)
    fd_raw, fd_z = os.open(tmp_path / "raw.bin", os.O_RDONLY), os.open(path, os.O_RDONLY)
    try:
        base, stride = _raw_args(arr, row_lo)
        if tower:
            want = e.embed_tower_file(fd_raw, base, T, stride)
            got = e.embed_tower_zchunks(fd_z, layout, origins, off, nb, row_lo, T)
        else:
            want = e.embed_file(fd_raw, base, T, stride)
            got = e.embed_zchunks(fd_z, layout, origins, off, nb, row_lo, T)
    finally:
        os.close(fd_raw)
        os.close(fd_z)
    assert got.shape == want.shape and np.array_equal(got, want)
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiles", "frames8", "channels", "4d"])
def test_the_whole_table_is_passed_and_unneeded_chunks_are_never_read(capi, tmp_path, name):
    """the library gets every chunk of the dataset, in index order; every chunk that holds no scored frame of rows
    [row_lo, row_lo + T) (another F-chunk, or rows outside the call) is random bytes, so reading or inflating one fails
    the call, and packing one into a batch or picking the wrong F-chunk changes the frames"""
    ob = _rows(T=41, size=64, F=4, seed=64)
    F, H, W = ob.shape[1:4]
    chunks, four = _layouts(F, H, W)[name]
    arr = np.ascontiguousarray(ob[:, -1]) if four else ob
    row_lo, T = 6, 27
    rc_lo, rc_hi = row_lo // chunks[0], (row_lo + T - 1) // chunks[0]
    fc = 0 if four else (F - 1) // chunks[1]
    unneeded = lambda o: not rc_lo <= o[0] // chunks[0] <= rc_hi or (not four and o[1] // chunks[1] != fc)  # noqa: E731
    ds = _ChunkedGzip(tmp_path / "all.h5", arr, chunks, garbage=unneeded)
    (tmp_path / "raw.bin").write_bytes(arr.tobytes())
    infos = [ds.id.get_chunk_info(i) for i in range(ds.id.get_num_chunks())]
    assert sum(map(unneeded, (i.chunk_offset for i in infos))) > len(infos) // 4
    origins = np.array([i.chunk_offset for i in infos], np.int64)
    off = np.array([i.byte_offset for i in infos], np.int64)
    nb = np.array([i.size for i in infos], np.int64)
    layout = (arr.shape, chunks)
    e = _engine(capi, "clip", H, W, groups=3)
    ep = _episodes(len(arr), row_lo, T)
    fd_raw, fd_z = os.open(tmp_path / "raw.bin", os.O_RDONLY), os.open(tmp_path / "all.h5", os.O_RDONLY)
    try:
        base, stride = _raw_args(arr, row_lo)
        want = e.label_file(fd_raw, base, T, stride, ep, 4)
        got = e.label_zchunks(fd_z, layout, origins, off, nb, row_lo, T, ep, 4)
        for i, (a, b) in enumerate(zip(got, want)):
            assert a.shape == b.shape and np.array_equal(a, b), i
        want_emb = e.embed_file(fd_raw, base, T, stride)
        got_emb = e.embed_zchunks(fd_z, layout, origins, off, nb, row_lo, T)
        assert np.array_equal(got_emb, want_emb)
    finally:
        os.close(fd_raw)
        os.close(fd_z)
    e.close()


@pytest.mark.gpu
def test_corrupt_chunk_is_named_by_origin_and_the_handle_stays_usable(capi, tmp_path):
    arr, chunks, ds = _data(tmp_path, "tiles", 64)
    e = _engine(capi, "clip", 64, 64)
    T = len(arr)
    ep = _episodes(T, 0, T)
    bad = (10, 2, 32, 0, 0)
    s = zlib.compress(_chunk_of(arr, bad, chunks).tobytes(), 4)
    bad_ds = _ChunkedGzip(tmp_path / "bad.h5", arr, chunks, streams={bad: s[:-1] + bytes([s[-1] ^ 1])})
    tab = _zchunk_table(bad_ds)
    fd = os.open(tab[0], os.O_RDONLY)
    out = [np.full(a.shape, 7, a.dtype) for a in e._host_outputs(T, 4)]
    try:
        with pytest.raises(capi.ArpError) as ei:
            e.label_zchunks(fd, tab[1], tab[2], tab[3], tab[4], 0, T, ep, 4, out=out)
    finally:
        os.close(fd)
    msg = str(ei.value)
    assert ei.value.code == capi.ARP_ERR_INVALID and "logical origin (10, 2, 32, 0, 0)" in msg, msg
    assert "row 10 of the call" in msg, msg
    assert "Adler-32 mismatch" in msg and "ArpInflateStatus 8" in msg, msg
    assert all((a == 7).all() for a in out)                     # nothing written
    tab = _zchunk_table(ds)
    fd_raw, fd = os.open(tmp_path / "raw.bin", os.O_RDONLY), os.open(tab[0], os.O_RDONLY)
    try:
        base, stride = _raw_args(arr, 0)
        want = e.label_file(fd_raw, base, T, stride, ep, 4)
        got = e.label_zchunks(fd, tab[1], tab[2], tab[3], tab[4], 0, T, ep, 4)
    finally:
        os.close(fd_raw)
        os.close(fd)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    e.close()


@pytest.mark.gpu
def test_c_abi_refusals(capi, tmp_path):
    arr, chunks, ds = _data(tmp_path, "tiles", 64, garbage=False)
    e = _engine(capi, "clip", 64, 64)
    T = len(arr)
    ep = _episodes(T, 0, T)
    _, layout, origins, off, nb = _zchunk_table(ds)
    fd = os.open(ds.file.filename, os.O_RDONLY)

    def refused(*, layout=layout, origins=origins, off=off, nb=nb, row_lo=0, T=T, ep=ep, match=""):
        with pytest.raises(capi.ArpError) as ei:
            e.label_zchunks(fd, layout, origins, off, nb, row_lo, T, ep, 4)
        assert ei.value.code == capi.ARP_ERR_INVALID and match in str(ei.value), str(ei.value)

    try:
        shape = arr.shape
        refused(layout=((T, 4, 64, 48, 3), chunks), match="dataset shape")
        refused(layout=(shape, (5, 2, 0, 32, 3)), match="chunk extent")
        refused(row_lo=1, T=T, match="not inside the dataset")
        o = origins.copy()
        o[3, 2] += 1
        refused(origins=o, match="not a multiple of the chunk shape")
        o = origins.copy()
        o[4] = o[5]
        refused(origins=o, match="share the logical origin")
        refused(origins=origins[1:], off=off[1:], nb=nb[1:], match="is not in the chunk table")
        neg = off.copy()
        neg[2] = -1
        refused(off=neg, match="negative file offset")
        big = nb.copy()
        big[0] = (64 << 20) + 1                        # one needed chunk larger than a pinned staging slot
        refused(nb=big, match="staging slot")
        # the scratch bound: one chunk of 2^20 rows of four 64x64 frames inflates to 48 GiB
        ep8 = np.array([0, 8], np.int64)
        refused(layout=((1 << 21, 4, 64, 64, 3), (1 << 20, 4, 64, 64, 3)), origins=np.zeros((1, 5), np.int64),
                off=off[:1], nb=nb[:1], T=8, ep=ep8, match="one chunk inflates to more than")
        # ... and a batch of 8 rows across two row-chunks of 1 GiB channel chunks needs 6 GiB (no chunk is read)
        big = [(r, 3, 0, 0, c) for r in (0, 1 << 18) for c in range(3)]
        refused(layout=((1 << 19, 4, 64, 64, 3), (1 << 18, 1, 64, 64, 1)), origins=np.array(big, np.int64),
                off=off[:6], nb=nb[:6], row_lo=(1 << 18) - 4, T=8, ep=ep8, match="one max_batch batch")
        # still usable
        base, stride = _raw_args(arr, 0)
        fd_raw = os.open(tmp_path / "raw.bin", os.O_RDONLY)
        want = e.label_file(fd_raw, base, T, stride, ep, 4)
        os.close(fd_raw)
        got = e.label_zchunks(fd, layout, origins, off, nb, 0, T, ep, 4)
        for a, b in zip(got, want):
            assert np.array_equal(a, b)
    finally:
        os.close(fd)
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,size", [("tiles", 64), ("channels", 64), ("rows3", 256), ("4d", 256)])
def test_gather_frames_matches_numpy_indexing(capi, tmp_path, name, size):
    ob = _rows(T=41, size=size, F=4, seed=1)
    T, F, H, W = ob.shape[:4]
    chunks, four = _layouts(F, H, W)[name]
    arr = np.ascontiguousarray(ob[:, -1]) if four else ob
    c5 = chunks if not four else (chunks[0], 1) + chunks[1:]
    s5 = arr.shape if not four else (T, 1) + arr.shape[1:]
    e = capi.Engine(device=0, patch=32, in_h=H, in_w=W, max_batch=8)
    for row0, n in ((0, 8), (5, 8), (37, 4), (11, 1)):
        blobs = []
        for rc in range(row0 // c5[0], (row0 + n - 1) // c5[0] + 1):
            for o in itertools.product(*[range(0, s, c) for s, c in zip(s5[2:], c5[2:])]):
                o5 = (rc * c5[0], (F - 1 if not four else 0) // c5[1] * c5[1]) + o
                blobs.append(_chunk_of(arr, o5 if not four else (o5[0],) + o5[2:], chunks).ravel())
        got = e.gather_frames((arr.shape, chunks), row0, n, torch.from_numpy(np.concatenate(blobs)).cuda())
        want = arr[row0:row0 + n, -1] if not four else arr[row0:row0 + n]
        assert np.array_equal(got.cpu().numpy(), want), (row0, n)
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["row", "rows3", "frames8", "tiles", "channels"])
def test_drop_in_writes_the_same_datasets_from_each_layout(tmp_path, monkeypatch, name):
    import arp_b200.label_reward as lr
    from arp_b200.store import NpyStore
    from arp_b200.synth import make_dataset, write_dataset
    from test_embeddings import _read
    data = make_dataset(n_episodes=6, len_lo=3, len_hi=11, size=64, num_frames=4, seed=5, kind="structured", tail_rows=2)
    plain, zipped = tmp_path / "plain", tmp_path / "zipped"
    for p in (plain, zipped):
        s = NpyStore(p, "w")
        write_dataset(s, data)
        s.close()
    chunks, _ = _layouts(4, 64, 64)[name]
    gz = _ChunkedGzip(tmp_path / "ob.h5", data["ob"], chunks, shuffle=name == "row")
    os.unlink(zipped / "ob.npy")

    class _Store(NpyStore):
        def __getitem__(self, key):
            return gz if key == "ob" else super().__getitem__(key)

        def get(self, key, default=None):
            return gz if key == "ob" else super().get(key, default)

    real_open = lr.open_store
    monkeypatch.setattr(lr, "open_store", lambda path, mode="a": _Store(path, mode) if str(path) == str(zipped)
                        else real_open(path, mode))
    seen = []
    real = lr.RewardLabeler.label_zchunks, lr.RewardLabeler.embed_zchunks
    monkeypatch.setattr(lr.RewardLabeler, "label_zchunks", lambda self, *a: seen.append(1) or real[0](self, *a))
    monkeypatch.setattr(lr.RewardLabeler, "embed_zchunks", lambda self, *a: seen.append(1) or real[1](self, *a))
    sd = __import__("arp_b200.weights", fromlist=["x"]).random_clip_state_dict("ViT-B/32", 0, "cpu")
    for p in (plain, zipped):
        lr.label_reward("coinrun", "hard", 500, 0, "the goal is to collect the coin.", str(tmp_path), data_path=str(p),
                        model_type="clip", clip_state_dict=sd, arch="ViT-B/32", max_batch=8, env_type="none",
                        tokenizer="standin", embeddings="save")
    assert seen, "the gzip chunks did not take the compressed-chunk path"
    want, got = _read(plain), _read(zipped)
    assert sorted(got) == sorted(want) and want
    for k in want:
        assert got[k].tobytes() == want[k].tobytes() and got[k].dtype == want[k].dtype, k
