"""Labeling gzip-chunked HDF5 rows from their compressed bytes (device zlib inflate).

h5py is not installed here, so _GzipDataset stands in for an h5py dataset chunked one row per chunk with gzip: it has
the attributes _zfile_rows reads (shape, dtype, chunks, compression, compression_opts, shuffle, fletcher32,
id.get_num_chunks / id.get_chunk_info, file.filename) over a real file of zlib streams, and __getitem__ inflates on the
host as h5py would.
CPU: which datasets take the compressed path and which keep the h5py path; each shard gets its own rows' chunk table;
the C ABI refuses a null handle.
GPU (-m gpu): arp_inflate_rows is byte-exact against zlib over levels, strategies, contents and both frame geometries;
arp_label_zfile / arp_embed_zfile / arp_embed_tower_zfile give the bits of their uncompressed twins; malformed streams
are reported with the right row and leave the handle usable; the drop-in writes from the gzip dataset what it writes
from an NpyStore of the same rows."""
import ctypes as C
import os
import zlib
from collections import namedtuple

import numpy as np
import pytest
import torch

from arp_b200.label_reward import _zfile_rows

TEXT = "the goal is to collect the coin."
StoreInfo = namedtuple("StoreInfo", "chunk_offset filter_mask byte_offset size")


class _GzipDataset:
    """uint8 rows [T, *row_shape] as one zlib stream per row in `path` (after a few header bytes, in shuffled order, as
    HDF5 places chunks wherever it allocates them), with h5py's attributes and chunk index."""

    def __init__(self, path, arr, level=4, streams=None, compression="gzip", chunks="row", shuffle=False,
                 fletcher32=False, filter_mask=None, missing=(), seed=0):
        arr = np.ascontiguousarray(arr)
        self.shape, self.dtype = arr.shape, arr.dtype
        self.chunks = (1,) + arr.shape[1:] if chunks == "row" else chunks
        self.compression, self.compression_opts = compression, level
        self.shuffle, self.fletcher32 = shuffle, fletcher32
        streams = list(streams) if streams is not None else [zlib.compress(r.tobytes(), level) for r in arr]
        order = np.random.default_rng(seed).permutation(len(streams))
        table = [None] * len(streams)
        with open(path, "wb") as f:
            f.write(b"\x89HDF-like header\n")
            for t in order:
                table[t] = (f.tell(), len(streams[t]))
                f.write(streams[t])
        self._infos = [StoreInfo((t,) + (0,) * (arr.ndim - 1), (filter_mask or {}).get(t, 0), o, n)
                       for t, (o, n) in enumerate(table) if t not in missing]
        self._infos = [self._infos[i] for i in np.random.default_rng(seed + 1).permutation(len(self._infos))]
        self._streams = streams
        ds = self

        class _Id:
            def get_num_chunks(self):
                return len(ds._infos)

            def get_chunk_info(self, i):
                return ds._infos[i]

        class _File:
            filename = os.fspath(path)

        self.id, self.file = _Id(), _File()

    @property
    def ndim(self):
        return len(self.shape)

    def __len__(self):
        return self.shape[0]

    def __getitem__(self, idx):
        rows = np.stack([np.frombuffer(zlib.decompress(s), np.uint8).reshape(self.shape[1:]) for s in self._streams])
        return rows[idx]


def _rows(T=12, size=64, F=4, seed=0):
    from arp_b200.synth import make_dataset
    d = make_dataset(n_episodes=max(1, T // 4), len_lo=4, len_hi=5, size=size, num_frames=F, seed=seed, kind="structured")
    return d["ob"][:T]


# ------------------------------------------------------------------------------------------------
# CPU: eligibility and chunk tables
# ------------------------------------------------------------------------------------------------
def test_eligible_dataset_gives_its_chunk_table(tmp_path):
    ob = _rows()
    ds = _GzipDataset(tmp_path / "d.h5", ob)
    path, off, nb, row_bytes = _zfile_rows(ds)
    assert path == os.fspath(tmp_path / "d.h5") and row_bytes == ob[0].nbytes
    raw = (tmp_path / "d.h5").read_bytes()
    for t in range(len(ob)):
        assert zlib.decompress(raw[off[t]:off[t] + nb[t]]) == ob[t].tobytes()
    # a 4-D dataset (one frame per row) is a row of F = 1
    assert _zfile_rows(_GzipDataset(tmp_path / "e.h5", ob[:, -1]))[3] == ob[0, -1].nbytes


@pytest.mark.parametrize("kw", [dict(compression="lzf"), dict(compression=None), dict(shuffle=True),
                                dict(fletcher32=True), dict(chunks="two"), dict(filter_mask={3: 1}),
                                dict(missing=(5,))], ids=lambda kw: next(iter(kw)))
def test_ineligible_datasets_keep_the_h5py_path(tmp_path, kw):
    ob = _rows()
    if kw.get("chunks") == "two":
        kw = dict(chunks=(2,) + ob.shape[1:])
    assert _zfile_rows(_GzipDataset(tmp_path / "d.h5", ob, **kw)) is None


def test_datasets_without_a_chunk_index_keep_their_path(tmp_path):
    from arp_b200.store import NpyStore
    s = NpyStore(tmp_path / "s", "w")
    s.create_dataset("ob", data=_rows())
    assert _zfile_rows(s["ob"]) is None
    s.close()


class _RecordingLabeler:
    """records which labeling call _label_rows / _embed_rows chose, and with which chunk rows"""
    goal = False
    embedding_dim = 4

    def __init__(self, raw):
        self.calls, self.raw = [], raw

    def label_zfile(self, fd, offsets, sizes, row_bytes, rel, num_frames):
        rows = [zlib.decompress(self.raw[o:o + n]) for o, n in zip(offsets, sizes)]
        self.calls.append(("zfile", rows, row_bytes))
        return self._out(len(rows), num_frames)

    def embed_zfile(self, fd, offsets, sizes, row_bytes):
        self.calls.append(("zfile", [zlib.decompress(self.raw[o:o + n]) for o, n in zip(offsets, sizes)], row_bytes))
        return np.zeros((len(offsets), 4), np.float32)

    def label_slab(self, ob, rel, num_frames):
        self.calls.append(("slab", [r.tobytes() for r in ob], None))
        return self._out(len(ob), num_frames)

    def embed_slab(self, ob):
        self.calls.append(("slab", [r.tobytes() for r in ob], None))
        return np.zeros((len(ob), 4), np.float32)

    @staticmethod
    def _out(T, F):
        return np.zeros(T, np.float32), None, np.zeros((T, F), np.float32), np.zeros((T, F), np.float32)


def test_each_shard_gets_its_own_rows_chunk_table(tmp_path):
    from arp_b200.label_reward import _embed_rows, _label_rows
    from arp_b200.sharding import partition_episodes
    ob = _rows(T=20)
    ds = _GzipDataset(tmp_path / "d.h5", ob)
    off = np.array([0, 3, 7, 12, 16, 20], np.int64)
    lab = _RecordingLabeler((tmp_path / "d.h5").read_bytes())
    for e_lo, e_hi in partition_episodes(off, 3):
        _label_rows(lab, ds, None, off, e_lo, e_hi, 4, 1 << 14)
        _embed_rows(lab, ds, None, off, e_lo, e_hi, 1 << 14)
        for kind, rows, row_bytes in lab.calls[-2:]:
            assert kind == "zfile" and row_bytes == ob[0].nbytes
            assert rows == [r.tobytes() for r in ob[off[e_lo]:off[e_hi]]]


def test_a_sidecar_keeps_the_h5py_path(tmp_path):
    from arp_b200.label_reward import _label_rows
    ob = _rows()
    ds = _GzipDataset(tmp_path / "d.h5", ob)
    side = np.ascontiguousarray(ob[:, -1])
    lab = _RecordingLabeler(b"")
    _label_rows(lab, ds, side, np.array([0, 12], np.int64), 0, 1, 4, 1 << 14)
    assert [c[0] for c in lab.calls] == ["slab"] and lab.calls[0][1] == [r.tobytes() for r in side]


def test_c_abi_refuses_a_null_handle(built_lib):
    from arp_b200 import capi
    lib = capi.load_library()
    tab = np.zeros(2, np.int64)
    hp = C.c_void_p(tab.ctypes.data)
    assert lib.arp_label_zfile(None, 0, hp, hp, 2, 49152, hp, 1, 4, None, None, None, None) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_zfile(None, 0, hp, hp, 2, 49152, hp) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_zfile(None, 0, hp, hp, 2, 49152, hp) == capi.ARP_ERR_INVALID
    assert lib.arp_inflate_rows(None, hp, hp, hp, 2, 49152, hp, hp, None) == capi.ARP_ERR_INVALID


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def capi():
    from arp_b200 import capi as m
    from arp_b200.build import build
    build()
    return m


def _compress(row: bytes, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    c = zlib.compressobj(level, zlib.DEFLATED, 15, 9, strategy)
    return c.compress(row) + c.flush()


def _corpus(size, F, seed=0):
    """(name, row bytes, zlib stream) over levels, strategies and contents, plus rows that force 258-byte matches and
    32 768-byte distances"""
    rng = np.random.default_rng(seed)
    n = size * size * 3 * F
    contents = {"random": rng.integers(0, 256, n, dtype=np.uint8).tobytes(), "constant": bytes([7]) * n,
                "procgen": _rows(T=1, size=size, F=F, seed=seed)[0].tobytes()}
    out = []
    for name, row in contents.items():
        out += [(f"{name}-l{lv}", row, zlib.compress(row, lv)) for lv in (0, 1, 4, 6, 9)]
        out += [(f"{name}-s{st}", row, _compress(row, 6, st))
                for st in (zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED)]
    period = rng.integers(0, 256, 32768, dtype=np.uint8).tobytes()          # repeats only at distance 32 768
    far = (period * (n // 32768 + 1))[:n]
    out.append(("distance-32768", far, zlib.compress(far, 9)))
    runs = b"".join(bytes([int(v)]) * 300 + bytes(rng.integers(0, 256, 7, dtype=np.uint8)) for v in rng.integers(0, 256, n // 300))
    runs = (runs + bytes(n))[:n]
    out.append(("length-258", runs, zlib.compress(runs, 9)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("size,F", [(64, 4), (256, 8)])
def test_inflate_rows_is_byte_exact_against_zlib(capi, size, F):
    corpus = _corpus(size, F)
    e = capi.Engine(device=0, patch=32, in_h=size, in_w=size, max_batch=4)
    src = b"".join(s for _, _, s in corpus)
    off = np.cumsum([0] + [len(s) for _, _, s in corpus[:-1]]).astype(np.int64)
    nb = np.array([len(s) for _, _, s in corpus], np.int64)
    rows, status = e.inflate_rows(torch.frombuffer(bytearray(src), dtype=torch.uint8).cuda(), torch.from_numpy(off),
                                  torch.from_numpy(nb), size * size * 3 * F)
    rows, status = rows.cpu().numpy(), status.cpu().numpy()
    for i, (name, row, _) in enumerate(corpus):
        assert status[i] == capi.ARP_INFLATE_OK and rows[i].tobytes() == row, name
    e.close()


def _sds():
    from arp_b200.weights import random_adapter_state_dict, random_clip_state_dict
    clip_sd = random_clip_state_dict("ViT-B/32", 0, "cpu")
    return clip_sd, random_adapter_state_dict("ViT-B/32", seed=1, device="cpu", clip_sd=clip_sd)


def _engine(capi, model_type, sd, max_batch=8):
    from arp_b200.label_reward import _head_for
    head, pre = _head_for(model_type)
    e = capi.Engine(device=0, patch=32, in_h=64, in_w=64, preprocess=pre, head=head, max_batch=max_batch)
    assert not e.load_state_dict(sd)
    return e


def _episodes(seed=3):
    from arp_b200.synth import make_dataset
    d = make_dataset(n_episodes=9, len_lo=3, len_hi=12, size=64, num_frames=4, seed=seed, kind="structured")
    ob = np.ascontiguousarray(d["ob"])
    return ob, np.concatenate([[0], np.cumsum(d["lengths"])]).astype(np.int64)


def _both_files(tmp_path, ob):
    """(fd of the raw rows, fd of the gzip rows, chunk offsets, chunk sizes)"""
    (tmp_path / "raw.bin").write_bytes(ob.tobytes())
    ds = _GzipDataset(tmp_path / "z.h5", ob)
    _, off, nb, _ = _zfile_rows(ds)
    return os.open(tmp_path / "raw.bin", os.O_RDONLY), os.open(tmp_path / "z.h5", os.O_RDONLY), off, nb


@pytest.mark.gpu
@pytest.mark.parametrize("model_type,groups", [("clip", 7), ("clip_ft", 1), ("clip_ft", 3), ("clip_goal_conditioned", 1),
                                               ("clip_ft_goal_conditioned", 1)])
def test_label_zfile_equals_label_file(capi, tmp_path, model_type, groups):
    """max_batch 8 against episodes of 3-11 rows: boundaries fall inside ring slots and across stager chunks"""
    from test_embeddings import _text
    from test_instruction_sets import COINRUN_TYPES
    from arp_b200.instructions import get_clip_instruct, get_clip_special_instruct
    clip_sd, adapter_sd = _sds()
    sd = adapter_sd if "ft" in model_type else clip_sd
    e = _engine(capi, model_type, sd)
    texts = [[get_clip_instruct("coinrun") if t == "none" else get_clip_special_instruct("coinrun", t)]
             for t in COINRUN_TYPES][:groups]
    _text(capi, e, sd, texts, groups > 1)
    ob, ep = _episodes()
    T, F = ob.shape[:2]
    frame = ob[0, 0].nbytes
    fd_raw, fd_z, off, nb = _both_files(tmp_path, ob)
    try:
        want = e.label_file(fd_raw, (F - 1) * frame, T, F * frame, ep, F)
        got = e.label_zfile(fd_z, off, nb, F * frame, ep, F)
    finally:
        os.close(fd_raw)
        os.close(fd_z)
    for i, (a, b) in enumerate(zip(got, want)):
        assert a.shape == b.shape and np.array_equal(a, b), i
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("model_type,tower", [("clip", False), ("clip_ft", False), ("clip_ft", True)])
def test_embed_zfile_equals_embed_file(capi, tmp_path, model_type, tower):
    clip_sd, adapter_sd = _sds()
    e = _engine(capi, model_type, adapter_sd if "ft" in model_type else clip_sd)
    ob, _ = _episodes()
    T, F = ob.shape[:2]
    frame = ob[0, 0].nbytes
    fd_raw, fd_z, off, nb = _both_files(tmp_path, ob)
    try:
        if tower:
            want = e.embed_tower_file(fd_raw, (F - 1) * frame, T, F * frame)
            got = e.embed_tower_zfile(fd_z, off, nb, F * frame)
        else:
            want = e.embed_file(fd_raw, (F - 1) * frame, T, F * frame)
            got = e.embed_zfile(fd_z, off, nb, F * frame)
    finally:
        os.close(fd_raw)
        os.close(fd_z)
    assert got.shape == want.shape and np.array_equal(got, want)
    e.close()


def _far_distance_stream(row_bytes):
    """a fixed-Huffman block: the literal 'a', then a 3-byte match at distance 5 (before the start of the row)"""
    acc, n = 0, 0

    def put(v, k, rev=False):
        nonlocal acc, n
        if rev:
            v = int(format(v, f"0{k}b")[::-1], 2)
        acc |= v << n
        n += k
    put(1, 1), put(1, 2)                       # BFINAL, BTYPE = fixed
    put(0x30 + ord("a"), 8, True)             # literal 'a'
    put(1, 7, True)                           # symbol 257: length 3
    put(4, 5, True), put(0, 1)                # distance symbol 4 + 1 extra bit: distance 5
    put(0, 7, True)                           # end of block
    return bytes([0x78, 0x01]) + acc.to_bytes((n + 7) // 8, "little") + b"\0\0\0\0"


@pytest.mark.gpu
def test_malformed_rows_are_reported_and_the_handle_stays_usable(capi, tmp_path):
    clip_sd, _ = _sds()
    e = _engine(capi, "clip", clip_sd)
    e.set_text(torch.nn.functional.normalize(torch.randn(1, 512), dim=1), 14.3)
    ob, ep = _episodes()
    T, F = ob.shape[:2]
    rb = ob[0].nbytes
    good = [zlib.compress(r.tobytes(), 4) for r in ob]
    fd_raw, fd_z, off, nb = _both_files(tmp_path, ob)
    want = e.label_file(fd_raw, rb - ob[0, 0].nbytes, T, rb, ep, F)
    os.close(fd_raw)
    os.close(fd_z)
    bad_row = 13
    s = good[bad_row]
    cases = {"truncated stream": s[:len(s) // 2], "bad zlib header": bytes([s[0] ^ 1]) + s[1:],
             "Adler-32 mismatch": s[:-1] + bytes([s[-1] ^ 1]),
             "distance before the start of the row": _far_distance_stream(rb),
             "output longer than row_bytes": zlib.compress(ob[bad_row].tobytes() + b"x", 4),
             "output shorter than row_bytes": zlib.compress(ob[bad_row].tobytes()[:-3], 4)}
    for k, (reason, stream) in enumerate(cases.items()):
        streams = list(good)
        streams[bad_row] = stream
        ds = _GzipDataset(tmp_path / f"bad{k}.h5", ob, streams=streams)
        _, boff, bnb, _ = _zfile_rows(ds)
        fd = os.open(tmp_path / f"bad{k}.h5", os.O_RDONLY)
        try:
            with pytest.raises(capi.ArpError) as ei:
                e.label_zfile(fd, boff, bnb, rb, ep, F)
        finally:
            os.close(fd)
        assert ei.value.code == capi.ARP_ERR_INVALID and f"row {bad_row} of the call" in str(ei.value), str(ei.value)
        assert reason in str(ei.value), (reason, str(ei.value))
        fd = os.open(tmp_path / "z.h5", os.O_RDONLY)
        try:
            got = e.label_zfile(fd, off, nb, rb, ep, F)
        finally:
            os.close(fd)
        for i, (a, b) in enumerate(zip(got, want)):
            assert np.array_equal(a, b), (reason, i)
    e.close()


@pytest.mark.gpu
def test_c_abi_refusals(capi):
    e = capi.Engine(device=0, patch=32, in_h=64, in_w=64, max_batch=4)
    lib, h = e._lib, e._h
    tab = np.zeros(3, np.int64)
    neg = np.array([0, -1, 0], np.int64)
    out = np.zeros((3, 4), np.float32)
    hp = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
    ep = np.array([0, 3], np.int64)
    rb = 64 * 64 * 3 * 4
    args = lambda fd, o, n, T, r: (h, fd, o, n, T, r, hp(ep), 1, 4, hp(out), hp(out), hp(out), hp(out))  # noqa: E731
    for bad in (args(-1, hp(tab), hp(tab), 3, rb), args(0, None, hp(tab), 3, rb), args(0, hp(tab), None, 3, rb),
                args(0, hp(tab), hp(tab), -1, rb), args(0, hp(neg), hp(tab), 3, rb), args(0, hp(tab), hp(neg), 3, rb),
                args(0, hp(tab), hp(tab), 3, rb + 1), args(0, hp(tab), hp(tab), 3, 0),
                args(0, hp(tab), hp(tab), 3, 64 * 64 * 3 * 65)):
        assert lib.arp_label_zfile(*bad) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_zfile(h, 0, hp(tab), hp(tab), 3, rb, None) == capi.ARP_ERR_INVALID
    assert lib.arp_embed_tower_zfile(h, 0, hp(tab), hp(tab), 3, rb, hp(out)) == capi.ARP_ERR_INVALID   # clip head
    d = torch.zeros(8, dtype=torch.int64, device="cuda")
    p = C.c_void_p(d.data_ptr())
    assert lib.arp_inflate_rows(h, p, p, p, -1, rb, p, p, None) == capi.ARP_ERR_INVALID
    assert lib.arp_inflate_rows(h, p, p, p, 2, rb - 3, p, p, None) == capi.ARP_ERR_INVALID
    assert lib.arp_inflate_rows(h, None, p, p, 2, rb, p, p, None) == capi.ARP_ERR_INVALID
    assert lib.arp_inflate_rows(h, p, p, p, 0, rb, p, p, None) == capi.ARP_OK
    e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("embeddings", [None, "save"])
def test_drop_in_writes_the_same_datasets_from_gzip_rows(tmp_path, monkeypatch, embeddings):
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
    gz = _GzipDataset(tmp_path / "ob.h5", data["ob"])
    os.unlink(zipped / "ob.npy")                       # the frames exist only as zlib streams

    class _Store(NpyStore):
        def __getitem__(self, key):
            return gz if key == "ob" else super().__getitem__(key)

        def get(self, key, default=None):
            return gz if key == "ob" else super().get(key, default)

    real_open = lr.open_store
    monkeypatch.setattr(lr, "open_store", lambda path, mode="a": _Store(path, mode) if str(path) == str(zipped)
                        else real_open(path, mode))
    seen = []
    real_zfile = lr.RewardLabeler.label_zfile, lr.RewardLabeler.embed_zfile
    monkeypatch.setattr(lr.RewardLabeler, "label_zfile", lambda self, *a: seen.append(1) or real_zfile[0](self, *a))
    monkeypatch.setattr(lr.RewardLabeler, "embed_zfile", lambda self, *a: seen.append(1) or real_zfile[1](self, *a))
    sd = __import__("arp_b200.weights", fromlist=["x"]).random_clip_state_dict("ViT-B/32", 0, "cpu")
    for p in (plain, zipped):
        lr.label_reward("coinrun", "hard", 500, 0, TEXT, str(tmp_path), data_path=str(p), model_type="clip",
                        clip_state_dict=sd, arch="ViT-B/32", max_batch=8, env_type="none", tokenizer="standin",
                        embeddings=embeddings)
    assert seen, "the gzip rows did not take the compressed path"
    want, got = _read(plain), _read(zipped)
    assert sorted(got) == sorted(want) and want
    for k in want:
        assert got[k].tobytes() == want[k].tobytes() and got[k].dtype == want[k].dtype, k
