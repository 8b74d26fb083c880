"""Variable inventory / checkpoint reader / seeded init (host logic, CPU)."""
import json
import os
import struct

import numpy as np
import pytest

from nhans_b200 import weights as W

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("tag,variant", [("sn", 0), ("ss", 1)])
def test_inventory_matches_reference_checkpoint_index(tag, variant):
    """Names, shapes and byte sizes of model()'s variables equal the reference's own checkpoint index
    (tests/golden/ckpt_index_*.json, extracted from trained_model/*.index)."""
    idx = json.load(open(os.path.join(GOLD, "ckpt_index_%s.json" % tag)))
    f32 = {k: v for k, v in idx.items() if v[0] == 1}
    inv = W.inventory(variant)
    assert set(inv) == set(f32)
    assert len(inv) == 571
    for k, shp in inv.items():
        assert list(shp) == f32[k][1], k
        assert int(np.prod(shp)) * 4 == f32[k][3], k
    assert W.n_params(variant) == 28999881
    assert sum(v[3] for v in f32.values()) == 115999524          # the git-LFS pointer's size
    offs = sorted((v[2], v[3]) for v in idx.values())
    assert all(offs[i][0] + offs[i][1] == offs[i + 1][0] for i in range(len(offs) - 1))   # contiguous


def test_index_reader_on_reference_files(tmp_path):
    """The reference's selective-noise checkpoint as its repository ships it: the .index (every entry of
    tests/golden/ckpt_index_sn.json, laid out like TF's table builder writes it: prefix-compressed keys, a restart
    point every 16 entries, ~4 KiB data blocks) next to a git-LFS pointer in place of the data shard."""
    idx = json.load(open(os.path.join(GOLD, "ckpt_index_sn.json")))
    d = str(tmp_path / "trained_model")
    os.makedirs(d)
    prefix = os.path.join(d, "81448_0-1000000")
    entries = [(k.encode(), _entry_proto(*v)) for k, v in sorted(idx.items())]
    _write_table(prefix + ".index", [(b"", _BUNDLE_HEADER)] + entries, block_size=4096, restart_interval=16)
    with open(prefix + ".data-00000-of-00001", "wb") as f:
        f.write(b"version https://git-lfs.github.com/spec/v1\noid sha256:0\nsize 115999524\n")
    e = W.read_bundle_index(prefix + ".index")
    assert {k: [v["dtype"], list(v["shape"]), v["offset"], v["size"]] for k, v in e.items()} == idx
    with pytest.raises(FileNotFoundError):                           # the data shard is an LFS pointer
        W.load_bundle(prefix)
    # like the reference (SN/apply.py:428-432), a checkpoint that cannot be restored is an error ...
    with pytest.raises(W.CheckpointMissing):
        W.load_or_init(0, d, allow_random=False)
    # ... unless random-init weights of the identical architecture are explicitly allowed
    w, src = W.load_or_init(0, d, allow_random=True)
    assert src == "random-init" and len(w) == 571


def _varint(n):
    out = b""
    while True:
        b = n & 0x7F
        n >>= 7
        out += bytes([b | (0x80 if n else 0)])
        if not n:
            return out


_BUNDLE_HEADER = b"\x08\x01"                  # BundleHeaderProto: num_shards = 1


def _block(entries, restart_interval=1):
    """LevelDB block: keys share their prefix with the previous key except at restart points."""
    body, restarts, prev = b"", [], b""
    for i, (k, v) in enumerate(entries):
        shared = 0
        if i % restart_interval == 0:
            restarts.append(len(body))
        else:
            while shared < min(len(k), len(prev)) and k[shared] == prev[shared]:
                shared += 1
        body += _varint(shared) + _varint(len(k) - shared) + _varint(len(v)) + k[shared:] + v
        prev = k
    restarts = restarts or [0]
    return body + b"".join(struct.pack("<I", r) for r in restarts) + struct.pack("<I", len(restarts))


def _write_table(path, entries, block_size=1 << 62, restart_interval=1):
    """LevelDB table of sorted (key, value) pairs: uncompressed data blocks of about `block_size` bytes, an empty
    meta-index block, the index block and the footer."""
    f, index, pending = b"", [], []

    def put(blk):
        nonlocal f
        handle = _varint(len(f)) + _varint(len(blk))
        f += blk + b"\x00" + b"\x00" * 4                 # trailer: type (uncompressed) + crc32c (not checked)
        return handle
    for i, (k, v) in enumerate(entries):
        pending.append((k, v))
        if i == len(entries) - 1 or sum(len(a) + len(b) for a, b in pending) >= block_size:
            index.append((k, put(_block(pending, restart_interval))))
            pending = []
    meta = put(_block([]))
    idx = put(_block(index))
    footer = meta + idx
    footer += b"\x00" * (40 - len(footer)) + struct.pack("<Q", 0xDB4775248B80FB57)
    with open(path, "wb") as out:
        out.write(f + footer)


def _entry_proto(dtype, shape, offset, size):
    """BundleEntryProto: dtype, shape, offset, size and a crc32c field (a stand-in value: the reader ignores it)."""
    dims = b"".join(b"\x12" + _varint(len(d)) + d for d in (b"\x08" + _varint(s) for s in shape))
    return (b"\x08" + _varint(dtype) + b"\x12" + _varint(len(dims)) + dims + b"\x20" + _varint(offset) + b"\x28" + _varint(size)
            + b"\x35" + struct.pack("<I", 0x5EED))


def _write_bundle(prefix, tensors):
    """Minimal TF tensor-bundle writer (one data block) to round-trip the reader."""
    chunks, off, entries = [], 0, [(b"", _BUNDLE_HEADER)]
    for name in sorted(tensors):
        a = np.ascontiguousarray(tensors[name], "<f4")
        entries.append((name.encode(), _entry_proto(1, a.shape, off, a.nbytes)))
        chunks.append(a.tobytes())
        off += a.nbytes
    _write_table(prefix + ".index", entries)
    with open(prefix + ".data-00000-of-00001", "wb") as f:
        f.write(b"".join(chunks))


def test_bundle_roundtrip(tmp_path):
    w = W.seeded_init(0, 3)
    small = {k: w[k] for k in list(sorted(w))[:40]}
    _write_bundle(str(tmp_path / "ckpt-1"), small)
    back = W.load_bundle(str(tmp_path / "ckpt-1"))
    assert set(back) == set(small)
    for k in small:
        assert back[k].shape == small[k].shape and np.array_equal(back[k], small[k])
    assert W.find_checkpoint(str(tmp_path)) == str(tmp_path / "ckpt-1")


def test_seeded_init_is_deterministic_and_non_degenerate():
    a, b = W.seeded_init(0, 0), W.seeded_init(0, 0)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    c = W.seeded_init(0, 1)
    assert not np.array_equal(a["last_dense/w"], c["last_dense/w"])
    # the reference initialises these with stddev 0 (main.py:136,142,146,238) -> identity network
    for k in ("last_dense/w", "resblock1_1_conv1_noise_pos_emb/w", "resblock1_1_conv1_temb_dense3/w"):
        assert float(np.abs(a[k]).max()) > 0
    assert set(W.seeded_init(1, 0)) == set(W.inventory(1))
