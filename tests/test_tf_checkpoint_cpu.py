"""Hermetic test of deepmimic_b200/tf_checkpoint.py: a TensorBundle checkpoint (LevelDB-format .index table + .data shard) is written here
byte by byte in the layout tf.train.Saver produces (prefix-compressed keys, restart array, block trailer, index block, 48-byte footer with
the table magic; BundleEntryProto values) and read back.  The tests against the reference's real checkpoints need a reference checkout
($DEEPMIMIC_REFERENCE_ROOT)."""
import os
import struct

import numpy as np
import pytest

from deepmimic_b200.tf_checkpoint import list_entries, load_actor, load_checkpoint

MAGIC = 0xdb4775248b80fb57


def varint(v):
    out = bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        if v:
            out.append(b | 0x80)
        else:
            out.append(b)
            return bytes(out)


def entry_proto(shape, offset, size, dtype=1):
    dims = b"".join(b"\x12" + varint(len(d)) + d for d in (b"\x08" + varint(s) for s in shape))      # TensorShapeProto.dim (field 2) {size = field 1}
    msg = b"\x08" + varint(dtype) + b"\x12" + varint(len(dims)) + dims                                 # dtype (1), shape (2)
    msg += b"\x18" + varint(0) + b"\x20" + varint(offset) + b"\x28" + varint(size)                     # shard_id (3), offset (4), size (5)
    msg += b"\x35" + struct.pack("<I", 0xDEADBEEF)                                                     # crc32c (6, fixed32): skipped by the reader
    return msg


def block(items, restart_interval=16):
    """LevelDB data block: entries (shared, non_shared, value_len, key delta, value), restart offsets, restart count; then the 5-byte trailer."""
    buf, restarts, prev = bytearray(), [], b""
    for i, (k, v) in enumerate(items):
        shared = 0
        if i % restart_interval == 0:
            restarts.append(len(buf))
        else:
            while shared < min(len(prev), len(k)) and prev[shared] == k[shared]:
                shared += 1
        buf += varint(shared) + varint(len(k) - shared) + varint(len(v)) + k[shared:] + v
        prev = k
    for r in restarts:
        buf += struct.pack("<I", r)
    buf += struct.pack("<I", len(restarts))
    return bytes(buf)


def write_bundle(prefix, tensors, keys_per_block=7):
    data = bytearray()
    items = [(b"", b"\x08\x01")]                                          # BundleHeaderProto under the empty key
    for name in sorted(tensors):
        arr = tensors[name]
        raw = arr.astype("<f4").tobytes() if arr.dtype != np.int32 else arr.astype("<i4").tobytes()
        items.append((name.encode(), entry_proto(list(arr.shape), len(data), len(raw), dtype=3 if arr.dtype == np.int32 else 1)))
        data += raw
    open(prefix + ".data-00000-of-00001", "wb").write(bytes(data))
    out, index_items = bytearray(), []
    for i in range(0, len(items), keys_per_block):
        chunk = items[i:i + keys_per_block]
        b = block(chunk, restart_interval=3)
        handle = varint(len(out)) + varint(len(b))
        out += b + b"\x00" + struct.pack("<I", 0)                          # trailer: no compression + (unchecked) crc
        index_items.append((chunk[-1][0] + b"\x00", handle))               # separator key >= last key of the block
    meta = block([])
    meta_handle = varint(len(out)) + varint(len(meta)); out += meta + b"\x00" + struct.pack("<I", 0)
    idx = block(index_items, restart_interval=1)
    idx_handle = varint(len(out)) + varint(len(idx)); out += idx + b"\x00" + struct.pack("<I", 0)
    footer = meta_handle + idx_handle
    footer += b"\x00" * (40 - len(footer)) + struct.pack("<Q", MAGIC)
    open(prefix + ".index", "wb").write(bytes(out + footer))


def test_reads_back_a_hand_written_tensor_bundle(tmp_path):
    rng = np.random.default_rng(0)
    a = "agent/main/actor/"
    tensors = {a + "0/dense/kernel": rng.standard_normal((7, 5)), a + "0/dense/bias": rng.standard_normal(5), a + "1/dense/kernel": rng.standard_normal((5, 4)),
               a + "1/dense/bias": rng.standard_normal(4), a + "dist_gauss_diag/mean/kernel": rng.standard_normal((4, 3)), a + "dist_gauss_diag/mean/bias": rng.standard_normal(3),
               a + "dist_gauss_diag/logstd/bias": rng.standard_normal(3), "agent/resource/s_norm/mean": rng.standard_normal(7), "agent/resource/s_norm/std": rng.random(7) + 0.5,
               "agent/resource/a_norm/mean": rng.standard_normal(3), "agent/resource/a_norm/std": rng.random(3) + 0.5, "agent/resource/s_norm/count": np.array([123], dtype=np.int32),
               "agent/main/critic/0/dense/kernel": rng.standard_normal((300, 40)), "scalar": np.array(2.5)}
    tensors = {k: (v if v.dtype == np.int32 else v.astype(np.float32)) for k, v in tensors.items()}
    prefix = str(tmp_path / "model.ckpt")
    write_bundle(prefix, tensors)
    ent = list_entries(prefix)
    assert set(ent) == set(tensors) and ent[a + "0/dense/kernel"]["shape"] == [7, 5] and ent["scalar"]["shape"] == []
    assert ent["agent/resource/s_norm/count"]["dtype"] == 3
    got = load_checkpoint(prefix)
    assert "agent/resource/s_norm/count" not in got                       # only float32 tensors are returned
    for k, v in tensors.items():
        if v.dtype == np.float32:
            assert got[k].shape == v.shape and np.array_equal(got[k], v), k
    act = load_actor(prefix)
    assert [w.shape for w, _ in act["hidden"]] == [(7, 5), (5, 4)] and act["mean"][0].shape == (4, 3) and "gate_common" not in act
    assert np.array_equal(act["s_norm_std"], tensors["agent/resource/s_norm/std"]) and "g_norm_mean" not in act


def test_reads_the_gate_layers_of_a_task_policy_bundle(tmp_path):
    """fc_2layers_gated_1024units layout (gate_common, per hidden layer gate<i>/0/dense -> gate<i>/dense bias head, gate<i>/dense_1 scale head)
    written with the tensors of the committed heading-policy fixture: load_actor returns the gate layers with the shapes of the reference's
    humanoid3d_amp_heading_locomotion checkpoint and the fixture's values."""
    f = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "policy_humanoid3d_amp_heading_locomotion_fp16.npz"))
    g = lambda k: f[k].astype(np.float32)
    a, r = "agent/main/actor/", "agent/resource/"
    tensors = {a + "0/dense/kernel": g("w0"), a + "0/dense/bias": g("b0"), a + "1/dense/kernel": g("w1"), a + "1/dense/bias": g("b1"),
               a + "dist_gauss_diag/mean/kernel": g("wm"), a + "dist_gauss_diag/mean/bias": g("bm"), a + "dist_gauss_diag/logstd/bias": g("logstd"),
               a + "gate_common/0/dense/kernel": g("gcw"), a + "gate_common/0/dense/bias": g("gcb")}
    for i in range(2):
        for head, key in (("0/dense", "hidden"), ("dense", "bias"), ("dense_1", "scale")):
            tensors[a + "gate%d/%s/kernel" % (i, head)] = g("g%d_%s_w" % (i, key))
            tensors[a + "gate%d/%s/bias" % (i, head)] = g("g%d_%s_b" % (i, key))
    for nm, key in (("s_norm", "s"), ("g_norm", "g"), ("a_norm", "a")):
        tensors[r + nm + "/mean"], tensors[r + nm + "/std"] = g(key + "_mean"), g(key + "_std")
    prefix = str(tmp_path / "model.ckpt")
    write_bundle(prefix, tensors)
    act = load_actor(prefix)
    assert [w.shape for w, _ in act["hidden"]] == [(229, 1024), (1024, 512)] and act["gate_common"][0].shape == (3, 128)
    assert [gt["scale"][0].shape for gt in act["gates"]] == [(64, 1024), (64, 512)] and act["g_norm_mean"].shape == (3,)
    for i in range(2):
        for key in ("hidden", "bias", "scale"):
            assert np.array_equal(act["gates"][i][key][0], g("g%d_%s_w" % (i, key))) and np.array_equal(act["gates"][i][key][1], g("g%d_%s_b" % (i, key)))
    assert np.array_equal(act["gate_common"][0], g("gcw")) and np.array_equal(act["g_norm_std"], g("g_std"))


def test_rejects_files_that_are_not_tensor_bundles(tmp_path):
    p = str(tmp_path / "bad")
    open(p + ".index", "wb").write(b"\x00" * 64)
    with pytest.raises(ValueError, match="not a TensorBundle"):
        list_entries(p)
