"""CPU tier for the actor row (N1): fixtures, the numpy oracle, the checkpoint reader."""
import os

import numpy as np
import pytest

import parity  # noqa: F401  (sys.path)
from oracle import actor_oracle
from pve_mcc_for_unsignalized_intersection_b200.actor import ACTOR_FLOATS, PARAM_SPECS, ActorWeights
from pve_mcc_for_unsignalized_intersection_b200.checkpoint import read_bundle, read_bundle_index

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_weight_fixture_layout():
    w = ActorWeights.from_npz(os.path.join(GOLD, "actor_agent1.npz"))
    assert ACTOR_FLOATS == 6393 and w.flat().shape == (6393,)
    flat = w.flat()
    # order of the flat vector = order of include/pve_mcc.h
    assert np.array_equal(flat[:28], w.tensors["LayerNorm/gamma"])
    assert np.array_equal(flat[56:56 + 28 * 64].reshape(28, 64), w.tensors["dense/kernel"])
    assert flat[-1] == w.tensors["dense_2/bias"][0]
    with pytest.raises(ValueError):
        ActorWeights({n: np.zeros((3,)) for n, _ in PARAM_SPECS})


def test_recorded_rollout_is_config1_of_the_reference():
    """BASELINE.md section 2: pretrained actor on arvTimeNewVeh_new_1000_12.mat, 1000 ticks."""
    z = np.load(os.path.join(GOLD, "actor_rollout_mat1000.npz"))
    assert z["outcome"].tolist() == [323, 0, 281, 548]
    assert abs(float(z["ptm"]) - 12.294) < 5e-4
    assert z["trace"].shape == (1000, 6) and z["trace"][-1, 1] == 323


def test_oracle_reproduces_recorded_actions():
    z = np.load(os.path.join(GOLD, "actor_rollout_mat1000.npz"))
    w = ActorWeights.from_npz(os.path.join(GOLD, "actor_agent1.npz"))
    a32 = actor_oracle.actor_forward(w, z["rows"], np.float32)
    a64 = actor_oracle.actor_forward(w, z["rows"], np.float64)
    np.testing.assert_allclose(a64, z["actions_f64"], rtol=0, atol=1e-12)
    # batched vs single-row BLAS summation order in fp32
    np.testing.assert_allclose(a32, z["actions_f32"], rtol=1e-5, atol=1e-5)
    # fp32 against float64: the network is ill-conditioned at the 1e-4 level (inputs ~160 m rounded to fp32
    # alone move some actions by 9e-5), see tests/test_gpu_actor.py for the bound the kernel is held to
    err = np.abs(a32 - a64)
    assert (err <= 1e-5 * np.abs(a64) + 1e-5).mean() >= 0.97 and err.max() <= 5e-4
    assert np.all(np.abs(a64) <= 3.0)


def test_policy_actions_zero_for_uncontrolled():
    w = ActorWeights.random(3)
    rows = np.random.RandomState(0).randn(10, 28)
    ctrl = np.array([1, 0, 1, 1, 0, 0, 1, 0, 0, 1], dtype=bool)
    a = actor_oracle.policy_actions(w, rows, ctrl)
    assert np.all(a[~ctrl] == 0) and np.all(a[ctrl] != 0)


def _varint(n):
    out = bytearray()
    while True:
        out.append((n & 0x7F) | (0x80 if n > 0x7F else 0))
        n >>= 7
        if not n:
            return bytes(out)


def _table_block(entries, restart_interval=4):
    """A LevelDB table block of (key, value) pairs: prefix-compressed keys, restart array, then the 5-byte trailer
    (type 0 = uncompressed, CRC left 0: the reader does not verify it)."""
    body, restarts, prev = bytearray(), [], b""
    for k, (key, val) in enumerate(entries):
        shared = 0
        if k % restart_interval:
            while shared < min(len(key), len(prev)) and key[shared] == prev[shared]:
                shared += 1
        else:
            restarts.append(len(body))
        body += _varint(shared) + _varint(len(key) - shared) + _varint(len(val)) + key[shared:] + val
        prev = key
    for r in restarts or [0]:
        body += r.to_bytes(4, "little")
    body += len(restarts or [0]).to_bytes(4, "little")
    return bytes(body) + b"\0" * 5


def _bundle_entry(dtype, shape, offset, size):
    """BundleEntryProto; proto3 leaves zero-valued fields out, the reader must default them."""
    dims = b"".join(b"\x12" + _varint(len(d)) + d for d in (b"\x08" + _varint(n) for n in shape))
    out = b"\x08" + _varint(dtype) + b"\x12" + _varint(len(dims)) + dims
    out += (b"\x20" + _varint(offset) if offset else b"") + b"\x28" + _varint(size)
    return out + b"\x35" + b"\x5a\x5a\x5a\x5a"          # field 6, crc32c (fixed32)


def write_bundle(prefix, tensors, per_block=5):
    """``tf.train.Saver`` layout of ``tensors`` (name -> array): ``prefix.index`` (sorted table, several data
    blocks, index block, empty metaindex, 48-byte footer) + ``prefix.data-00000-of-00001``."""
    data, entries = bytearray(), [(b"", b"\x08\x01")]        # header entry: BundleHeaderProto, num_shards 1
    for name in sorted(tensors):
        arr = np.asarray(tensors[name])
        dtype = {np.dtype("<f4"): 1, np.dtype("<i8"): 9}[arr.dtype]
        entries.append((name.encode(), _bundle_entry(dtype, arr.shape, len(data), arr.nbytes)))
        data += arr.tobytes()
    index_file, handles = bytearray(), []
    for k in range(0, len(entries), per_block):
        chunk = entries[k:k + per_block]
        block = _table_block(chunk)
        handles.append((chunk[-1][0], _varint(len(index_file)) + _varint(len(block) - 5)))
        index_file += block
    footer = bytearray()
    for block in (_table_block([]), _table_block(handles, restart_interval=1)):       # metaindex, index
        footer += _varint(len(index_file)) + _varint(len(block) - 5)
        index_file += block
    index_file += bytes(footer) + b"\0" * (40 - len(footer)) + (0xDB4775248B80FB57).to_bytes(8, "little")
    with open(prefix + ".index", "wb") as f:
        f.write(index_file)
    with open(prefix + ".data-00000-of-00001", "wb") as f:
        f.write(data)


def test_checkpoint_reader_on_a_written_bundle(tmp_path):
    """The reader on a bundle in the reference's checkpoint format (model_data/baseline/66.cptk), written here from
    the stored agent-1 tensors: two actor scopes, a critic tensor and the int64 global step the reader must skip."""
    f = ActorWeights.from_npz(os.path.join(GOLD, "actor_agent1.npz"))
    tensors = {"global_step": np.array(66, "<i8"), "agent1_critic/dense/kernel": np.full((30, 64), 0.5, np.float32)}
    for n, _ in PARAM_SPECS:
        tensors["agent1actor/" + n] = f.tensors[n]
        tensors["agent1_target_actor/" + n] = f.tensors[n] * np.float32(2)
    write_bundle(str(tmp_path / "66.cptk"), tensors)
    (tmp_path / "checkpoint").write_text('model_checkpoint_path: "66.cptk"\nall_model_checkpoint_paths: "66.cptk"\n')

    index = read_bundle_index(str(tmp_path / "66.cptk.index"))
    assert sorted(index) == sorted(tensors)
    assert sum(int(np.prod(e["shape"])) for e in index.values()) == 2 * ACTOR_FLOATS + 30 * 64 + 1
    assert index["agent1_critic/dense/kernel"] == {"dtype": 1, "shape": (30, 64), "shard": 0, "offset": 0, "size": 7680}
    assert index["global_step"] == {"dtype": 9, "shape": (), "shard": 0, "offset": 4 * (2 * ACTOR_FLOATS + 30 * 64),
                                    "size": 8}
    assert index["agent1actor/dense/kernel"]["dtype"] == 1 and index["agent1actor/dense/kernel"]["shape"] == (28, 64)
    assert index["agent1actor/dense/kernel"]["size"] == 7168 and index["agent1actor/dense/kernel"]["shard"] == 0
    w = ActorWeights.from_checkpoint(str(tmp_path))
    t = ActorWeights.from_checkpoint(str(tmp_path / "66.cptk"), scope="agent1_target_actor")
    for n, _ in PARAM_SPECS:
        assert np.array_equal(w.tensors[n], f.tensors[n]), n
        assert np.array_equal(t.tensors[n], f.tensors[n] * np.float32(2)), n
    assert "global_step" not in read_bundle(str(tmp_path / "66.cptk"))
    with pytest.raises(KeyError):
        ActorWeights.from_checkpoint(str(tmp_path), scope="agent2actor")


def test_actor_needs_a_gpu_and_says_so():
    import torch
    from pve_mcc_for_unsignalized_intersection_b200 import _native
    from pve_mcc_for_unsignalized_intersection_b200.actor import BatchedActor
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible")
    with pytest.raises(_native.NativeError):
        BatchedActor(ActorWeights.random(0))
    with pytest.raises(_native.NativeError):
        BatchedActor(ActorWeights.random(0), device="cpu")


def test_report_line_and_mat_ingest(tmp_path):
    """Row N4: the batch_test result line (main.py:576-581) and scipy .mat ingest (main.py:388-389)."""
    import scipy.io as scio
    from pve_mcc_for_unsignalized_intersection_b200 import evaluate
    z = np.load(os.path.join(GOLD, "actor_rollout_mat1000.npz"))
    v, c, p, l = z["outcome"].tolist()
    line = evaluate.format_report(v, c, p, int(z["trace"][-1, 5]), float(z["jerk_total"]), l)
    assert line == ("vehicle number 323  collisions occurred number 0 collisions rate 0.0 pT-m 12.2943 s "
                    "jerks 208.79941400944244 lock_num 548")
    path = str(tmp_path / "arvTimeNewVeh_new_1000_12.mat")
    scio.savemat(path, {"arvTimeNewVeh": z["arrive_time"]})
    arr = evaluate.load_arrivals(path)
    assert arr.dtype == np.float64 and np.array_equal(arr, z["arrive_time"])
    stacked = evaluate.stack_tables([arr, arr[:10]])
    assert stacked.shape == (2,) + arr.shape and np.all(stacked[1, 10:] == 0) and np.array_equal(stacked[0], arr)
    scio.savemat(path, {"arvTimeNewVeh": np.zeros((5, 4))})
    with pytest.raises(ValueError):
        evaluate.load_arrivals(path)
