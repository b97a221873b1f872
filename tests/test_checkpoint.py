"""TF tensor-bundle checkpoints (reference main.py:153-165,226-228) without TensorFlow, and forward parity on the
reference's own TRAINED weights: the ml-1m SASRec checkpoint shipped under saved_models/ (global_step 9400; fixture
tests/golden/ml1m_sasrec_ckpt.npz, produced by tests/golden/make_golden.py with the reader tested here).  Trained
LayerNorm betas are non-zero, so padded query rows are live and fully-masked rows are uniform over all T keys
(SURVEY A-6/A-8) — the cases a textbook attention kernel gets wrong."""
import os
import struct

import numpy as np
import pytest
import torch

from helpers import O, make_args, oracle_batch, rel_err
import cast_b200
from cast_b200 import checkpoint as ck

HERE = os.path.dirname(os.path.abspath(__file__))
FIX = os.path.join(HERE, "golden", "ml1m_sasrec_ckpt.npz")


def fixture_params():
    g = np.load(FIX)
    return {k: g[k] for k in g.files if k != "global_step"}


def test_fixture_shapes_match_the_reference_run():
    p = fixture_params()
    assert p["item_emb"].shape == (3417, 50) and p["pos_emb"].shape == (200, 50)   # ml-1m: itemnum 3416, maxlen 200
    assert len(p) == 32 and int(np.load(FIX)["global_step"]) == 9400
    assert np.abs(p["main.0.ln1.beta"]).mean() > 0.05                               # trained, not the init


def test_writer_reader_round_trip(tmp_path):
    p = fixture_params()
    tfv = ck.to_tf_names("sasrec", p, 2)
    assert tfv["SASRec/num_blocks_0/multihead_attention/conv1d/kernel"].shape == (1, 50, 50)
    ck.write_bundle(str(tmp_path / "model.ckpt"), tfv, checksum_data=False)
    back = ck.to_role_names("sasrec", ck.read_bundle(str(tmp_path / "model.ckpt")), 2)
    assert sorted(back) == sorted(p)
    for k in p:
        assert np.array_equal(back[k], p[k]), k


def test_block_entries_decodes_prefix_shared_keys():
    """Known answer, bytes written by hand in the LevelDB block format TensorFlow's table writer uses: each entry is
    varint(shared) varint(unshared) varint(value length) key-suffix value, a restart point every 2 entries here."""
    body = (b"\x00\x05\x01apple" + b"1"       # offset 0, restart
            + b"\x05\x01\x01t" + b"2"          # "apple" + "t"
            + b"\x00\x05\x01apply" + b"3"      # offset 14, restart
            + b"\x05\x05\x01/Adam" + b"4")     # "apply" + "/Adam"
    block = body + struct.pack("<III", 0, 14, 2)
    assert list(ck._block_entries(block)) == [(b"apple", b"1"), (b"applet", b"2"), (b"apply", b"3"),
                                              (b"apply/Adam", b"4")]


def _tf_block(pairs, restart_interval):
    """One table block as TensorFlow's (LevelDB's) BlockBuilder lays it out: a key shares its prefix with the previous
    key except at a restart point, every `restart_interval` entries."""
    body, restarts, prev = bytearray(), [], b""
    for i, (k, v) in enumerate(pairs):
        shared = 0
        if i % restart_interval == 0:
            restarts.append(len(body))
        else:
            while shared < min(len(k), len(prev)) and k[shared] == prev[shared]:
                shared += 1
        body += ck._put_varint(shared) + ck._put_varint(len(k) - shared) + ck._put_varint(len(v)) + k[shared:] + v
        prev = k
    for r in restarts or [0]:
        body += struct.pack("<I", r)
    return bytes(body + struct.pack("<I", max(1, len(restarts))))


def _separator(start, limit):
    """LevelDB's BytewiseComparator::FindShortestSeparator: the index key between two data blocks"""
    n = 0
    while n < min(len(start), len(limit)) and start[n] == limit[n]:
        n += 1
    if n < min(len(start), len(limit)) and start[n] < 0xFF and start[n] + 1 < limit[n]:
        return start[:n] + bytes([start[n] + 1])
    return start


def _successor(key):
    """... FindShortSuccessor: the index key after the last data block"""
    for i, b in enumerate(key):
        if b != 0xFF:
            return key[:i] + bytes([b + 1])
    return key


def _tf_table(pairs, block_size):
    """SSTable with TensorFlow's defaults: data blocks cut at `block_size` bytes with a restart point every 16 keys,
    an empty meta-index block, an index block of shortened separator keys (restart interval 1), the 48-byte footer.
    Returns (file bytes, number of data blocks)."""
    out, index, cur, last = bytearray(), [], [], None

    def emit(block):
        handle = ck._put_varint(len(out)) + ck._put_varint(len(block))
        out.extend(ck._with_trailer(block))
        return handle

    for k, v in pairs:
        if last is not None:
            index.append((_separator(last[0], k), last[1]))
            last = None
        cur.append((k, v))
        if len(_tf_block(cur, 16)) >= block_size:
            last, cur = (k, emit(_tf_block(cur, 16))), []
    if cur:
        last = (cur[-1][0], emit(_tf_block(cur, 16)))
    index.append((_successor(last[0]), last[1]))
    meta = emit(_tf_block([], 16))
    idx = emit(_tf_block(index, 1))
    footer = meta + idx
    return bytes(out + footer + b"\x00" * (40 - len(footer)) + struct.pack("<Q", ck._MAGIC)), len(index)


def _tf_entry(dtype, shape, offset, size, crc):
    """BundleEntryProto: dtype, shape, offset (omitted when 0), size, crc32c"""
    dims = b"".join(b"\x12" + ck._put_varint(len(d)) + d for d in (b"\x08" + ck._put_varint(s) for s in shape))
    e = b"\x08" + ck._put_varint(dtype) + b"\x12" + ck._put_varint(len(dims)) + dims
    if offset:
        e += b"\x20" + ck._put_varint(offset)
    return e + b"\x28" + ck._put_varint(size) + b"\x35" + struct.pack("<I", crc)


@pytest.mark.parametrize("block_size", [262144, 1024], ids=["tf_default_blocks", "small_blocks"])
def test_reader_parses_a_tensorflow_layout_index(tmp_path, block_size):
    """The reference's ml-1m SASRec checkpoint as tf.train.Saver wrote it: its 99 entries (32 weights, their Adam and
    Adam_1 slots, beta1_power, beta2_power, global_step) with the masked crc32c TensorFlow stored for each
    (tests/golden/ref_bundle_crc.npz), in an index laid out the way TensorFlow's table writer lays it out (prefix-shared
    keys, restart points every 16 keys, shortened index keys; several data blocks when they are small).  The weights
    are the fixture's, the other tensors seeded, stored in the data file in shuffled order at recorded offsets."""
    g = np.load(os.path.join(HERE, "golden", "ref_bundle_crc.npz"))
    crcs = dict(zip([str(x) for x in g["names"]], [int(x) for x in g["crcs"]]))
    weights = ck.to_tf_names("sasrec", fixture_params(), 2)
    rng = np.random.RandomState(0)
    tensors = {}
    for name in crcs:
        if name in weights:
            tensors[name] = weights[name]
        elif name.endswith(("/Adam", "/Adam_1")):
            tensors[name] = rng.rand(*weights[name.rsplit("/", 1)[0]].shape).astype(np.float32)
        elif name == "global_step":
            tensors[name] = np.asarray(np.load(FIX)["global_step"], np.int32)
        else:
            tensors[name] = np.asarray(rng.rand(), np.float32)
    assert len(tensors) == 99
    data, offsets = bytearray(), {}
    for name in rng.permutation(sorted(tensors)):
        offsets[name] = len(data)
        data += tensors[name].tobytes()
    pairs = [(b"", b"\x08\x01\x1a\x02\x08\x01")]            # BundleHeaderProto: num_shards 1, version {producer 1}
    for name in sorted(tensors):
        a = tensors[name]
        pairs.append((name.encode(), _tf_entry({np.float32: 1, np.int32: 3}[a.dtype.type], a.shape, offsets[name],
                                               a.nbytes, crcs[name])))
    index, n_blocks = _tf_table(pairs, block_size)
    assert (n_blocks == 1) == (block_size == 262144)
    prefix = str(tmp_path / "model.ckpt")
    with open(prefix + ".index", "wb") as f:
        f.write(index)
    with open(prefix + ".data-00000-of-00001", "wb") as f:
        f.write(bytes(data))

    assert ck.read_bundle_crcs(prefix) == crcs
    tfv = ck.read_bundle(prefix)
    assert sorted(tfv) == sorted(tensors)
    assert int(tfv["global_step"]) == 9400 and tfv["global_step"].dtype == np.int32
    assert tfv["SASRec/input_embeddings/lookup_table/Adam_1"].shape == (3417, 50)   # optimizer slots are there too
    for name, a in tensors.items():
        assert tfv[name].dtype == a.dtype and np.array_equal(tfv[name], a), name
    fx = fixture_params()
    p = ck.to_role_names("sasrec", tfv, 2)
    assert sorted(p) == sorted(fx)
    for k in fx:
        assert np.array_equal(p[k], fx[k]), k


def _synthetic_sequences(B, T, itemnum, seed=0):
    rng = np.random.RandomState(seed)
    seq = rng.randint(1, itemnum + 1, (B, T)).astype(np.int32)
    lens = [T, 1, 2, 37, 150, T - 1, 64, 9][:B]
    for b, n in enumerate(lens):
        seq[b, :T - n] = 0
    return seq


def test_oracle_on_trained_weights_shows_the_reference_quirks():
    """Oracle sanity on real weights: a padded query row attends uniformly (1/T) over all keys."""
    p = {k: torch.from_numpy(v) for k, v in fixture_params().items()}
    args = make_args(hidden_units=50, maxlen=200, num_heads=1, num_blocks=2, dropout_rate=0.0)
    seq = _synthetic_sequences(4, 200, 3416)
    b = {"seq": seq, "pos": seq, "neg": seq, "timeseq": seq * 0, "hours": seq * 0, "days": seq * 0}
    _, _, attn = O.forward("sasrec", p, args, oracle_batch(b))
    a = attn.detach().numpy()
    assert a.shape == (4, 200, 200)
    assert np.allclose(a[1, 0], 1.0 / 200, atol=1e-7)        # sequence 1 has a single item: row 0 is padding


@pytest.mark.gpu
def test_forward_and_predict_parity_on_trained_reference_weights():
    p = fixture_params()
    args = make_args(hidden_units=50, maxlen=200, num_heads=1, num_blocks=2, dropout_rate=0.2)
    m = cast_b200.SASRec(6040, 3416, args)
    m.load_state_dict(p)
    seq = _synthetic_sequences(8, 200, 3416)
    item_idx = np.concatenate([[seq[0, -1]], np.random.RandomState(1).randint(1, 3417, 100)]).astype(np.int32)
    logits, attn = m.predict(None, np.arange(8), seq, item_idx)
    pt = {k: torch.from_numpy(v) for k, v in p.items()}
    b = {"seq": seq, "pos": seq, "neg": seq, "timeseq": seq * 0, "hours": seq * 0, "days": seq * 0}
    so, table, attn_o = O.forward("sasrec", pt, args, oracle_batch(b))
    lo = O.test_logits(so, table, item_idx).detach().numpy()
    assert rel_err(logits, lo) <= 1e-4
    assert np.abs(attn - attn_o.detach().numpy()).max() <= 1e-5
    seq_emb = m.engine.ctx(8).seq_emb.cpu().numpy().reshape(8, 200, 50)
    live = seq != 0
    assert rel_err(seq_emb[live], so.detach().numpy()[live]) <= 1e-4
    # ranks through the fused scorer == the reference expression on the oracle's logits
    cand = np.tile(item_idx, (8, 1))
    _, cgt, ceq = m.score_candidates(seq, cand)
    for u in range(8):
        if ceq[u] == 0:
            assert cgt[u] == O.rank_of_target(lo[u])


# ---------------------------------------------------------------------------------------------------------------------
# the reference's six CAST checkpoints (saved_models/ml-1m.txt/cast_{1..6}_*), mapped by role, and the full Saver state
def cast_fixture(n):
    g = np.load(os.path.join(HERE, "golden", f"ml1m_cast{n}_ckpt.npz"))
    return {k: g[k] for k in g.files if k != "global_step"}


def _context_batch(B, T, itemnum, seed=3):
    rng = np.random.RandomState(seed)
    seq = _synthetic_sequences(B, T, itemnum, seed)
    live = seq != 0
    ts = np.where(live, np.minimum(200, rng.geometric(0.05, (B, T)) - 1), 0).astype(np.int32)
    ts[:, -1] = 0
    hrs = np.where(live, rng.randint(1, 25, (B, T)), 0).astype(np.int32)
    dys = np.where(live, rng.randint(1, 8, (B, T)), 0).astype(np.int32)
    return seq, ts, hrs, dys


def test_writer_checksums_equal_tensorflows_byte_for_byte(tmp_path):
    """The masked crc32c our writer stores for each tensor == the one TensorFlow stored in the reference's own
    model.ckpt.index for the same bytes (known answers: tests/golden/ref_bundle_crc.npz); TF's BundleReader refuses
    entries whose checksum does not match."""
    g = np.load(os.path.join(HERE, "golden", "ref_bundle_crc.npz"))
    want = dict(zip([str(x) for x in g["names"]], [int(x) for x in g["crcs"]]))
    tfv = ck.to_tf_names("sasrec", fixture_params(), 2)
    prefix = str(tmp_path / "model.ckpt")
    ck.write_bundle(prefix, tfv)
    got = ck.read_bundle_crcs(prefix)
    assert len(got) == 32
    for k, v in got.items():
        assert v == want[k], k
    assert ck._mask_crc(ck._crc32c_py(b"123456789")) == ck._mask_crc(0xE3069283)      # crc32c check value
    assert ck._crc32c(b"123456789") == 0xE3069283


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6])
def test_cast_checkpoints_map_by_role(n, tmp_path):
    p = cast_fixture(n)
    model = f"cast_{n}"
    assert p["time_emb"].shape == (201, 50) and p["time.1.ln2.gamma"].shape == (50,)
    if n >= 2:
        k = {2: 2, 3: 3, 4: 4, 5: 3, 6: 4}[n]
        assert p["mlp.0.w"].shape == (k * 50, k * 50) and p["mlp.1.w"].shape == (k * 50, 50)
    assert np.abs(p["time.0.ln1.beta"]).mean() > 0.01          # trained
    tfv = ck.to_tf_names(model, p, 2)
    dead = "CONTEXT/timeseq_num_blocks_0/ln/Variable_1"
    assert np.all(tfv[dead] == 1.0) and np.all(tfv[dead[:-2]] == 0.0)   # the unused LayerNorm pair keeps its init
    ck.write_bundle(str(tmp_path / "m.ckpt"), tfv)
    back = ck.to_role_names(model, ck.read_bundle(str(tmp_path / "m.ckpt")), 2)
    assert sorted(back) == sorted(p) and all(np.array_equal(back[k], p[k]) for k in p)
    # the oracle accepts exactly this parameter set
    args = make_args(hidden_units=50, maxlen=200, num_heads=1, num_blocks=2)
    assert sorted(O.init_params(model, args, 3416, seed=0)) == sorted(p)


@pytest.mark.emu
def test_full_training_state_round_trip(tmp_path):
    """save_model / restore_model carry weights, Adam slots, beta powers and global_step under the reference's names:
    a run restored from the bundle continues bit-identically to the run that never stopped."""
    from helpers import backend, golden_batch
    lib, dev = backend("emu")
    args = make_args(hidden_units=12, maxlen=10, num_heads=2, num_blocks=2, dropout_rate=0.2)
    gb = golden_batch(B=4, T=10)

    def step(m):
        return m.train_step(gb["u"], gb["seq"], gb["pos"], gb["neg"], gb["timeseq"], gb["hours"], gb["days"])

    a = cast_b200.build_model("cast_4", 80, 300, 5, args, device=dev, _lib=lib, use_graph=False, seed=4)
    step(a)
    step(a)
    prefix = str(tmp_path / "model.ckpt")
    ck.save_model(prefix, a, "cast_4", 2)
    tfv = ck.read_bundle(prefix)
    assert int(tfv["global_step"]) == 2 and tfv["global_step"].dtype == np.int32
    assert abs(float(tfv["beta1_power"]) - 0.9 ** 3) < 1e-6 and abs(float(tfv["beta2_power"]) - 0.98 ** 3) < 1e-6
    assert tfv["SASRec/MLP/dense/kernel/Adam_1"].shape == (48, 48)
    assert "CONTEXT/timeseq_num_blocks_0/ln/Variable/Adam" not in tfv          # dead variables have no slots in TF either
    b = cast_b200.build_model("cast_4", 80, 300, 5, args, device=dev, _lib=lib, use_graph=False, seed=4)
    b.engine.w.add_(0.5)     # (same dropout seed — it is an argument, not a variable — but different parameters)
    ck.restore_model(prefix, b, "cast_4", 2)
    assert b.engine.state_step() == 2
    la, lb = step(a), step(b)
    assert la == lb
    assert torch.equal(a.engine.w, b.engine.w) and torch.equal(a.engine.m, b.engine.m)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6])
def test_cast_forward_parity_on_trained_reference_weights(n):
    """CUDA path vs oracle on the reference's own trained CAST weights: 101-candidate logits (1e-4), the exposed
    attention map of the time tower (1e-5) and the live rows of the sequence embedding."""
    model = f"cast_{n}"
    p = cast_fixture(n)
    args = make_args(hidden_units=50, maxlen=200, num_heads=1, num_blocks=2, dropout_rate=0.2)
    m = cast_b200.build_model(model, 6040, 3416, 5, args)
    m.load_state_dict(p)
    seq, ts, hrs, dys = _context_batch(8, 200, 3416)
    item_idx = np.concatenate([[seq[0, -1]], np.random.RandomState(1).randint(1, 3417, 100)]).astype(np.int32)
    logits, attn = m.predict(None, np.arange(8), seq, item_idx, timeseq=ts, hours_seq=hrs, days_seq=dys)
    pt = {k: torch.from_numpy(v) for k, v in p.items()}
    b = {"seq": seq, "pos": seq, "neg": seq, "timeseq": ts, "hours": hrs, "days": dys}
    so, table, attn_o = O.forward(model, pt, args, oracle_batch(b))
    lo = O.test_logits(so, table, item_idx).detach().numpy()
    assert rel_err(logits, lo) <= 1e-4
    assert np.abs(attn - attn_o.detach().numpy()).max() <= 1e-5
    seq_emb = m.engine.ctx(8).seq_emb.cpu().numpy().reshape(8, 200, 50)
    live = seq != 0
    assert rel_err(seq_emb[live], so.detach().numpy()[live]) <= 1e-4
