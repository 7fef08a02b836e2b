"""Reader for neural-speed's native `.bin` (NE / ggjt) model files.  The test file is written the way the reference's own
converter writes it (convert/convert_quantized_llama.py:131-260): header and vocab in that order, tensor headers as the
reference's `write_header` (convert/common.py:467) writes them -- the bytes it wrote for this file are stored in
tests/golden/reference.npz -- or through a restatement of it."""
import importlib.util
import os
import struct

import numpy as np
import pytest

import neural_speed_b200 as ns
from neural_speed_b200 import ne_loader
from oracle import golden


class _Tap:
    """the bytes a header writer leaves in the file, the alignment gap it seeks over included"""

    def __init__(self, f):
        self.f, self.data = f, bytearray()

    def write(self, b):
        self.data += b
        return self.f.write(b)

    def tell(self):
        return self.f.tell()

    def seek(self, pos):
        self.data += bytes(pos - self.f.tell())
        return self.f.seek(pos)


def _ref_write_header():
    """the reference's write_header, replaying the bytes it wrote for each tensor header of _write's file"""
    def live():
        spec = importlib.util.spec_from_file_location("ref_common_ne", os.path.join(golden.SOURCE, "neural_speed", "convert", "common.py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        return m.write_header

    def write_header(f, shape, name, ftype):
        def written():
            tap = _Tap(f)
            live()(tap, shape, name, ftype)
            return np.frombuffer(bytes(tap.data), np.uint8)

        key = f"ne_header[{f.tell()}].{name}"
        if golden.recording():
            golden.value(key, written)
        else:
            f.write(golden.value(key, None).tobytes())

    return write_header


def _own_write_header(f, shape, name, ftype):
    s = name.encode()
    f.write(struct.pack("iii", len(shape), len(s), ftype))
    f.write(struct.pack("i" * len(shape), *shape[::-1]))
    f.write(s)
    f.seek((f.tell() + 31) & -32)


def _write(path, write_header):
    rng = np.random.default_rng(9)
    V, E, H, HK, NL, FF = 48, 256, 4, 2, 2, 384
    kvd = E // H * HK
    ref = {}
    with open(path, "wb") as f:
        f.write(b"ggjt"[::-1])
        f.write(struct.pack("i" * 9, 1, V, E, 256, H, HK, NL, E // H, 0))
        f.write(struct.pack("i", 0))                      # max_seq_len
        f.write(struct.pack("f", 0))
        f.write(struct.pack("f", 0))
        f.write(struct.pack("iii", 0, 0, 0))              # par_res, word_embed_proj_dim, do_layer_norm_before
        f.write(struct.pack("i", 0))                      # multi_query_group_num
        f.write(struct.pack("i", FF))
        f.write(struct.pack("iiii", 0, 0, 0, 0))          # inner_hidden_size, n_experts, n_experts_used, n_embd_head_k
        f.write(struct.pack("fff", 1e-5, 10000.0, 1.0))
        f.write(struct.pack("f", 0.0))
        f.write(struct.pack("ii", 0, 0))
        f.write(struct.pack("iiii", 1, 2, 0, 0))          # bos eos pad sep
        for i in range(V):
            t = f"tok{i}".encode()
            f.write(struct.pack("i", len(t)))
            f.write(t)
            f.write(struct.pack("f", -float(i)))

        def fp32(name, arr):
            ref[name] = arr
            write_header(f, list(arr.shape), name, 0)
            arr.tofile(f)

        def btla(name, n, k):
            w = rng.uniform(-0.5, 0.5, (n, k)).astype(np.float32)
            blob = ns.np_bestla_quantize(w, "int4", 128, "sym", "fp32", "int8")
            ref[name] = blob.copy()
            write_header(f, [n, k], name, 19)
            blob.tofile(f)

        fp32("tok_embeddings.weight", rng.normal(0, 1, (V, E)).astype(np.float32))
        fp32("norm.weight", rng.uniform(0.5, 1.5, E).astype(np.float32))
        btla("output.weight", V, E)
        for il in range(NL):
            for nm, (n, k) in dict(wq=(E, E), wk=(kvd, E), wv=(kvd, E), wo=(E, E)).items():
                btla(f"layers.{il}.attention.{nm}.weight", n, k)
            for nm, (n, k) in dict(w1=(FF, E), w2=(E, FF), w3=(FF, E)).items():
                btla(f"layers.{il}.feed_forward.{nm}.weight", n, k)
            fp32(f"layers.{il}.attention_norm.weight", rng.uniform(0.5, 1.5, E).astype(np.float32))
            fp32(f"layers.{il}.ffn_norm.weight", rng.uniform(0.5, 1.5, E).astype(np.float32))
    return ref, dict(n_vocab=V, n_embd=E, n_head=H, n_head_kv=HK, n_layer=NL, n_ff=FF)


@pytest.mark.parametrize("writer", ["reference", "own"])
def test_parse_ne_llama_file_with_btla_blobs(tmp_path, writer):
    wh = _ref_write_header() if writer == "reference" else _own_write_header
    path = str(tmp_path / "tiny.bin")
    ref, hp = _write(path, wh)
    raw_hp, vocab, special, tensors = ne_loader.read_file(path)
    assert raw_hp["n_rot"] == hp["n_embd"] // hp["n_head"] and raw_hp["ffn_hidden_size"] == hp["n_ff"]
    assert special == dict(bos=1, eos=2, pad=0, sep=0)
    assert vocab[5] == (b"tok5", -5.0) and len(vocab) == hp["n_vocab"]
    m = ne_loader.parse(path)
    for k, v in hp.items():
        assert m.hparams[k] == v, k
    assert abs(m.hparams["norm_eps"] - 1e-5) < 1e-9 and m.hparams["rope_theta"] == 10000.0 and m.hparams["n_ctx"] == 2048
    assert np.array_equal(m.tok_embd, ref["tok_embeddings.weight"]) and np.array_equal(m.out_norm, ref["norm.weight"])
    assert m.output[0] == "btla" and np.array_equal(m.output[1], ref["output.weight"])
    for il, L in enumerate(m.layers):
        assert np.array_equal(L["attn_norm"], ref[f"layers.{il}.attention_norm.weight"])
        for nm in ("wq", "wk", "wv", "wo"):
            assert np.array_equal(L[nm][1], ref[f"layers.{il}.attention.{nm}.weight"])
        for nm in ("w1", "w2", "w3"):
            assert np.array_equal(L[nm][1], ref[f"layers.{il}.feed_forward.{nm}.weight"])
    # the blobs survive the round trip through the file at a different alignment: same dequantised weights
    E, kvd = hp["n_embd"], hp["n_embd"] // hp["n_head"] * hp["n_head_kv"]
    wk = m.layers[1]["wk"][1]
    assert np.array_equal(ns.unpack_blob(wk, kvd, E), ns.unpack_blob(ref["layers.1.attention.wk.weight"], kvd, E))


def test_bad_files_are_refused(tmp_path):
    p = tmp_path / "bad.bin"
    p.write_bytes(b"GGUF" + bytes(64))
    with pytest.raises(ValueError, match="not an NE"):
        ne_loader.read_file(str(p))
