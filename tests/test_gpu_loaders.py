"""SURVEY 8(f).3 on the GPU: model FILES (llama.cpp GGUF with Q4_0 / Q6_K tensors; neural-speed's native NE .bin with BesTLA int4
blobs, tensor headers as the reference converter's own header writer wrote them, tests/golden/reference.npz) -> the readers
(neural_speed_b200/gguf_loader.py, ne_loader.py) -> the device eval step (ns_llama_*), logits against the CPU graph oracle
within the north-star 1e-2 and equal greedy ids where the top-2 margin allows."""
import importlib.util
import os

import numpy as np
import pytest
import torch

import neural_speed_b200 as ns
import oracle
from neural_speed_b200 import gguf_loader, ne_loader
from oracle.llama_model import OracleLlama, greedy

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    ns.lib().bestla_init()
    yield


def _sibling(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(HERE, name + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _check(got, want, tol=1e-2):
    scale = max(1.0, float(np.abs(want).max()))
    assert float(np.abs(got - want).max()) <= tol * scale
    top = np.sort(want)[-2:]
    if top[1] - top[0] > 2 * tol * scale:
        assert int(np.argmax(got)) == greedy(want)


def test_gguf_file_to_device_engine(tmp_path):
    pytest.importorskip("gguf")
    w = _sibling("test_gguf_cpu")
    path = str(tmp_path / "tiny.gguf")
    w._write(path)                                      # Q4_0 layers, Q4_0 embeddings, Q6_K output head, 4 heads over 2 KV heads
    m = gguf_loader.parse(path)
    eng = gguf_loader.load_into_engine(m, n_ctx=64)
    hp = dict(m.hparams, n_ctx=64)
    orc = OracleLlama(hp, m.tok_embd, m.out_norm, m.output[1],
                      [{k: (v[1] if isinstance(v, tuple) else v) for k, v in L.items()} for L in m.layers], fmt="q6_K")
    prompt = [1, 5, 9]
    _check(eng.eval(prompt, 0)[0], orc.eval(prompt, 0))
    for pos, t in enumerate([33, 7, 60, 2], start=3):
        _check(eng.eval([t], pos)[0], orc.eval([t], pos))
    eng.close()


class _BtlaOracleLlama(OracleLlama):
    """matmul weights as (q [K,N] int8, scales, zp, g): BesTLA int8 compute (kernel_ref.h:1825, :2372)"""

    @staticmethod
    def _mm(w, a):
        q, sc, zp, g = w
        a8, asc, azp = oracle.btla_quantize_act_u8(np.ascontiguousarray(a, np.float32), g)
        return oracle.btla_gemv_u8s8(a8, asc, azp, q, sc, zp, g)


@pytest.mark.parametrize("writer", ["reference", "own"])
def test_ne_file_with_btla_blobs_to_device_engine(tmp_path, monkeypatch, writer):
    w = _sibling("test_ne_loader_cpu")
    wh = w._ref_write_header() if writer == "reference" else w._own_write_header
    seen = {}
    real = ns.np_bestla_quantize

    def recording(wf, *a, **k):                          # remember which float matrix every blob of the file came from
        blob = real(wf, *a, **k)
        seen[blob.tobytes()] = np.array(wf, np.float32)
        return blob

    monkeypatch.setattr(ns, "np_bestla_quantize", recording)
    path = str(tmp_path / "tiny.bin")
    w._write(path, wh)
    monkeypatch.setattr(ns, "np_bestla_quantize", real)
    m = ne_loader.parse(path)
    eng = gguf_loader.load_into_engine(m, n_ctx=64)

    def orc_w(tr):
        wf = seen[np.asarray(tr[1]).tobytes()]
        q, sc, zp = oracle.btla_quantize(np.ascontiguousarray(wf.T), 128, 4, False)
        return (q, sc, zp, 128)

    layers = [{k: (orc_w(v) if isinstance(v, tuple) else v) for k, v in L.items()} for L in m.layers]
    orc = _BtlaOracleLlama(dict(m.hparams, n_ctx=64), m.tok_embd, m.out_norm, orc_w(m.output), layers)
    prompt = [1, 5, 9]
    _check(eng.eval(prompt, 0)[0], orc.eval(prompt, 0))
    for pos, t in enumerate([33, 7, 40, 2], start=3):
        _check(eng.eval([t], pos)[0], orc.eval([t], pos))
    eng.close()
