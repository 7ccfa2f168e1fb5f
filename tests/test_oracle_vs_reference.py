"""CPU tests: pin the oracle (oracle/nano_oracle.c) to the reference through the committed goldens.

The reference has no test suite (SURVEY section 4); what pins behaviour is the embedded sort model
(infer/main_sort.c:6-3098, README.md:379) plus outputs of the unmodified strict reference, stored by
tests/golden/make_golden.py (reference_outputs.json holds bit-exact results as SHA-256 digests of their bytes).
"""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, assert_bits_equal, sha256
from nano_b200 import modelfile as mf
from oracle import bindings as ob

REF = json.load(open(os.path.join(GOLDEN, "reference_outputs.json")))

TOY = [("toy-nano", mf.QUANT_F32, 128), ("toy-nano", mf.QUANT_Q80, 64), ("toy-nano", mf.QUANT_Q4K, 128),
       ("toy-qwen3", mf.QUANT_F32, 128), ("toy-qwen3", mf.QUANT_Q80, 64), ("toy-qwen3", mf.QUANT_Q4K, 128)]


def seq2seq_ids(eng, ids):
    """seq2seq of infer.c:1365-1402 restated over a forward(token,pos,causal=0) callable."""
    n = len(ids)
    for _ in range(eng.n_layer):
        for p in range(n):
            eng.forward(ids[p], p, 0)
    return [int(np.argmax(eng.forward(ids[p], p, 0))) for p in range(n)]


def test_sort_model_known_answers_oracle(sort_model):
    kat = json.load(open(os.path.join(GOLDEN, "sort6_kat.json")))
    assert kat["114515"] == "111455"          # README.md:379
    for src, want in kat.items():
        o = ob.NanoOracle(sort_model, 6)
        got = seq2seq_ids(o, [17 + int(c) for c in src])     # digits are ids 17..26 (tokenizer/nano_80.json)
        assert "".join(str(t - 17) for t in got) == want, (src, got)
        o.close()


def test_sort_model_fixture_is_the_embedded_one(sort_model):
    """The committed fixture is the model embedded in the reference (its digest); sort6_kat.json holds the reference's answers on it."""
    assert sha256(np.frombuffer(sort_model, np.uint8)) == REF["sort6_model_sha256"]
    assert len(sort_model) == 49452


@pytest.mark.parametrize("name,quant,gs", TOY)
def test_oracle_matches_golden_logits(name, quant, gs):
    spec = mf.PRESETS[name]
    path = mf.cached_model(spec, quant, gs)
    gold = np.load(os.path.join(GOLDEN, "toy_logits.npz"))[f"{name}_{quant:02x}_{gs}"]
    o = ob.NanoOracle(path, 24)
    toks = mf.teacher_tokens(24, spec.vocab)
    rows = []
    for pos in range(24):
        lg = o.forward(toks[pos], pos)
        if pos in (0, 1, 7, 23):
            rows.append(lg)
    assert_bits_equal(np.stack(rows), gold, f"{name} {quant:#x}")
    o.close()


@pytest.mark.parametrize("name,quant,gs", TOY + [("toy-nano-odd", mf.QUANT_F32, 128), ("mini-qwen3", mf.QUANT_Q80, 128)])
def test_oracle_bit_identical_to_strict_reference(name, quant, gs):
    spec = mf.PRESETS[name]
    path = mf.cached_model(spec, quant, gs)
    want = REF["oracle_strict"][f"{name}_{quant:02x}_{gs}"]
    S = 20
    o = ob.NanoOracle(path, S)
    toks = mf.teacher_tokens(S, spec.vocab)
    for pos in range(S):
        assert sha256(o.forward(toks[pos], pos)) == want["logits"][pos], f"{name} logits differ from the reference at pos {pos}"
    ok, ov = o.kv()
    assert sha256(ok) == want["k_cache"], "k cache"
    assert sha256(ov) == want["v_cache"], "v cache"
    o.close()


def test_oracle_greedy_with_penalty_matches_reference():
    spec = mf.PRESETS["toy-nano"]
    path = mf.cached_model(spec, mf.QUANT_Q80, 64)
    S, P = 24, 5
    o = ob.NanoOracle(path, S)
    ids_o = np.zeros(S + 1, np.uint32); ids_o[:P] = [9, 8, 7, 9, 8]
    for pos in range(S - 1):
        pre = 1 if pos < P - 1 else 0
        ids_o[pos + 1] = o.next_greedy(ids_o, pos, pre, 1.3)
    assert ids_o.tolist() == REF["greedy_penalty_ids"]
    o.close()


def test_q4k_writer_matches_reference_quantiser():
    """nano_b200.modelfile.quantize_q4k_blocks (NumPy) == tensor.c:312 quantize_tensor_q4k, byte for byte."""
    rng = np.random.default_rng(7)
    w = (rng.standard_normal((37, 512), dtype=np.float32) * np.float32(0.05)).astype(np.float32)
    w[3, :32] = 0.0                       # all-zero group
    w[5, 32:64] = np.abs(w[5, 32:64])     # all-positive group (bias 0)
    w[6, 64:96] = -np.abs(w[6, 64:96])    # all-negative group (FLT_TRUE_MIN max quirk)
    mine = mf.q4k_frame((37, 512), 37 * 2) + mf.quantize_q4k_blocks(w).tobytes()
    assert sha256(np.frombuffer(mine, np.uint8)) == REF["q4k_writer_sha256"], "q4k tensor bytes differ from the reference quantiser"


def test_q4k_kat_oracle():
    """Recipe of infer/tools/export_q4k.c:394-450 (seed 39, d=8, n=768): committed reference outputs."""
    k = np.load(os.path.join(GOLDEN, "q4k_kat.npz"))
    L = ob.NanoOracle.lib()
    W, x = k["W"], k["x"]
    wb = np.zeros(8 * 3 * 160, np.uint8); xb = np.zeros(3 * 160, np.uint8)
    L.nor_q4k_quantize_rows(wb.ctypes.data_as(ob.u8p), W.ctypes.data_as(ob.f32p), 8, 768)
    L.nor_q4k_quantize_rows(xb.ctypes.data_as(ob.u8p), x.ctypes.data_as(ob.f32p), 1, 768)
    assert_bits_equal(wb, k["w_tensor"][44:], "weight blocks")
    assert_bits_equal(xb, k["x_tensor"][44:], "activation blocks")
    y = np.zeros(8, np.float32)
    L.nor_matvec_q4k(y.ctypes.data_as(ob.f32p), xb.ctypes.data_as(ob.u8p), wb.ctypes.data_as(ob.u8p), 0, 8, 768)
    assert_bits_equal(y, k["y"], "matmul_q4k")
    assert_bits_equal(mf.quantize_q4k_blocks(W.reshape(8, 768)).reshape(-1), k["w_tensor"][44:], "numpy writer")


def test_q80_ops_match_reference():
    O = ob.NanoOracle.lib()
    want = REF["q80_ops"]
    rng = np.random.default_rng(3)
    n, d, gs = 512, 40, 64
    x = rng.standard_normal(n, dtype=np.float32)
    x[64:128] = 0.0
    q_o = np.zeros(n, np.int8); s_o = np.zeros(n // gs, np.float32)
    O.nor_q80_quantize(q_o.ctypes.data_as(ob.i8p), s_o.ctypes.data_as(ob.f32p), x.ctypes.data_as(ob.f32p), n, gs)
    assert sha256(q_o) == want["codes"], "codes"
    assert sha256(s_o) == want["scales"], "scales"
    wq, ws = mf.quantize_q80(rng.standard_normal((d, n), dtype=np.float32) * 0.02, gs)
    y_o = np.zeros(d, np.float32)
    O.nor_matvec_q80(y_o.ctypes.data_as(ob.f32p), q_o.ctypes.data_as(ob.i8p), s_o.ctypes.data_as(ob.f32p),
                     wq.ctypes.data_as(ob.i8p), ws.ctypes.data, n, d, gs)
    assert sha256(y_o) == want["matmul_quant"], "matmul_quant"


def test_expf_ref_equals_host_libm():
    """The exact-mode device expf (csrc/expf_ref.cuh) evaluated on the host == libm expf on sampled floats."""
    from nano_b200 import engine as E
    import struct
    fb = lambda f: struct.unpack("<I", struct.pack("<f", f))[0]
    L = ob.NanoOracle.lib()
    for lo, hi in ((0, fb(89.0)), (0x80000000, fb(-104.5))):
        b = np.arange(lo, hi, 997, dtype=np.uint32)
        x = b.view(np.float32)
        want = np.empty_like(x)
        L.nor_expf_array(want.ctypes.data_as(ob.f32p), x.ctypes.data_as(ob.f32p), x.size)
        assert_bits_equal(E.host_expf_ref(x), want, "expf")


def test_lora_golden_is_what_the_reference_computes():
    """Pins tests/golden/lora_logits.npz (the GPU LoRA tests' fixture) to what the unmodified strict reference computed with
    the same synthetic plug-in (the digests of its logits at every position), checks that the plug-in is the one those were
    computed with and that its layout is the one parse_lora_file reads (infer.c:436-500)."""
    spec = mf.PRESETS["toy-nano"]
    lora = mf.write_lora(spec, 8, 16, seed=7)
    assert len(lora) == 256 + 4 * spec.n_layer * 8 * (4 * spec.n_embd + 2 * spec.n_embd + 2 * spec.kv_dim)
    assert sha256(np.frombuffer(lora, np.uint8)) == REF["lora_plugin_sha256"]
    gold = np.load(os.path.join(GOLDEN, "lora_logits.npz"))
    base = np.load(os.path.join(GOLDEN, "toy_logits.npz"))
    for quant, gs in [(mf.QUANT_F32, 128), (mf.QUANT_Q80, 64)]:
        key = f"toy-nano_{quant:02x}_{gs}"
        digests = REF["lora_strict"][key]["logits"]
        for row, pos in zip(gold[key], (0, 1, 7, 23)):
            assert sha256(row) == digests[pos], f"lora golden {quant:#x} pos {pos}"
        assert (np.abs(gold[key] - base[key]).max(axis=1) > 1e-2).all(), "the plug-in must change the logits"
