"""GPU tests through the REFERENCE's host API (libnano_infer_b200.so: llm_context_init, generate_next_token,
llm_session_step, seq2seq ...) -- the calls nano_cli / nano_sort / nano_wss make -- against the oracle port and against
what the unmodified reference computed (tests/golden).  tests/host_stub.c stands in for the host objects the shim imports."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, assert_bits_equal, load_host_stub
from nano_b200 import build as nb_build, modelfile as mf
from oracle import bindings as ob

pytestmark = pytest.mark.gpu
REF = json.load(open(os.path.join(GOLDEN, "reference_outputs.json")))


class Session(C.Structure):       # infer.h:236-250
    _fields_ = [("prompt", C.c_void_p), ("num_prompt_tokens", C.c_uint32), ("max_seq_len", C.c_uint32), ("output_ids", C.POINTER(C.c_uint32)),
                ("output_count", C.c_uint32), ("output_text", C.c_wchar_p), ("next_token", C.c_uint32), ("pos", C.c_uint32),
                ("is_prefilling", C.c_int32), ("t_0", C.c_uint64), ("t_1", C.c_uint64), ("tps", C.c_float)]


_shim = None


def shim():
    global _shim
    if _shim is None:
        load_host_stub()                                       # allocation, sampler RNG, tokenizer: what a host links beside the shim
        L = C.CDLL(nb_build.SHIM_SO, mode=C.RTLD_GLOBAL)
        L.llm_context_init.restype = C.c_void_p
        L.llm_context_init.argtypes = [C.c_char_p, C.c_char_p, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_uint32, C.c_uint64]
        L.llm_context_init_from_buffer.restype = C.c_void_p
        L.llm_context_init_from_buffer.argtypes = [C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_uint32, C.c_uint64]
        L.llm_context_free.argtypes = [C.c_void_p]
        L.generate_next_token.restype = C.c_uint32
        L.generate_next_token.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.c_uint32, C.c_int]
        L.seq2seq.argtypes = [C.c_void_p, C.c_wchar_p, C.c_wchar_p, C.c_uint32]
        L.llm_session_init.restype = C.POINTER(Session)
        L.llm_session_init.argtypes = [C.c_void_p, C.c_wchar_p, C.c_uint32, C.c_int32]
        L.llm_session_step.restype = C.c_int32
        L.llm_session_step.argtypes = [C.c_void_p, C.POINTER(Session)]
        L.llm_session_free.argtypes = [C.POINTER(Session)]
        _shim = L
    return _shim


def test_sort_demo_through_reference_api(sort_model):
    """main_sort.c's calls: llm_context_init_from_buffer(model, 6, 0, 0, 0, 1, 39) + seq2seq (README.md:379)."""
    L = shim()
    img = np.frombuffer(sort_model, np.uint8).copy()
    ctx = L.llm_context_init_from_buffer(img.ctypes.data, 6, 0.0, 0.0, 0.0, 1, 39)
    kat = json.load(open(os.path.join(GOLDEN, "sort6_kat.json")))
    for src, want in kat.items():
        out = C.create_unicode_buffer(16)
        L.seq2seq(ctx, src, out, 6)
        assert out.value == want, (src, out.value)


@pytest.mark.parametrize("penalty", [1.0, 1.3])
def test_generate_next_token_greedy_matches_reference(penalty, monkeypatch):
    """generate_next_token(ctx, ids, pos, is_prefilling) with temperature 0: ids identical to the oracle (exact mode)."""
    monkeypatch.setenv("NB200_EXACT", "1")
    spec = mf.PRESETS["toy-qwen3"]
    path = mf.cached_model(spec, mf.QUANT_Q80, 64)
    S, P = 32, 5
    L = shim()
    ctx = L.llm_context_init(path.encode(), None, S, penalty, 0.0, 0.8, 20, 39)
    ids = (C.c_uint32 * (S + 1))(); want = np.zeros(S + 1, np.uint32)
    for i, t in enumerate([7, 8, 9, 8, 7]):
        ids[i] = t; want[i] = t
    o = ob.NanoOracle(path, S)
    for pos in range(S - 1):
        pre = 1 if pos < P - 1 else 0
        ids[pos + 1] = L.generate_next_token(ctx, ids, pos, pre)
        want[pos + 1] = o.next_greedy(want, pos, pre, penalty)
    assert list(ids)[:S] == want[:S].tolist()
    L.llm_context_free(ctx)
    o.close()


@pytest.mark.parametrize("host_sampler", ["0", "1"], ids=["device-sampler", "host-sampler"])
@pytest.mark.parametrize("name,quant,gs", [("toy-nano", mf.QUANT_Q80, 64), ("mini-qwen3", mf.QUANT_Q80, 128)])
def test_temperature_sampling_matches_reference(name, quant, gs, host_sampler, monkeypatch):
    """temperature 0.7 / top-p 0.8 (main_cli.c:227) over 60 (toy-nano) / 96 (mini-qwen3) sampled steps: with bit-identical logits (exact mode) and the reference's own xorshift
    coin, the ids equal those the unmodified strict reference produced (stored in tests/golden) -- for the device-side sampler (softmax, cutoff, stable descending order,
    sequential top-p scan on the GPU; 32 bytes back per token) and for the host restatement (NB200_HOST_SAMPLER=1, logits D2H)."""
    monkeypatch.setenv("NB200_EXACT", "1")
    monkeypatch.setenv("NB200_HOST_SAMPLER", host_sampler)
    spec = mf.PRESETS[name]
    path = mf.cached_model(spec, quant, gs)
    S, P = min(100, spec.block_size), 4            # never beyond the model's RoPE table
    L = shim()
    ctx = L.llm_context_init(path.encode(), None, S, 1.1, 0.7, 0.8, 20, 39)
    want = REF["sampling_ids"][f"{name}_{quant:02x}_{gs}"]
    ids = (C.c_uint32 * (S + 1))()
    for i, t in enumerate([17, 18, 19, 20]):
        ids[i] = t
    for pos in range(S - 1):
        pre = 1 if pos < P - 1 else 0
        ids[pos + 1] = L.generate_next_token(ctx, ids, pos, pre)
    assert list(ids)[:S] == want
    assert len(set(list(ids)[P:S])) > 20          # it really sampled: not a constant stream
    L.llm_context_free(ctx)


def test_session_api_runs_and_stops_at_length():
    spec = mf.PRESETS["toy-nano"]
    path = mf.cached_model(spec, mf.QUANT_Q80, 64)
    L = shim()
    ctx = L.llm_context_init(path.encode(), None, 24, 1.0, 0.0, 0.8, 20, 39)
    s = L.llm_session_init(ctx, "0123", 24, 0)
    assert s.contents.num_prompt_tokens == 4
    statuses = []
    for _ in range(30):
        st = L.llm_session_step(ctx, s)
        statuses.append(st)
        if st <= 0:
            break
    assert statuses[:3] == [11, 11, 11] and 12 in statuses          # LLM_RUNNING_IN_PREFILLING x3, then decoding
    assert statuses[-1] in (-10, -20)                                # EOS (ids 0/3) or length limit (infer.h:52-55)
    L.llm_session_free(s)
    L.llm_context_free(ctx)


@pytest.mark.skipif(not os.path.exists(ob.NANO_CLI), reason="needs the reference's main_cli.c objects (oracle/Makefile)")
def test_nano_cli_binary_starts_and_reports_missing_model():
    """The unmodified main_cli.c linked against our libraries runs; its model path is hard-coded (main_cli.c:12),
    so without that file it must exit through the reference's own error path."""
    r = subprocess.run([ob.NANO_CLI], input=b"", capture_output=True, timeout=60)
    assert r.returncode != 0
    assert b"open" in r.stderr.lower() or b"couldn" in r.stderr.lower()


def test_q4k_tensor_functions_through_reference_names():
    """tensor.h:160-166 as the reference's tools/export_q4k.c calls them (quantize_tensor_q4k -> matmul_q4k on a 3-D
    weight with a layer index), against the outputs committed from the unmodified reference and the oracle."""
    L = shim()
    L.quantize_tensor_q4k.restype = C.c_void_p
    L.quantize_tensor_q4k.argtypes = [C.POINTER(C.c_float), C.c_uint32, C.POINTER(C.c_uint32)]
    L.bytes_num_of_q4k_tensor.restype = C.c_uint64
    L.bytes_num_of_q4k_tensor.argtypes = [C.c_void_p]
    L.matmul_q4k.argtypes = [C.POINTER(C.c_float), C.c_void_p, C.c_void_p, C.c_uint32]
    f32p = C.POINTER(C.c_float)
    k = np.load(os.path.join(GOLDEN, "q4k_kat.npz"))

    def qt(arr, shape):
        a = np.ascontiguousarray(arr, np.float32)
        sh = (C.c_uint32 * len(shape))(*shape)
        T = L.quantize_tensor_q4k(a.ctypes.data_as(f32p), len(shape), sh)
        n = L.bytes_num_of_q4k_tensor(T)
        return T, np.frombuffer(C.string_at(T, n), np.uint8).copy()

    xT, xb = qt(k["x"], [768])
    wT, wb = qt(k["W"], [8, 768])
    assert_bits_equal(xb, k["x_tensor"], "x tensor image"); assert_bits_equal(wb, k["w_tensor"], "w tensor image")
    y = np.zeros(8, np.float32)
    L.matmul_q4k(y.ctypes.data_as(f32p), xT, wT, 0)
    assert_bits_equal(y, k["y"], "matmul_q4k")
    # 3-D weight, layer slice 1 (tensor.c:452-461)
    rng = np.random.default_rng(5)
    W3 = (rng.standard_normal((3, 10, 512), dtype=np.float32) * np.float32(0.05)).astype(np.float32)
    x = rng.standard_normal(512, dtype=np.float32)
    w3T, _ = qt(W3, [3, 10, 512]); x2T, x2b = qt(x, [512])
    y3 = np.zeros(10, np.float32)
    L.matmul_q4k(y3.ctypes.data_as(f32p), x2T, w3T, 1)
    want = np.zeros(10, np.float32)
    wblk = mf.quantize_q4k_blocks(W3[1]).reshape(-1)
    ob.NanoOracle.lib().nor_matvec_q4k(want.ctypes.data_as(ob.f32p), x2b[44:].ctypes.data_as(ob.u8p), wblk.ctypes.data_as(ob.u8p), 0, 10, 512)
    assert_bits_equal(y3, want, "matmul_q4k layer 1")
