"""GPU parity tests of the LoRA plug-in path (SURVEY 8f row f4; infer.c:408-545 loader, :792-808 q/k/v branches,
:898-903 o branch) against what the unmodified reference computed with the same synthetic plug-in attached
(tests/golden/lora_logits.npz and reference_outputs.json, made by tests/golden/make_golden.py from the strict reference).

Exact mode is bit-identical (logits and the K/V rows that received a LoRA term); fast mode is held to the north-star
tolerance.
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, assert_bits_equal, sha256
from nano_b200 import engine as E, modelfile as mf

pytestmark = pytest.mark.gpu
REF = json.load(open(os.path.join(GOLDEN, "reference_outputs.json")))
SPEC = mf.PRESETS["toy-nano"]
LORA = mf.write_lora(SPEC, 8, 16, seed=7)
S = 24


@pytest.mark.parametrize("quant,gs", [(mf.QUANT_F32, 128), (mf.QUANT_Q80, 64), (mf.QUANT_Q4K, 128)])
def test_lora_exact_mode_bit_identical_to_reference(quant, gs):
    path = mf.cached_model(SPEC, quant, gs)
    want = REF["lora_strict"][f"toy-nano_{quant:02x}_{gs}"]
    eng = E.Engine(path, S, flags=E.FLAG_EXACT); eng.lora_load(LORA)
    toks = mf.teacher_tokens(S, SPEC.vocab)
    for pos in range(S):
        assert sha256(eng.forward(toks[pos], pos)) == want["logits"][pos], f"logits pos {pos}"
    for layer in range(SPEC.n_layer):
        for pos in (0, 5, S - 1):
            k, v = want["kv_rows"][f"{layer}_{pos}"]
            assert sha256(eng.read(E.F_VROW, SPEC.kv_dim, layer, pos)) == v, f"V row L{layer} p{pos}"
            assert sha256(eng.read(E.F_KROW, SPEC.kv_dim, layer, pos)) == k, f"K row L{layer} p{pos}"
    eng.close()


def test_lora_matches_committed_reference_logits():
    g = np.load(os.path.join(GOLDEN, "lora_logits.npz"))
    positions = [0, 1, 7, 23]
    for quant, gs in [(mf.QUANT_F32, 128), (mf.QUANT_Q80, 64)]:
        path = mf.cached_model(SPEC, quant, gs)
        want = g[f"toy-nano_{quant:02x}_{gs}"]
        toks = mf.teacher_tokens(S, SPEC.vocab)
        ex = E.Engine(path, S, flags=E.FLAG_EXACT); ex.lora_load(LORA)
        fa = E.Engine(path, S); fa.lora_load(LORA)
        assert "multi-kernel" in fa.path                        # a plug-in moves the engine to the multi-kernel path
        tol = 1e-4 if quant == mf.QUANT_F32 else 1e-2
        for pos in range(S):
            a = ex.forward(toks[pos], pos); b = fa.forward(toks[pos], pos)
            if pos in positions:
                assert_bits_equal(a, want[positions.index(pos)], f"exact mode {quant:02x} pos {pos}")
                assert np.abs(b - want[positions.index(pos)]).max() <= tol, (quant, pos)
        ex.close(); fa.close()


def test_lora_enable_disable_and_unload_restore_the_base_model():
    path = mf.cached_model(SPEC, mf.QUANT_Q80, 64)
    base = E.Engine(path, S, flags=E.FLAG_NO_STREAM)
    eng = E.Engine(path, S)
    path_before = eng.path
    toks = mf.teacher_tokens(S, SPEC.vocab)
    eng.lora_load(LORA)
    with_lora = [eng.forward(toks[p], p) for p in range(4)]
    eng.lora_enable(False)                                                    # llm_forward(..., lora = NULL)
    assert eng.path == path_before
    for p in range(4):
        got, want = eng.forward(toks[p], p), base.forward(toks[p], p)
        if "multi" in path_before: assert_bits_equal(got, want, f"disabled pos {p}")
        else: assert np.abs(got - want).max() <= 1e-2                          # another execution path: fast-mode tolerance
    eng.lora_enable(True)
    for p in range(4):
        assert_bits_equal(eng.forward(toks[p], p), with_lora[p], f"re-enabled pos {p}")
    eng.lora_unload()
    assert eng.path == path_before
    if "multi" in path_before:
        for p in range(4):
            assert_bits_equal(eng.forward(toks[p], p), base.forward(toks[p], p), f"unloaded pos {p}")
    assert np.abs(with_lora[3] - base.forward(toks[3], 3)).max() > 1e-2        # the plug-in really changed the model
    with pytest.raises(E.NB200Error):
        eng.lora_enable(True)                                                  # nothing loaded any more
    bad = bytearray(LORA); bad[36:40] = (SPEC.n_embd + 1).to_bytes(4, "little")
    with pytest.raises(E.NB200Error):
        eng.lora_load(bytes(bad))                                              # does not fit the base model (infer.c:463-471)
    with pytest.raises(E.NB200Error):
        eng.lora_load(LORA[:1000])                                             # truncated
    eng.close(); base.close()


def test_lora_through_the_reference_api(tmp_path, monkeypatch):
    """llm_context_init(model, lora_path, ...) + generate_next_token: same ids as the reference (exact mode)."""
    monkeypatch.setenv("NB200_EXACT", "1")
    from test_gpu_shim import shim
    path = mf.cached_model(SPEC, mf.QUANT_Q80, 64)
    lp = tmp_path / "toy.lora"
    lp.write_bytes(LORA)
    L = shim()
    ctx = L.llm_context_init(path.encode(), str(lp).encode(), S, 1.2, 0.0, 0.8, 20, 39)
    ids = (C.c_uint32 * (S + 1))()
    for i, t in enumerate([17, 18, 19, 20]):
        ids[i] = t
    for pos in range(S - 1):
        pre = 1 if pos < 3 else 0
        ids[pos + 1] = L.generate_next_token(ctx, ids, pos, pre)
    assert list(ids)[:S] == REF["lora_greedy_penalty_ids"]
    L.llm_context_free(ctx)
