"""Regenerates the committed golden fixtures from the UNMODIFIED reference (strict build).

Needs the original project's sources, compiled into oracle/_ref by oracle/Makefile:
    python tests/golden/make_golden.py                      # the files below
    python tests/golden/make_golden.py reference-outputs    # reference_outputs.json (see reference_outputs())

  sort6_model.bin      the reference's only in-tree fixture: the FP32 sort model embedded in
                       infer/main_sort.c:6-3098 (49,452 bytes), extracted through oracle/ref_harness.c
  sort6_kat.json       seq2seq answers of the reference on it (README.md:379 "114515 -> 111455" and four more)
  toy_logits.npz       teacher-forced logits of the strict reference on seeded synthetic toy files
                       (nano_b200/modelfile.py presets, seed 39) at a few positions, F32 / Q80 / Q4K
  lora_logits.npz      the same with a seeded synthetic LoRA plug-in (rank 8, alpha 16) attached to toy-nano
  q4k_kat.npz          Q4K op-level vectors following the recipe of infer/tools/export_q4k.c:394-450
                       (seed 39 xorshift, d=8, n=768): reference quantize_tensor_q4k bytes + matmul_q4k outputs
"""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from nano_b200 import modelfile as mf            # noqa: E402
from oracle import bindings as ob               # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
TOY_CONFIGS = [("toy-nano", mf.QUANT_F32, 128), ("toy-nano", mf.QUANT_Q80, 64), ("toy-nano", mf.QUANT_Q4K, 128),
               ("toy-qwen3", mf.QUANT_F32, 128), ("toy-qwen3", mf.QUANT_Q80, 64), ("toy-qwen3", mf.QUANT_Q4K, 128)]
TOY_SEQ = 24
TOY_POSITIONS = [0, 1, 7, 23]


def xorshift_f32(n, seed=39):
    """utils.c:959-970 random_f32 stream."""
    M = 0xFFFFFFFFFFFFFFFF
    st = seed
    out = np.zeros(n, np.float32)
    for i in range(n):
        st ^= st >> 12; st ^= (st << 25) & M; st ^= st >> 27
        out[i] = np.float32((((st * 0x2545F4914F6CDD1D) & M) >> 32 >> 8) / 16777216.0)
    return out


def main():
    ob.build()
    sm = ob.sort_model_bytes()
    open(os.path.join(HERE, "sort6_model.bin"), "wb").write(sm)
    ref = ob.RefEngine(sm, 6, penalty=0.0, temperature=0.0, top_p=0.0, top_k=1)
    kat = {s: ref.seq2seq(s, 6) for s in ["251212", "114515", "654321", "000000", "909090", "123321", "777111"]}
    json.dump(kat, open(os.path.join(HERE, "sort6_kat.json"), "w"), indent=1)
    print("sort KAT", kat)

    out = {}
    for name, quant, gs in TOY_CONFIGS:
        spec = mf.PRESETS[name]
        path = mf.cached_model(spec, quant, gs)
        r = ob.RefEngine(path, TOY_SEQ, "strict")
        toks = mf.teacher_tokens(TOY_SEQ, spec.vocab)
        rows = []
        for pos in range(TOY_SEQ):
            lg = r.forward(toks[pos], pos)
            if pos in TOY_POSITIONS:
                rows.append(lg)
        key = f"{name}_{quant:02x}_{gs}"
        out[key] = np.stack(rows)
        r.close()
        print(key, out[key].shape, float(np.abs(out[key]).max()))
    np.savez_compressed(os.path.join(HERE, "toy_logits.npz"), **out)

    # LoRA plug-in (infer.c:792-808, 898-903): strict-reference logits with a seeded synthetic plug-in attached
    lora_out = {}
    for quant, gs in [(mf.QUANT_F32, 128), (mf.QUANT_Q80, 64)]:
        spec = mf.PRESETS["toy-nano"]
        path = mf.cached_model(spec, quant, gs)
        r = ob.RefEngine(path, TOY_SEQ, "strict")
        r.load_lora(mf.write_lora(spec, 8, 16, seed=7))
        toks = mf.teacher_tokens(TOY_SEQ, spec.vocab)
        rows = [r.forward(toks[pos], pos) for pos in range(TOY_SEQ)]
        lora_out[f"toy-nano_{quant:02x}_{gs}"] = np.stack([rows[p] for p in TOY_POSITIONS])
        r.close()
    np.savez_compressed(os.path.join(HERE, "lora_logits.npz"), **lora_out)

    # Noise floor of the reference itself: max |logit(fast build) - logit(strict build)| of the SAME source on the
    # SAME file (SURVEY finding 11).  The fast-mode GPU tolerance is max(north-star tolerance, 1.5 x this floor).
    floors = {}
    S = 40
    for name, quant, gs in TOY_CONFIGS + [("mini-qwen3", mf.QUANT_Q80, 128), ("mini-nano", mf.QUANT_Q80, 128), ("mini-nano", mf.QUANT_Q4K, 128)]:
        spec = mf.PRESETS[name]
        path = mf.cached_model(spec, quant, gs)
        a = ob.RefEngine(path, S, "strict")
        toks = mf.teacher_tokens(S, spec.vocab)
        strict = [a.forward(toks[p], p) for p in range(S)]
        worst = 0.0
        for fl in ("fast_v3", "fast_v4"):
            b = ob.RefEngine(path, S, fl)
            for p in range(S):
                worst = max(worst, float(np.abs(b.forward(toks[p], p) - strict[p]).max()))
            b.close()
        a.close()
        floors[f"{name}_{quant:02x}_{gs}"] = worst
    json.dump(floors, open(os.path.join(HERE, "reference_noise_floor.json"), "w"), indent=1)
    print("floors", floors)

    # Q4K KAT
    L = ob.RefEngine.lib("strict")
    d, n = 8, 768
    rnd = xorshift_f32(d * n + n)
    W = (rnd[: d * n] - np.float32(0.5)).astype(np.float32)
    x = (rnd[d * n:] - np.float32(0.5)).astype(np.float32)
    shape_w = (C.c_uint32 * 2)(d, n)
    shape_x = (C.c_uint32 * 1)(n)
    TW = L.quantize_tensor_q4k(W.ctypes.data_as(ob.f32p), 2, shape_w)
    TX = L.quantize_tensor_q4k(x.ctypes.data_as(ob.f32p), 1, shape_x)
    nbw = L.bytes_num_of_q4k_tensor(TW); nbx = L.bytes_num_of_q4k_tensor(TX)
    wb = np.ctypeslib.as_array(C.cast(TW, ob.u8p), shape=(nbw,)).copy()
    xb = np.ctypeslib.as_array(C.cast(TX, ob.u8p), shape=(nbx,)).copy()
    y = np.zeros(d, np.float32)
    L.matmul_q4k(y.ctypes.data_as(ob.f32p), TX, TW, 0)
    np.savez_compressed(os.path.join(HERE, "q4k_kat.npz"), W=W, x=x, w_tensor=wb, x_tensor=xb, y=y)
    print("q4k kat y", y)


def sha256(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


ORACLE_CONFIGS = TOY_CONFIGS + [("toy-nano-odd", mf.QUANT_F32, 128), ("mini-qwen3", mf.QUANT_Q80, 128)]
SAMPLING_CONFIGS = [("toy-nano", mf.QUANT_Q80, 64), ("mini-qwen3", mf.QUANT_Q80, 128)]
LORA_CONFIGS = [(mf.QUANT_F32, 128), (mf.QUANT_Q80, 64), (mf.QUANT_Q4K, 128)]
Q4K_SHAPES = [[256], [3, 512], [2, 5, 768]]
Q80_GROUPS = [32, 64, 128]


class Q80(C.Structure):                # tensor.h:87-90
    _fields_ = [("q", C.c_void_p), ("s", C.c_void_p)]


def q4k_image(t: np.ndarray) -> bytes:
    """The reference's quantize_tensor_q4k image of t, written by nano_b200.modelfile (checked equal below)."""
    return mf.q4k_frame(t.shape, t.size // 256) + mf.quantize_q4k_blocks(t.reshape(-1, t.shape[-1])).tobytes()


def q80_file_buffer(x: np.ndarray, gs: int) -> np.ndarray:
    """n tensors in file layout [int8 codes | fp32 scales] (tensor.c:49-62), written by nano_b200.modelfile."""
    parts = []
    for row in x:
        q, s = mf.quantize_q80(row, gs)
        parts += [np.ascontiguousarray(q, np.int8).view(np.uint8).reshape(-1), np.ascontiguousarray(s, np.float32).view(np.uint8).reshape(-1)]
    return np.concatenate(parts)


def nano_export() -> dict:
    """test_export_nano.py: the reference's PyTorch model (model.py) loaded with the test's seeded weights, exported by the reference's
    export.py; writes its RoPE tables and logits to nano_export.npz and returns the digests of the exported files."""
    import tempfile
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_export_nano import CONFIG, S, TinyNano, tiny_lora, tokenizer_config
    ref_root = os.environ.get("NANO_REFERENCE_ROOT", os.path.dirname(ob.REFERENCE_SRC))
    sys.path.insert(0, ref_root)
    import model as ref_model
    import importlib.util
    spec = importlib.util.spec_from_file_location("nano_ref_export", os.path.join(ref_root, "export.py"))
    ref_export = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_export)

    def gpt(seed):
        m = ref_model.GPT(ref_model.ModelConfig(**CONFIG)).float().eval()
        tiny = TinyNano(seed, m.freqs_cos.numpy(), m.freqs_sin.numpy())
        missing, unexpected = m.load_state_dict(tiny.state_dict(), strict=False)
        assert not unexpected and all(k.endswith("attention.mask") for k in missing), (missing, unexpected)
        assert m.output.weight is m.tok_embeddings.weight
        return m

    def logits(m, toks):
        with torch.no_grad():
            return np.stack([m(torch.tensor([list(map(int, toks[: p + 1]))], dtype=torch.long))[0][0, -1].float().numpy() for p in range(S)])

    def digest(path):
        return sha256(np.fromfile(path, np.uint8))

    res = {}
    with tempfile.TemporaryDirectory() as td:
        m = gpt(5)
        V = m.config.vocab_size
        toks = mf.teacher_tokens(S, V)
        ref_export.export_model(m, tokenizer_config(V, True), os.path.join(td, "f32.bin"))
        ref_export.export_quantized(m, tokenizer_config(V, True), os.path.join(td, "q80.bin"), group_size=64)
        res["f32"], res["q80"] = digest(os.path.join(td, "f32.bin")), digest(os.path.join(td, "q80.bin"))
        np.savez_compressed(os.path.join(HERE, "nano_export.npz"), freqs_cos=m.freqs_cos.numpy(), freqs_sin=m.freqs_sin.numpy(), logits=logits(m, toks))

        m = gpt(9)
        base = os.path.join(td, "base.bin")
        ref_export.export_model(m, tokenizer_config(V, False), base)
        res["lora_base_f32"] = digest(base)
        lora_sd = tiny_lora(m.config, 4, 11)
        m.to_lora(lora_rank=4, lora_alpha=8)
        with torch.no_grad():
            params = dict(m.named_parameters())
            for k, v in lora_sd.items():
                params[k].copy_(v)
        m.eval()
        plug = os.path.join(td, "lora.bin")
        ref_export.export_lora(m.get_lora_state_dict(), {"lora_rank": 4, "lora_alpha": 8}, m.config, plug)
        res["lora"] = digest(plug)
        want = logits(m, toks)
        r = ob.RefEngine(base, S)
        r.load_lora(open(plug, "rb").read())
        got = np.stack([r.forward(int(toks[p]), p) for p in range(S)])
        r.close()
        err, scale = float(np.abs(got - want).max()), float(np.abs(want).max())
        print(f"reference engine (base file + plug-in) vs the PyTorch LoRA model: max|dlogit| {err:.3e} (logit scale {scale:.2f})")
        assert err < 2e-4 * max(1.0, scale)
    return res


def reference_outputs():
    """tests/golden/reference_outputs.json: what the unmodified strict reference computes in the comparisons of
    test_oracle_vs_reference.py, test_shim_host_helpers.py, test_gpu_shim.py and test_gpu_lora.py.  Bit-exact results are
    stored as SHA-256 digests of their bytes, token ids as lists."""
    ob.build()
    out = {"sort6_model_sha256": sha256(np.frombuffer(ob.sort_model_bytes(), np.uint8))}

    S = 20
    out["oracle_strict"] = {}
    for name, quant, gs in ORACLE_CONFIGS:
        spec = mf.PRESETS[name]
        r = ob.RefEngine(mf.cached_model(spec, quant, gs), S, "strict")
        toks = mf.teacher_tokens(S, spec.vocab)
        logits = [sha256(r.forward(toks[pos], pos)) for pos in range(S)]
        k, v = r.kv()
        out["oracle_strict"][f"{name}_{quant:02x}_{gs}"] = {"logits": logits, "k_cache": sha256(k), "v_cache": sha256(v)}
        r.close()

    S, P = 24, 5
    r = ob.RefEngine(mf.cached_model(mf.PRESETS["toy-nano"], mf.QUANT_Q80, 64), S, "strict", penalty=1.3)
    ids = np.zeros(S + 1, np.uint32); ids[:P] = [9, 8, 7, 9, 8]
    for pos in range(S - 1):
        ids[pos + 1] = r.next(ids, pos, 1 if pos < P - 1 else 0)
    out["greedy_penalty_ids"] = ids.tolist()
    r.close()

    L = ob.RefEngine.lib("strict")
    rng = np.random.default_rng(7)
    w = (rng.standard_normal((37, 512), dtype=np.float32) * np.float32(0.05)).astype(np.float32)
    w[3, :32] = 0.0
    w[5, 32:64] = np.abs(w[5, 32:64])
    w[6, 64:96] = -np.abs(w[6, 64:96])
    T = L.quantize_tensor_q4k(w.ctypes.data_as(ob.f32p), 2, (C.c_uint32 * 2)(37, 512))
    out["q4k_writer_sha256"] = sha256(np.ctypeslib.as_array(C.cast(T, ob.u8p), shape=(L.bytes_num_of_q4k_tensor(T),)))

    rng = np.random.default_rng(3)
    n, d, gs = 512, 40, 64
    x = rng.standard_normal(n, dtype=np.float32)
    x[64:128] = 0.0
    q = np.zeros(n, np.int8); s = np.zeros(n // gs, np.float32)
    t = ob.Q80Tensor(q.ctypes.data_as(ob.i8p), s.ctypes.data_as(ob.f32p))
    L.quantize(C.byref(t), x.ctypes.data_as(ob.f32p), n, gs)
    wq, ws = mf.quantize_q80(rng.standard_normal((d, n), dtype=np.float32) * 0.02, gs)
    tw = ob.Q80Tensor(wq.ctypes.data_as(ob.i8p), ws.ctypes.data_as(ob.f32p))
    y = np.zeros(d, np.float32)
    L.matmul_quant(y.ctypes.data_as(ob.f32p), C.byref(t), C.byref(tw), n, d, gs)
    out["q80_ops"] = {"codes": sha256(q), "scales": sha256(s), "matmul_quant": sha256(y)}

    out["lora_plugin_sha256"] = sha256(np.frombuffer(mf.write_lora(mf.PRESETS["toy-nano"], 8, 16, seed=7), np.uint8))

    # tensor.h:153-163 framing helpers (test_shim_host_helpers.py)
    L.dequantize.argtypes = [C.POINTER(Q80), ob.f32p, C.c_int, C.c_uint32]
    L.parse_quantized_tensors.restype = C.c_void_p
    L.parse_quantized_tensors.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_uint32]
    L.make_q4k_tensor.restype = C.c_void_p
    L.make_q4k_tensor.argtypes = [C.c_uint32, ob.u32p]
    L.dequantize_tensor_q4k.argtypes = [C.c_void_p, ob.f32p, ob.u32p, ob.u32p]
    L.pack_q4k_tensor.restype = C.c_void_p
    L.pack_q4k_tensor.argtypes = [C.c_void_p]
    L.unpack_q4k_tensor.restype = C.c_void_p
    L.unpack_q4k_tensor.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    image = lambda T: np.frombuffer(C.string_at(T, L.bytes_num_of_q4k_tensor(T)), np.uint8).copy()
    out["q4k_framing"] = {}
    for shape in Q4K_SHAPES:
        rng = np.random.default_rng(len(shape))
        t = (rng.standard_normal(shape, dtype=np.float32) * np.float32(0.3)).astype(np.float32)
        sh = (C.c_uint32 * len(shape))(*shape)
        T = L.quantize_tensor_q4k(t.ctypes.data_as(ob.f32p), len(shape), sh)
        img = image(T)
        assert img.tobytes() == q4k_image(t), shape
        empty = image(L.make_q4k_tensor(len(shape), sh))
        deq = np.zeros(t.size, np.float32)
        nd, dims = C.c_uint32(0), (C.c_uint32 * 6)()
        L.dequantize_tensor_q4k(T, deq.ctypes.data_as(ob.f32p), C.byref(nd), dims)
        assert nd.value == len(shape) and list(dims)[:len(shape)] == shape
        packed = L.pack_q4k_tensor(T)
        total = C.c_uint64(0)
        unpacked = L.unpack_q4k_tensor(packed, C.byref(total))
        out["q4k_framing"][str(shape)] = {"image": sha256(img), "empty_header": empty[:44].tobytes().hex(), "empty_size": int(empty.size),
                                          "dequantize": sha256(deq), "pack": sha256(image(packed)), "unpack": sha256(image(unpacked)),
                                          "unpack_total": int(total.value)}
    out["q80_parse"] = {}
    for gs in Q80_GROUPS:
        n_t, size_each = 3, 4 * gs * 5
        rng = np.random.default_rng(gs)
        x = rng.standard_normal((n_t, size_each), dtype=np.float32)
        buf = np.zeros(n_t * (size_each + 4 * (size_each // gs)), np.uint8)
        off = 0
        for i in range(n_t):
            qt = ob.Q80Tensor(C.cast(buf.ctypes.data + off, ob.i8p), C.cast(buf.ctypes.data + off + size_each, ob.f32p))
            L.quantize(C.byref(qt), x[i].ctypes.data_as(ob.f32p), size_each, gs)
            off += size_each + 4 * (size_each // gs)
        assert buf.tobytes() == q80_file_buffer(x, gs).tobytes(), gs
        p = C.c_void_p(buf.ctypes.data)
        tt = L.parse_quantized_tensors(C.byref(p), n_t, size_each, gs)
        assert p.value == buf.ctypes.data + buf.size
        ptrs = np.frombuffer(C.string_at(tt, n_t * 16), np.uint64)
        deq = []
        for i in range(n_t):
            yv = np.zeros(size_each, np.float32)
            L.dequantize(C.byref(Q80(int(ptrs[2 * i]), int(ptrs[2 * i + 1]))), yv.ctypes.data_as(ob.f32p), size_each, gs)
            deq.append(sha256(yv))
        out["q80_parse"][str(gs)] = {"buffer": sha256(buf), "offsets": [int(a) - buf.ctypes.data for a in ptrs], "dequantize": deq}

    # sampled decode through the reference API (test_gpu_shim.py): temperature 0.7, top-p 0.8, penalty 1.1, seed 39
    out["sampling_ids"] = {}
    for name, quant, gs in SAMPLING_CONFIGS:
        spec = mf.PRESETS[name]
        S, P = min(100, spec.block_size), 4
        r = ob.RefEngine(mf.cached_model(spec, quant, gs), S, "strict", penalty=1.1, temperature=0.7, top_p=0.8, top_k=20, seed=39)
        ids = np.zeros(S + 1, np.uint32); ids[:P] = [17, 18, 19, 20]
        for pos in range(S - 1):
            ids[pos + 1] = r.next(ids, pos, 1 if pos < P - 1 else 0)
        out["sampling_ids"][f"{name}_{quant:02x}_{gs}"] = ids[:S].tolist()
        r.close()

    # LoRA plug-in attached (test_gpu_lora.py)
    spec, S = mf.PRESETS["toy-nano"], 24
    lora = mf.write_lora(spec, 8, 16, seed=7)
    out["lora_strict"] = {}
    for quant, gs in LORA_CONFIGS:
        r = ob.RefEngine(mf.cached_model(spec, quant, gs), S, "strict"); r.load_lora(lora)
        toks = mf.teacher_tokens(S, spec.vocab)
        logits = [sha256(r.forward(toks[pos], pos)) for pos in range(S)]
        k, v = r.kv()
        rows = {f"{layer}_{pos}": [sha256(k[layer, pos]), sha256(v[layer, pos])] for layer in range(spec.n_layer) for pos in (0, 5, S - 1)}
        out["lora_strict"][f"toy-nano_{quant:02x}_{gs}"] = {"logits": logits, "kv_rows": rows}
        r.close()
    r = ob.RefEngine(mf.cached_model(spec, mf.QUANT_Q80, 64), S, "strict", penalty=1.2, temperature=0.0); r.load_lora(lora)
    ids = np.zeros(S + 1, np.uint32); ids[:4] = [17, 18, 19, 20]
    for pos in range(S - 1):
        ids[pos + 1] = r.next(ids, pos, 1 if pos < 3 else 0)
    out["lora_greedy_penalty_ids"] = ids[:S].tolist()
    r.close()

    out["nano_export"] = nano_export()

    json.dump(out, open(os.path.join(HERE, "reference_outputs.json"), "w"), indent=1)
    print("reference_outputs.json:", ", ".join(out))


if __name__ == "__main__":
    reference_outputs() if sys.argv[1:] == ["reference-outputs"] else main()
