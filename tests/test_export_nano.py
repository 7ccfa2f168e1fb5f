"""CPU test of the Nano checkpoint export (nano_b200/export_nano.py; SURVEY section 8 row f1): a small seeded instance of a Nano
checkpoint, in the naming of the reference's PyTorch model (model.py), is exported by OUR exporter; the files must be byte-identical
(F32 and Q80, and a LoRA plug-in) to what the reference's export.py wrote for the same weights, and the file's logits (oracle) must
equal the reference PyTorch model's forward pass.  The reference's digests and logits are stored in tests/golden by make_golden.py,
which also checks there that the unmodified reference engine with the exported base file + plug-in reproduces the PyTorch LoRA model."""
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from conftest import GOLDEN, sha256  # noqa: E402
from nano_b200 import export_nano, modelfile as mf  # noqa: E402
from oracle import bindings as ob  # noqa: E402

S = 12
CONFIG = dict(block_size=32, vocab_size=160, n_layer=2, n_embd=128, n_head=4, n_kv_head=2, n_hidden=256)


class TinyNano:
    """What export_nano reads from a checkpoint's model: .config, .state_dict() in model.py's naming (tied classifier), RoPE tables."""

    def __init__(self, seed, freqs_cos, freqs_sin):
        c = self.config = SimpleNamespace(**CONFIG)
        rng = np.random.default_rng(seed)
        kv = c.n_embd // c.n_head * c.n_kv_head
        w = lambda *shape: torch.from_numpy((rng.standard_normal(shape, dtype=np.float32) * np.float32(0.06)).astype(np.float32))
        norm = lambda: torch.from_numpy((1.0 + 0.1 * rng.standard_normal(c.n_embd, dtype=np.float32)).astype(np.float32))
        sd = {"tok_embeddings.weight": w(c.vocab_size, c.n_embd)}
        for i in range(c.n_layer):
            sd.update({f"layers.{i}.attention_norm.weight": norm(), f"layers.{i}.attention.wq.weight": w(c.n_embd, c.n_embd),
                       f"layers.{i}.attention.wk.weight": w(kv, c.n_embd), f"layers.{i}.attention.wv.weight": w(kv, c.n_embd),
                       f"layers.{i}.attention.wo.weight": w(c.n_embd, c.n_embd), f"layers.{i}.ffn_norm.weight": norm(),
                       f"layers.{i}.feed_forward.w1.weight": w(c.n_hidden, c.n_embd), f"layers.{i}.feed_forward.w2.weight": w(c.n_embd, c.n_hidden),
                       f"layers.{i}.feed_forward.w3.weight": w(c.n_hidden, c.n_embd)})
        sd["norm.weight"] = norm()
        sd["output.weight"] = sd["tok_embeddings.weight"]
        self._sd = sd
        self.freqs_cos, self.freqs_sin = torch.as_tensor(freqs_cos), torch.as_tensor(freqs_sin)

    def state_dict(self):
        return dict(self._sd)


def tiny_lora(config, rank, seed):
    """A LoRA checkpoint entry (model.py's get_lora_state_dict naming) with both factors non-zero."""
    rng = np.random.default_rng(seed)
    kv = config.n_embd // config.n_head * config.n_kv_head
    out = {}
    for i in range(config.n_layer):
        for proj, dout in (("wq", config.n_embd), ("wk", kv), ("wv", kv), ("wo", config.n_embd)):
            out[f"layers.{i}.attention.{proj}.lora_a.weight"] = torch.from_numpy(rng.standard_normal((rank, config.n_embd), dtype=np.float32) * np.float32(0.05))
            out[f"layers.{i}.attention.{proj}.lora_b.weight"] = torch.from_numpy(rng.standard_normal((dout, rank), dtype=np.float32) * np.float32(0.05))
    return out


def tokenizer_config(V, special):
    return {"itos": [chr(0x4E00 + i) for i in range(V)], "vocab_size": V, "special_tokens": [chr(0x4E00), chr(0x4E01)] if special else []}


@pytest.fixture(scope="module")
def golden():
    return json.load(open(os.path.join(GOLDEN, "reference_outputs.json")))["nano_export"], np.load(os.path.join(GOLDEN, "nano_export.npz"))


def _digest(path):
    return sha256(np.fromfile(path, np.uint8))


def test_export_is_byte_identical_to_the_reference_exporter_and_matches_the_model(tmp_path, golden):
    want_digests, g = golden
    m = TinyNano(5, g["freqs_cos"], g["freqs_sin"])
    V = m.config.vocab_size
    tok = tokenizer_config(V, True)
    toks = mf.teacher_tokens(S, V)
    want = g["logits"]                                  # the reference PyTorch model's last-position logits after tokens[:p + 1]

    ours = str(tmp_path / "ours.bin")
    export_nano.export_nano(m, ours, mf.QUANT_F32, tokenizer_config=tok)
    assert _digest(ours) == want_digests["f32"], "F32 export differs from the reference exporter"

    o = ob.NanoOracle(ours, S)
    got = np.stack([o.forward(int(toks[p]), p) for p in range(S)])
    o.close()
    err, scale = float(np.abs(got - want).max()), float(np.abs(want).max())
    print(f"exported F32 file vs the PyTorch model: max|dlogit| {err:.3e} (logit scale {scale:.2f})")
    assert err < 2e-4 * max(1.0, scale)

    oursq = str(tmp_path / "ours_q80.bin")
    export_nano.export_nano(m, oursq, mf.QUANT_Q80, 64, tokenizer_config=tok)
    assert _digest(oursq) == want_digests["q80"], "Q80 export differs from the reference exporter"


def test_lora_export_is_byte_identical_and_the_reference_engine_reproduces_the_lora_model(tmp_path, golden):
    """export.py:117-226 / infer.c:436-500: the base file and the plug-in equal the reference exporter's, byte for byte; those
    files, run by the unmodified reference engine (infer.c:792-808, :898-903), reproduce the PyTorch model with the same low-rank
    branches attached (checked where the digests are made, tests/golden/make_golden.py)."""
    want_digests, g = golden
    m = TinyNano(9, g["freqs_cos"], g["freqs_sin"])
    tok = tokenizer_config(m.config.vocab_size, False)
    base = str(tmp_path / "base.bin")
    export_nano.export_nano(m, base, mf.QUANT_F32, tokenizer_config=tok)           # the base model, before the branches are attached
    assert _digest(base) == want_digests["lora_base_f32"], "base export differs from the reference exporter"
    ours = str(tmp_path / "lora_ours.bin")
    export_nano.export_lora(tiny_lora(m.config, 4, 11), 4, 8, m.config, ours)
    assert _digest(ours) == want_digests["lora"], "LoRA export differs from the reference exporter"
