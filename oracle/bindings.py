"""ctypes bindings for the CHECKERS (test infrastructure only).

* `NanoOracle`  -> oracle/libnano_oracle.so  (our C restatement, oracle/nano_oracle.c)
* `RefEngine`   -> oracle/_ref/libnano_ref_<flavour>.so (the unmodified reference, oracle/Makefile)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional

import numpy as np

# libgomp reads these once, when the first OpenMP library is loaded into the process.  Parity tests run tiny
# models: a full-machine team that spin-waits between hundreds of small parallel regions is pathological on
# the many-core GPU hosts.  bench.py's CPU baselines set their own values in a subprocess.
os.environ.setdefault("OMP_NUM_THREADS", "8")
os.environ.setdefault("OMP_WAIT_POLICY", "passive")

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")
NANO_CLI = os.path.join(HERE, "nano_cli")                   # the reference's main_cli.c linked against our libraries
NANO_CLI_HOST = os.path.join(REF_DIR, "libnano_cli_host.a")  # its unmodified objects
REFERENCE_SRC = "/root/reference/infer"

f32p = C.POINTER(C.c_float)
u32p = C.POINTER(C.c_uint32)
u8p = C.POINTER(C.c_uint8)
i8p = C.POINTER(C.c_int8)

# infer.h:65-76
PHASE = dict(EMBEDDING=1, ATTN_NORM=2, QKV=3, QK_ROPE=4, MHA=5, O=6, FFN_NORM=7, W1W3=8, W2=9, FINAL_NORM=10, CLASSIFY=11)
FIELD = dict(x=0, xb=1, xba=2, xb2=3, hb=4, hb2=5, q=6, k=7, v=8, logits=9, k_cache=10, v_cache=11, att=12)


def build(quiet: bool = True) -> None:
    """Compile the restatement and (when /root/reference exists) the reference flavours."""
    subprocess.run(["make", "-C", HERE, "-j4", "all"], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def link_nano_cli() -> str:
    """Link oracle/nano_cli afresh from the reference's objects and our libraries (oracle/Makefile, target cli)."""
    if os.path.exists(NANO_CLI):
        os.remove(NANO_CLI)
    subprocess.run(["make", "-C", HERE, "cli"], check=True, stdout=subprocess.DEVNULL)
    return NANO_CLI


def _ptr(a: np.ndarray, typ):
    return a.ctypes.data_as(typ)


def cpu_flags() -> set:
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    return set(line.split(":", 1)[1].split())
    except OSError:
        pass
    return set()


def ref_available(flavour: str = "strict") -> bool:
    return os.path.exists(os.path.join(REF_DIR, f"libnano_ref_{flavour}.so"))


def best_fast_flavour() -> Optional[str]:
    fl = cpu_flags()
    if {"avx512f", "avx512bw", "avx512vl", "avx512dq", "avx512cd", "avx512_vnni"} <= fl and ref_available("fast_v4"):
        return "fast_v4"
    if {"avx2", "fma", "bmi2"} <= fl and ref_available("fast_v3"):
        return "fast_v3"
    return None


class NanoOracle:
    """Restatement engine over a model file image."""

    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            path = os.path.join(HERE, "libnano_oracle.so")
            if not os.path.exists(path):
                build()
            L = C.CDLL(path)
            L.nor_open.restype = C.c_void_p
            L.nor_open.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32]
            L.nor_close.argtypes = [C.c_void_p]
            L.nor_forward.restype = f32p
            L.nor_forward.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_int]
            L.nor_next_greedy.restype = C.c_uint32
            L.nor_next_greedy.argtypes = [C.c_void_p, u32p, C.c_uint32, C.c_int, C.c_float]
            L.nor_config.argtypes = [C.c_void_p, u32p]
            L.nor_set_probe.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, f32p, C.c_uint32]
            for n in ("nor_kcache", "nor_vcache", "nor_logits"):
                getattr(L, n).restype = f32p
                getattr(L, n).argtypes = [C.c_void_p]
            L.nor_rmsnorm.argtypes = [f32p, f32p, f32p, C.c_int]
            L.nor_softmax.argtypes = [f32p, C.c_int]
            L.nor_matvec_f32.argtypes = [f32p, f32p, C.c_void_p, C.c_int, C.c_int]
            L.nor_q80_quantize.argtypes = [i8p, f32p, f32p, C.c_int, C.c_int]
            L.nor_matvec_q80.argtypes = [f32p, i8p, f32p, i8p, C.c_void_p, C.c_int, C.c_int, C.c_int]
            L.nor_rope.argtypes = [f32p, C.c_int, f32p, f32p, C.c_int]
            L.nor_q4k_quantize_rows.argtypes = [u8p, f32p, C.c_uint64, C.c_uint32]
            L.nor_q4k_dequant_block.restype = C.c_uint32
            L.nor_q4k_dequant_block.argtypes = [u8p, f32p]
            L.nor_matvec_q4k.argtypes = [f32p, u8p, u8p, C.c_uint64, C.c_uint32, C.c_uint32]
            L.nor_expf_array.argtypes = [f32p, f32p, C.c_uint64]
            L.nor_set_threads.argtypes = [C.c_int]
            L.nor_max_threads.restype = C.c_int
            cls._lib = L
        return cls._lib

    def __init__(self, path_or_bytes, max_seq: int):
        L = self.lib()
        if isinstance(path_or_bytes, (bytes, bytearray, np.ndarray)):
            self.image = np.frombuffer(bytes(path_or_bytes), dtype=np.uint8).copy()
        else:
            self.image = np.fromfile(path_or_bytes, dtype=np.uint8)
        self.h = L.nor_open(self.image.ctypes.data, self.image.size, max_seq)
        cfg = (C.c_uint32 * 16)()
        L.nor_config(self.h, cfg)
        (self.block_size, self.vocab, self.n_layer, self.n_embd, self.n_head, self.n_kv_head, self.n_hidden,
         self.tied, self.head_dim, self.arch, self.quant, self.gs, self.max_seq, self.q_dim, self.kv_dim) = list(cfg)[:15]

    def close(self):
        if self.h:
            self.lib().nor_close(self.h)
            self.h = None

    def forward(self, token: int, pos: int, causal: int = 1) -> np.ndarray:
        p = self.lib().nor_forward(self.h, int(token), int(pos), causal)
        return np.ctypeslib.as_array(p, shape=(self.vocab,)).copy()

    def next_greedy(self, ids: np.ndarray, pos: int, prefilling: int, penalty: float = 1.0) -> int:
        return int(self.lib().nor_next_greedy(self.h, _ptr(ids, u32p), pos, prefilling, penalty))

    def logits(self) -> np.ndarray:
        return np.ctypeslib.as_array(self.lib().nor_logits(self.h), shape=(self.vocab,)).copy()

    def kv(self):
        n = self.n_layer * self.max_seq * self.kv_dim
        k = np.ctypeslib.as_array(self.lib().nor_kcache(self.h), shape=(n,)).reshape(self.n_layer, self.max_seq, self.kv_dim)
        v = np.ctypeslib.as_array(self.lib().nor_vcache(self.h), shape=(n,)).reshape(self.n_layer, self.max_seq, self.kv_dim)
        return k, v

    def probe(self, layer: int, phase: str, field: str, count: int) -> np.ndarray:
        buf = np.zeros(count, dtype=np.float32)
        self.lib().nor_set_probe(self.h, layer, PHASE[phase], FIELD[field], _ptr(buf, f32p), count)
        return buf


class Q80Tensor(C.Structure):          # tensor.h:84-90
    _fields_ = [("q", i8p), ("s", f32p)]


class RefEngine:
    """The unmodified reference (strict or fast build) behind oracle/ref_harness.c."""

    _libs = {}

    @classmethod
    def lib(cls, flavour: str):
        if flavour not in cls._libs:
            path = os.path.join(REF_DIR, f"libnano_ref_{flavour}.so")
            if not os.path.exists(path):
                if os.path.isdir(REFERENCE_SRC):
                    build()
                else:
                    raise FileNotFoundError(path)
            L = C.CDLL(path)
            L.orh_open_file.restype = C.c_void_p
            L.orh_open_file.argtypes = [C.c_char_p, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_uint32, C.c_uint64]
            L.orh_open_buffer.restype = C.c_void_p
            L.orh_open_buffer.argtypes = [C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_uint32, C.c_uint64]
            L.orh_close_file.argtypes = [C.c_void_p]
            L.orh_load_lora.argtypes = [C.c_void_p, C.c_void_p]
            L.orh_forward.restype = f32p
            L.orh_forward.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]
            L.orh_next.restype = C.c_uint32
            L.orh_next.argtypes = [C.c_void_p, u32p, C.c_uint32, C.c_int]
            L.orh_config.argtypes = [C.c_void_p, u32p]
            L.orh_state.restype = f32p
            L.orh_state.argtypes = [C.c_void_p, C.c_int]
            L.orh_probe_add.restype = C.c_int
            L.orh_probe_add.argtypes = [C.c_int32, C.c_int32, C.c_int32, f32p, C.c_uint32]
            L.orh_sort_model.restype = u8p
            L.orh_sort_model.argtypes = [u32p]
            L.orh_abi_layout.restype = C.c_uint32
            L.orh_abi_layout.argtypes = [u32p, C.c_uint32]
            L.seq2seq.argtypes = [C.c_void_p, C.c_wchar_p, C.c_wchar_p, C.c_uint32]
            # raw reference ops (non-static symbols of infer.c / tensor.c)
            L.rmsnorm.argtypes = [f32p, f32p, f32p, C.c_int]
            L.softmax.argtypes = [f32p, C.c_int]
            L.matmul.argtypes = [f32p, f32p, f32p, C.c_int, C.c_int]
            L.quantize.argtypes = [C.POINTER(Q80Tensor), f32p, C.c_int, C.c_uint32]
            L.matmul_quant.argtypes = [f32p, C.POINTER(Q80Tensor), C.POINTER(Q80Tensor), C.c_int, C.c_int, C.c_uint32]
            L.rope.argtypes = [f32p, C.c_uint32, C.c_uint32, f32p, f32p]
            L.rope_qwen3.argtypes = [f32p, C.c_uint32, C.c_uint32, f32p, f32p]
            L.quantize_tensor_q4k.restype = C.c_void_p
            L.quantize_tensor_q4k.argtypes = [f32p, C.c_uint32, u32p]
            L.bytes_num_of_q4k_tensor.restype = C.c_uint64
            L.bytes_num_of_q4k_tensor.argtypes = [C.c_void_p]
            L.matmul_q4k.argtypes = [f32p, C.c_void_p, C.c_void_p, C.c_uint32]
            cls._libs[flavour] = L
        return cls._libs[flavour]

    def __init__(self, path_or_bytes, max_seq: int, flavour: str = "strict", penalty: float = 1.0,
                 temperature: float = 0.0, top_p: float = 0.8, top_k: int = 20, seed: int = 39):
        L = self.lib(flavour)
        self.L = L
        self.from_file = isinstance(path_or_bytes, str)
        if self.from_file:
            self.h = L.orh_open_file(path_or_bytes.encode(), max_seq, penalty, temperature, top_p, top_k, seed)
        else:
            self.image = np.frombuffer(bytes(path_or_bytes), dtype=np.uint8).copy()
            self.h = L.orh_open_buffer(self.image.ctypes.data, max_seq, penalty, temperature, top_p, top_k, seed)
        cfg = (C.c_uint32 * 16)()
        L.orh_config(self.h, cfg)
        (self.block_size, self.vocab, self.n_layer, self.n_embd, self.n_head, self.n_kv_head, self.n_hidden,
         self.tied, self.head_dim, self.arch, self.quant, self.gs, self.max_seq) = list(cfg)[:13]
        hd = self.head_dim if self.arch == 3 else self.n_embd // self.n_head
        self.kv_dim = hd * self.n_kv_head
        self._probe_bufs = []

    def close(self):
        if self.h and self.from_file:
            self.L.orh_close_file(self.h)
        self.h = None

    def load_lora(self, image: bytes) -> None:
        """Attach a LoRA plug-in (the reference points into the buffer: keep it alive with the engine)."""
        self._lora_image = np.frombuffer(bytes(image), dtype=np.uint8).copy()
        self.L.orh_load_lora(self.h, self._lora_image.ctypes.data)

    def forward(self, token: int, pos: int, causal: int = 1) -> np.ndarray:
        p = self.L.orh_forward(self.h, int(token), int(pos), causal)
        return np.ctypeslib.as_array(p, shape=(self.vocab,)).copy()

    def next(self, ids: np.ndarray, pos: int, prefilling: int) -> int:
        return int(self.L.orh_next(self.h, _ptr(ids, u32p), pos, prefilling))

    def state(self, field: str, count: int) -> np.ndarray:
        return np.ctypeslib.as_array(self.L.orh_state(self.h, FIELD[field]), shape=(count,)).copy()

    def kv(self):
        n = self.n_layer * self.max_seq * self.kv_dim
        k = self.state("k_cache", n).reshape(self.n_layer, self.max_seq, self.kv_dim)
        v = self.state("v_cache", n).reshape(self.n_layer, self.max_seq, self.kv_dim)
        return k, v

    def probe_clear(self):
        self.L.orh_probe_clear()
        self._probe_bufs = []

    def probe(self, layer: int, phase: str, field: str, count: int) -> np.ndarray:
        buf = np.zeros(count, dtype=np.float32)
        self._probe_bufs.append(buf)
        self.L.orh_probe_add(layer, PHASE[phase], FIELD[field], _ptr(buf, f32p), count)
        return buf

    def seq2seq(self, text: str, n: int) -> str:
        out = C.create_unicode_buffer(n + 8)
        self.L.seq2seq(self.h, text, out, n)
        return out.value


def sort_model_bytes(flavour: str = "strict") -> bytes:
    """The reference's embedded fixture (main_sort.c:6-3098)."""
    L = RefEngine.lib(flavour)
    n = C.c_uint32(0)
    p = L.orh_sort_model(C.byref(n))
    return bytes(np.ctypeslib.as_array(p, shape=(n.value,)))
