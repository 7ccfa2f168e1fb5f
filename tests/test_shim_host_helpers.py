"""CPU tests of the host-side framing helpers of the reference API that our shim re-implements (tensor.h:153-163):
dequantize, parse_quantized_tensors, bytes_num_of_q4k_tensor, make_q4k_tensor, dequantize_tensor_q4k, pack_q4k_tensor,
unpack_q4k_tensor -- called on the same host buffers the unmodified reference (strict build) was given, and compared bit for bit
with what it returned (tests/golden/reference_outputs.json, written by tests/golden/make_golden.py).  The inputs are the
reference's own quantiser outputs, reproduced byte for byte by nano_b200.modelfile's writers, so no GPU is involved
(VERDICT r1 rows a16 / a17)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_host_stub, sha256
from nano_b200 import build as nb_build, modelfile as mf

REF = json.load(open(os.path.join(GOLDEN, "reference_outputs.json")))
f32p, u32p, u8p = C.POINTER(C.c_float), C.POINTER(C.c_uint32), C.POINTER(C.c_uint8)


class Q80(C.Structure):                # tensor.h:87-90
    _fields_ = [("q", C.c_void_p), ("s", C.c_void_p)]


@pytest.fixture(scope="module")
def ours():
    load_host_stub()                                                            # the host objects the shim imports
    L = C.CDLL(nb_build.SHIM_SO, mode=C.RTLD_LOCAL)
    L.dequantize.argtypes = [C.POINTER(Q80), f32p, C.c_int, C.c_uint32]
    L.parse_quantized_tensors.restype = C.c_void_p
    L.parse_quantized_tensors.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_uint32]
    L.bytes_num_of_q4k_tensor.restype = C.c_uint64
    L.bytes_num_of_q4k_tensor.argtypes = [C.c_void_p]
    L.make_q4k_tensor.restype = C.c_void_p
    L.make_q4k_tensor.argtypes = [C.c_uint32, u32p]
    L.dequantize_tensor_q4k.argtypes = [C.c_void_p, f32p, u32p, u32p]
    L.pack_q4k_tensor.restype = C.c_void_p
    L.pack_q4k_tensor.argtypes = [C.c_void_p]
    L.unpack_q4k_tensor.restype = C.c_void_p
    L.unpack_q4k_tensor.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    return L


def _image(L, T):
    return np.frombuffer(C.string_at(T, L.bytes_num_of_q4k_tensor(T)), np.uint8).copy()


@pytest.mark.parametrize("shape", [[256], [3, 512], [2, 5, 768]])
def test_q4k_framing_helpers_match_the_reference(ours, shape):
    want = REF["q4k_framing"][str(shape)]
    rng = np.random.default_rng(len(shape))
    t = (rng.standard_normal(shape, dtype=np.float32) * np.float32(0.3)).astype(np.float32)
    sh = (C.c_uint32 * len(shape))(*shape)
    img = np.frombuffer(mf.q4k_frame(shape, t.size // 256) + mf.quantize_q4k_blocks(t.reshape(-1, shape[-1])).tobytes(), np.uint8).copy()
    assert sha256(img) == want["image"], "the input is not the reference quantiser's tensor image"
    T = img.ctypes.data
    # size and raw image
    assert ours.bytes_num_of_q4k_tensor(T) == img.size
    # an empty tensor of the same shape has the same header fields and size (tensor.c:76-111)
    b = _image(ours, ours.make_q4k_tensor(len(shape), sh))
    nhdr = 8 + 4 + 4 + 24 + 4                                                    # tensor.h:129-134: bytes, header, ndim, shape[6], num_blocks
    assert b[:nhdr].tobytes().hex() == want["empty_header"], "make_q4k_tensor header"
    assert b.size == want["empty_size"]
    # dequantise the reference's tensor
    out_o = np.zeros(t.size, np.float32)
    nd_o, sh_o = C.c_uint32(0), (C.c_uint32 * 6)()
    ours.dequantize_tensor_q4k(T, out_o.ctypes.data_as(f32p), C.byref(nd_o), sh_o)
    assert nd_o.value == len(shape) and list(sh_o)[:len(shape)] == shape
    assert sha256(out_o) == want["dequantize"], "dequantize_tensor_q4k"
    # pack / unpack round trip (tensor.c: the packed form is the tensor image itself)
    po = ours.pack_q4k_tensor(T)
    assert sha256(_image(ours, po)) == want["pack"], "pack_q4k_tensor"
    tot_o = C.c_uint64(0)
    uo = ours.unpack_q4k_tensor(po, C.byref(tot_o))
    assert tot_o.value == want["unpack_total"]
    assert sha256(_image(ours, uo)) == want["unpack"], "unpack_q4k_tensor"


@pytest.mark.parametrize("gs", [32, 64, 128])
def test_q80_parse_and_dequantize_match_the_reference(ours, gs):
    """parse_quantized_tensors walks a file-layout buffer of n tensors [int8 codes | fp32 scales] (tensor.c:49-62); dequantize tensor.c:12-17."""
    want = REF["q80_parse"][str(gs)]
    n_t, size_each = 3, 4 * gs * 5
    rng = np.random.default_rng(gs)
    x = rng.standard_normal((n_t, size_each), dtype=np.float32)
    parts = []
    for i in range(n_t):                                                         # the reference's quantiser output, in file layout
        q, s = mf.quantize_q80(x[i], gs)
        parts += [np.ascontiguousarray(q, np.int8).view(np.uint8).reshape(-1), np.ascontiguousarray(s, np.float32).view(np.uint8).reshape(-1)]
    buf = np.concatenate(parts)
    assert sha256(buf) == want["buffer"], "the input is not the reference quantiser's buffer"
    po = C.c_void_p(buf.ctypes.data)
    to = ours.parse_quantized_tensors(C.byref(po), n_t, size_each, gs)
    assert po.value == buf.ctypes.data + buf.size                                # the cursor advances past the n tensors
    ao = np.frombuffer(C.string_at(to, n_t * 16), np.uint64)                     # Typed_Tensor = union of {q, s} pointers (16 bytes)
    assert [int(a) - buf.ctypes.data for a in ao] == want["offsets"], "parse_quantized_tensors"
    for i in range(n_t):
        q = Q80(int(ao[2 * i]), int(ao[2 * i + 1]))
        yo = np.zeros(size_each, np.float32)
        ours.dequantize(C.byref(q), yo.ctypes.data_as(f32p), size_each, gs)
        assert sha256(yo) == want["dequantize"][i], f"dequantize tensor {i}"
        assert np.abs(yo - x[i]).max() < np.abs(x[i]).max() / 100.0              # and it is a dequantisation of what went in
