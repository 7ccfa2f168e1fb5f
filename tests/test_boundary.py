"""CPU tests for the drop-in boundary: ABI layout of include/nano_infer_abi.h == the reference's headers,
libnano_infer_b200.so exports the reference API, and the reference's main_cli.c links against it unchanged."""
import json
import os
import re
import subprocess
import tempfile

import pytest

from conftest import GOLDEN, ROOT
from nano_b200 import build as nb_build
from oracle import bindings as ob


def my_layout():
    with tempfile.TemporaryDirectory() as td:
        exe = os.path.join(td, "abi_probe")
        subprocess.run(["gcc", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "abi_probe.c"), "-o", exe], check=True)
        return [int(v) for v in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]


def test_abi_layout_matches_committed_reference_layout():
    """abi_layout.json: the sizes and offsets read from the reference's own headers (oracle/ref_harness.c:orh_abi_layout)."""
    want = json.load(open(os.path.join(GOLDEN, "abi_layout.json")))
    assert len(want) > 60
    assert my_layout() == want


def exported_api():
    hdr = open(os.path.join(ROOT, "include", "nano_infer_abi.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    exported = hdr.split("imported from the reference")[0] if "imported from the reference" in hdr else hdr
    # the "imported" block was stripped together with its comment; cut at the first imported prototype instead
    exported = exported.split("void *platform_calloc")[0]
    return sorted(set(re.findall(r"\b([a-z_0-9]+)\s*\(", exported)) - {"sizeof", "observation", "on_prefilling", "on_decoding", "on_finished", "int32_t", "void"})


def test_shim_exports_reference_api():
    out = subprocess.run(["nm", "-D", "--defined-only", nb_build.SHIM_SO], capture_output=True, text=True, check=True).stdout
    have = set(re.findall(r" T (\w+)", out))
    api = exported_api()
    for must in ("llm_context_init", "llm_context_init_from_buffer", "llm_context_free", "generate_next_token", "llm_session_init",
                 "llm_session_step", "llm_session_free", "generate_sync", "seq2seq", "load_llm", "load_llm_from_buffer",
                 "build_sampler", "free_llm", "free_sampler", "load_lora", "load_lora_from_buffer", "free_lora", "llm_forward",
                 "quantize", "dequantize", "parse_quantized_tensors"):
        assert must in api, must
    missing = [f for f in api if f not in have]
    assert not missing, missing
    und = subprocess.run(["nm", "-D", "--undefined-only", nb_build.SHIM_SO], capture_output=True, text=True).stdout
    for imp in ("platform_calloc", "random_f32", "encode_nano", "decode_bpe", "build_bpe_tokenizer", "new_trie"):
        assert re.search(rf" U {imp}\b", und), f"{imp} should be imported from the reference's unchanged objects"
    assert "nb200_engine_create" in und and "oracle" not in subprocess.run(["ldd", nb_build.SHIM_SO], capture_output=True, text=True).stdout


@pytest.mark.skipif(not os.path.exists(ob.NANO_CLI_HOST), reason="needs the reference's main_cli.c objects (oracle/Makefile)")
def test_reference_nano_cli_links_unchanged():
    exe = ob.link_nano_cli()
    und = subprocess.run(["nm", "-D", "--undefined-only", exe], capture_output=True, text=True, check=True).stdout
    assert " U llm_context_init" in und and " U generate_sync" in und
    ldd = subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
    assert "libnano_infer_b200.so" in ldd and "libnano_b200.so" in ldd
