"""The C-ABI library loads and exports every symbol include/dcscn_b200.h declares (no compute without a GPU),
and construction fails loudly (never silently falls back) when no B200 is present.  CPU only."""
import ctypes
import os
import re

import pytest

from helper import engine as E
from conftest import ROOT


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "dcscn_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dcscn_[a-z_0-9]+)\s*\(", text)))


def test_header_symbols_exported():
    syms = declared_symbols()
    assert "dcscn_forward" in syms and "dcscn_create" in syms and len(syms) >= 12
    lib = E.load_library()
    for s in syms:
        assert hasattr(lib, s), "libdcscn_b200.so does not export %s" % s
    assert sorted(E.EXPORTED_SYMBOLS) == syms


def test_config_struct_matches_header():
    text = open(os.path.join(ROOT, "include", "dcscn_b200.h")).read()
    body = text[text.index("typedef struct dcscn_config {"):text.index("} dcscn_config;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for line in body.splitlines()[1:]:
        m = re.match(r"\s*(int32_t|float)\s+([^;]+);", line)
        if m:
            fields += [(n.strip(), m.group(1)) for n in m.group(2).split(",")]
    py = [(n, "int32_t" if t is ctypes.c_int32 else "float") for n, t in E.DcscnConfig._fields_]
    assert fields == py
    assert ctypes.sizeof(E.DcscnConfig) == 4 * len(py)


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(E.EngineError) as ei:
        E.Engine(E.make_config())
    assert "no CPU path" in str(ei.value) or "CUDA" in str(ei.value)


def test_missing_library_is_loud(tmp_path):
    with pytest.raises(E.EngineError):
        E.load_library(str(tmp_path / "nope.so"))


def test_every_option_key_is_documented_in_the_header():
    """dcscn_set_option's keys live in csrc/engine.cu; the header is the only documentation a binding author reads, so a
    key the engine accepts but the header does not mention (or the other way round) is a documentation bug."""
    src = open(os.path.join(ROOT, "dcscn-super-resolution_b200", "csrc", "engine.cu")).read()
    body = src[src.index("int dcscn_set_option("):]
    body = body[:body.index("\nint dcscn_get_timings")] if "\nint dcscn_get_timings" in body else body[:6000]
    keys = set(re.findall(r'k == "([a-z_0-9]+)"', body))
    assert {"graph", "store_mode", "wide_tiles", "seg_chunks", "conv_impl", "timing"} <= keys
    header = open(os.path.join(ROOT, "include", "dcscn_b200.h")).read()
    doc = header[header.index("int dcscn_set_option") - 6000:header.index("int dcscn_set_option")]
    documented = set(re.findall(r'"([a-z_0-9]+)"', doc))
    assert keys <= documented, sorted(keys - documented)
