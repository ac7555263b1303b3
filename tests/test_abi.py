"""CPU tests of the drop-in boundary: the shared library loads without a GPU and exports exactly the
symbols include/twb200.h declares; the ctypes table mirrors the header; argument errors are reported
through the status / tw_last_error() convention without launching anything."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from turbo_whisper_workspace_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.load()


def _header_functions():
    text = open(os.path.join(ROOT, "include", "twb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(tw_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported(lib):
    names = _header_functions()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/twb200.h but not exported by libtwb200.so"


def test_ctypes_table_mirrors_header():
    from turbo_whisper_workspace_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _header_functions()


def test_struct_layouts_match_header(tmp_path):
    """sizeof and the offsetof of every field of every struct of the public header, as gcc lays it out in plain C99,
    equal the ctypes mirror's."""
    import subprocess
    from turbo_whisper_workspace_b200 import _lib
    structs = {"tw_gemm_args": _lib.GemmArgs, "tw_skinny_args": _lib.SkinnyArgs, "tw_grammar": _lib.Grammar,
               "tw_row_state": _lib.RowState, "tw_beam_config": _lib.BeamConfig, "tw_beam_state": _lib.BeamState,
               "tw_flac_info": _lib.FlacInfo}
    src = tmp_path / "sizes.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "twb200.h"\nint main(void) {\n' +
                   "".join(f'  printf("{n} %zu\\n", sizeof({n}));\n' for n in structs) +
                   "".join(f'  printf("{n}.{f} %zu\\n", offsetof({n}, {f}));\n'
                           for n, cls in structs.items() for f, _ in cls._fields_) + "  return 0;\n}\n")
    exe = tmp_path / "sizes"
    subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for name, cls in structs.items():
        assert int(out[name]) == C.sizeof(cls), f"{name}: header {out[name]} bytes, ctypes {C.sizeof(cls)}"
        for f, _ in cls._fields_:
            off = getattr(cls, f).offset
            assert int(out[f"{name}.{f}"]) == off, f"{name}.{f}: header offset {out[f'{name}.{f}']}, ctypes {off}"
    assert C.sizeof(_lib.GemmArgs) == 144 and C.sizeof(_lib.SkinnyArgs) == 120 and C.sizeof(_lib.Grammar) == 36
    assert C.sizeof(_lib.RowState) == 32


def test_error_convention_without_gpu(lib):
    assert lib.tw_abi_version() == 1
    rc = lib.tw_layernorm(None, None, None, None, 4, 1280, 1e-5, None)
    assert rc != 0 and b"null" in lib.tw_last_error()
    rc = lib.tw_gemm_bf16(None, None)
    assert rc != 0 and b"tw_gemm_bf16" in lib.tw_last_error()
    assert lib.tw_logmel_tables_bytes() > 0 and lib.tw_logmel_scratch_bytes(2) > 0
    assert lib.tw_dec_lmhead_parts(51866) % 8 == 0


def test_product_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    import helpers
    from turbo_whisper_workspace_b200 import _lib
    from turbo_whisper_workspace_b200.config import WhisperDims
    from turbo_whisper_workspace_b200.engine import WhisperEngine
    with pytest.raises(_lib.TwError):
        WhisperEngine(WhisperDims(**helpers.TINY), {}, device="cuda:0", max_batch=1)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "turbo-whisper-workspace_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), fn


def test_header_is_plain_c():
    """The boundary is a C ABI: include/twb200.h must compile as C99 (no C++-only constructs, no torch types)."""
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    hdr = os.path.join(ROOT, "include", "twb200.h")
    r = subprocess.run([gcc, "-fsyntax-only", "-x", "c", "-std=c99", "-Wall", "-Werror", hdr], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    text = open(hdr).read()
    assert "torch" not in re.sub(r"/\*.*?\*/", "", text, flags=re.S).lower()
