"""CPU: the C-ABI shared library loads without a GPU and exports every symbol include/otter_b200.h declares;
argument validation returns error codes (never throws / exits); no compute is launched here."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "otter_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(otb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from otter_b200 import _lib
    lib = _lib.load()
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/otter_b200.h but not exported"
    assert sorted(_lib.SIGNATURES) == syms, "ctypes SIGNATURES table out of sync with the header"
    assert lib.otb_compiled_arch() == 100 and lib.otb_version() >= 1


def test_struct_layouts_match_header():
    from otter_b200 import _lib
    lib = _lib.load()
    # the C compiler's layout (otb_abi_sizeof) vs the ctypes mirror, and vs the header's field lists
    assert lib.otb_abi_sizeof(0) == C.sizeof(_lib.GemmEpilogue) == 6 * 8 + 4 * 8 + 6 * 4
    assert lib.otb_abi_sizeof(1) == C.sizeof(_lib.AttnDesc) == 6 * 8 + 4 * 8 + 17 * 4 + 4 + 2 * 4
    assert lib.otb_abi_sizeof(2) == C.sizeof(_lib.AttnGrads) == 5 * 8 + 4 * 8 + 8 * 4


def test_invalid_arguments_return_error_codes():
    from otter_b200 import _lib
    lib = _lib.load()
    e = _lib.GemmEpilogue()
    rc = lib.otb_gemm_bf16(None, 0, 0, None, 0, 0, 0, 0, 0, C.byref(e), None)
    assert rc == 1 and b"otb_gemm_bf16" in lib.otb_last_error()
    assert lib.otb_text_time(None, 0, 0, 1, None, None) == 1
    assert lib.otb_layernorm_fwd(None, 0, None, None, None, 0, None, None, 0, 0, 1e-5, None) == 1
    d = _lib.AttnDesc()
    assert lib.otb_attn_fwd(C.byref(d), None) == 1
    assert lib.otb_ln_chunks(2048, 4096) >= 1 and lib.otb_dot_blocks() > 0
    assert lib.otb_launch_count() == 0      # nothing was launched by the calls above


@pytest.mark.parametrize("operand", ["A", "B", "out", "bias", "residual", "aux_in", "aux_out"])
def test_gemm_rejects_misaligned_operands(operand):
    """Every pointer the GEMM reads with TMA or 16-byte vector loads / stores must be 16-byte aligned: a misaligned
    one is OTB_ERR_INVALID naming the operand.  The pointers are fake integers, and every call also carries an invalid
    activation code that is checked after the alignment, so none of these calls can reach a launch."""
    from otter_b200 import _lib
    lib = _lib.load()
    n0 = lib.otb_launch_count()
    base = {name: 0x10000 * (i + 1) for i, name in enumerate(("A", "B", "out", "bias", "residual", "aux_in", "aux_out"))}
    for off in (2, 4, 8):
        ptr = dict(base)
        ptr[operand] += off
        e = _lib.GemmEpilogue()
        e.out, e.bias, e.residual, e.aux_in, e.aux_out = (ptr[k] for k in ("out", "bias", "residual", "aux_in", "aux_out"))
        e.ld_out = e.ld_res = e.ld_aux_in = e.ld_aux_out = 64
        e.alpha = 1.0
        e.act = 7                                    # invalid: the backstop if the alignment check were missing
        rc = lib.otb_gemm_bf16(ptr["A"], 0, 64, ptr["B"], 0, 64, 64, 64, 64, C.byref(e), None)
        assert rc == 1, (operand, off, rc)
        assert lib.otb_last_error().decode() == f"otb_gemm_bf16: {operand} is not 16-byte aligned", (operand, off)
    # the same call with every pointer aligned fails on the activation code, which proves the backstop is live
    e = _lib.GemmEpilogue()
    e.out, e.bias, e.residual, e.aux_in, e.aux_out = (base[k] for k in ("out", "bias", "residual", "aux_in", "aux_out"))
    e.ld_out = e.ld_res = e.ld_aux_in = e.ld_aux_out = 64
    e.alpha, e.act = 1.0, 7
    assert lib.otb_gemm_bf16(base["A"], 0, 64, base["B"], 0, 64, 64, 64, 64, C.byref(e), None) == 1
    assert b"bad act" in lib.otb_last_error()
    assert lib.otb_launch_count() == n0


def test_ops_reject_cpu_tensors_loudly():
    import torch
    from otter_b200 import _lib
    from otter_b200 import functional as F
    with pytest.raises(_lib.OtbError, match="CUDA tensor"):
        F.linear_fwd(torch.zeros(8, 8, dtype=torch.bfloat16), torch.zeros(8, 8, dtype=torch.bfloat16))


def test_sass_is_blackwell_native():
    """The built library must contain 5th-gen tensor-core / TMA / TMEM machine code (B200_PROFILING.md:
    tcgen05.mma -> UTC*MMA, TMA -> UTMALDG, tcgen05.ld -> LDTM) and no legacy mma.sync path (HMMA)."""
    import shutil
    import subprocess
    from otter_b200 import _lib
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    assert "sm_100a" in sass or "SM100" in sass.upper()
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM", "UTCBAR", "SYNCS"):
        assert mnemonic in sass, f"{mnemonic} missing from the SASS"
    assert "UTCHMMA.2CTA" in sass or "2CTA" in sass, "cta_group::2 MMA missing"
    assert "HMMA." not in sass.replace("UTCHMMA", ""), "legacy mma.sync (HMMA) found"


def test_integration_guide_names_every_entry_point():
    """INTEGRATION.md's table (entry point -> reference file:line it replaces) covers the whole header."""
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "otter_b200.h")).read()
    doc = open(os.path.join(root, "INTEGRATION.md")).read()
    syms = sorted(set(re.findall(r"\b(otb_[a-z0-9_]+)\s*\(", hdr)))
    assert len(syms) >= 50
    assert [s for s in syms if s not in doc] == []
