"""The C-ABI library loads on a CPU box and exports every entry point that include/agcn_b200.h declares
(no compute calls here -- those need a GPU)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "agcn_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(agcn_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound():
    from fusion_gcn_b200 import build, capi
    build.build()
    names = declared_symbols()
    assert len(names) >= 15
    handle = ctypes.CDLL(capi.LIB_PATH)
    for n in names:
        assert hasattr(handle, n), f"{n} declared in agcn_b200.h but not exported"
    assert sorted(capi.SIGNATURES) == names, "fusion_gcn_b200/capi.py must bind exactly the declared entry points"
    lib = capi.lib()
    assert lib.agcn_version() >= 100
    assert lib.agcn_bn_workspace_bytes(64) > 0
    assert lib.agcn_conv_wgrad_workspace_bytes(2, 8, 8, 25, 64, 64, 9) > 0
    assert lib.agcn_conv_fwd_workspace_bytes(64, 64, 9, capi.PREC_FP32) == 2 * 64 * 64 * 9 * 4
    assert lib.agcn_conv_fwd_workspace_bytes(64, 64, 9, capi.PREC_TF32) == 0


def test_argument_validation_without_gpu():
    """Shape / null checks run before any CUDA call, so the error paths are testable on a CPU box."""
    from fusion_gcn_b200 import capi
    lib = capi.lib()
    rc = lib.agcn_conv_fwd(None, None, None, None, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, None, 0, None)
    assert rc == 6 and b"null" in lib.agcn_last_error_string()
    rc = lib.agcn_joint_mix(1, 1, 1, 1, 4, 25, 8, 24, 8, 7, 0, 0, None, 0, None)       # mix mode 7 does not exist
    assert rc == 2 and b"unknown mode" in lib.agcn_last_error_string()
    rc = lib.agcn_joint_gram(1, 1, 1, 1, 4, 40, 8, 8, 3, 0, 0, 0, 0, 8, 2, 0, None)    # V = 40 > 32 runs as ONE chunk
    assert rc == 2 and b"one chunk" in lib.agcn_last_error_string()
    rc = lib.agcn_conv_fwd(1, 1, None, 1, 0, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, None, 0, None)
    assert rc == 1
    with pytest.raises(RuntimeError, match="status 1"):
        capi.check(rc, "agcn_conv_fwd")


@pytest.mark.parametrize("operands,status,message", [
    (dict(frozen=1, pool_rows=4, mask_bits=1), 2, b"frozen statistics"),
    (dict(frozen=1, phase=1), 2, b"frozen statistics"),
    (dict(frozen=1, phase=2), 2, b"frozen statistics"),
    (dict(phase=3), 2, b"phase 3"),
    (dict(phase=-1), 2, b"phase -1"),
    (dict(mask_out=1, mask_bits=1), 2, b"mask_out and mask_bits"),
    (dict(dy=None, dy_split=1), 6, b"dy_split needs dy"),
])
def test_batchnorm_backward_rejects_contradictory_operands(operands, status, message):
    """agcn_bn_bwd refuses operand combinations that no form of the backward covers before it launches anything (the workspace is
    NULL, so a call that got past these checks would stop at the null-pointer check instead of reaching the device)."""
    from fusion_gcn_b200 import capi
    lib = capi.lib()
    a = dict(mask_out=None, mask_bits=None, dy=1, dy_split=None, frozen=0, pool_rows=0, phase=0)
    a.update(operands)
    rc = lib.agcn_bn_bwd(1, a["mask_out"], a["mask_bits"], 1, 1, 1, 1, a["dy"], a["dy_split"], 1, 1, None, 0, a["frozen"],
                         1, 64, 0, 64, a["pool_rows"], a["phase"], 1, 64.0, None, 0, None)
    assert rc == status and message in lib.agcn_last_error_string()
