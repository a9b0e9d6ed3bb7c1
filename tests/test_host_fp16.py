"""The float16 precision on the host side: C header constant, Python dtype code, packed operand sizes (no GPU needed)."""
import os
import re

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_and_binding_define_f16():
    import xvec_b200
    with open(os.path.join(ROOT, "include", "xvec_b200.h")) as f:
        header = f.read()
    assert re.search(r"#define\s+XVEC_F16\s+2\b", header)
    assert xvec_b200._lib.F16 == 2
    assert xvec_b200._lib.dtype_code(torch.float16) == 2
    assert xvec_b200.xvector.PRECISIONS["fp16"] == torch.float16


def test_packed_k_of_f16_equals_bf16():
    import xvec_b200
    lib = xvec_b200._lib.load()
    F16, BF16 = xvec_b200._lib.F16, xvec_b200._lib.BF16
    assert lib.xvec_packed_k(512, 3, F16) == 1536
    for cin, taps in ((24, 5), (3000, 1), (40, 3), (120, 1)):
        assert lib.xvec_packed_k(cin, taps, F16) == lib.xvec_packed_k(cin, taps, BF16)


def test_fp16_range_guard_on_host_tensors():
    """The preparation-time guard itself needs no device: it refuses weights float16 cannot hold."""
    import pytest
    import xvec_b200
    check_fp16_range = xvec_b200.tdnn_layer.check_fp16_range
    check_fp16_range("ok", torch.full((4, 4), 65000.0), torch.zeros(4))
    with pytest.raises(ValueError, match="tf32"):
        check_fp16_range("segment_layer6", torch.full((4, 4), 65504.0))
    with pytest.raises(ValueError, match="bias"):
        check_fp16_range("segment_layer6", torch.zeros(4, 4), torch.tensor([0.0, -1e6]))
