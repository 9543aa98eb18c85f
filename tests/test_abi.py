"""CPU-only: the C-ABI library loads, exports every symbol include/climsr_b200.h declares, and fails loudly without a GPU."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "climsr_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(csr_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_expected_entry_points():
    syms = _declared_symbols()
    for must in ("csr_plan_forward", "csr_generator_forward", "csr_pack_weights", "csr_conv2d_nhwc", "csr_masked_metrics"):
        assert must in syms


def test_library_exports_every_declared_symbol():
    from climsr_b200 import _lib
    raw = C.CDLL(_lib.LIB_PATH)
    for s in _declared_symbols():
        assert hasattr(raw, s), f"{s} declared in include/climsr_b200.h but not exported"
    assert set(_declared_symbols()) == set(_lib.EXPORTS)
    assert _lib.lib.csr_abi_version() == 2


def test_layer_table_matches_reference_state_dict_order():
    from climsr_b200._lib import NetDesc, lib
    from oracle import synth
    for in_ch, nb, gc in ((4, 11, 16), (3, 23, 32), (2, 1, 16)):
        d = NetDesc(in_ch, 1, 64, nb, gc, 4)
        specs = synth.conv_specs(in_ch, 1, 64, nb, gc)
        assert lib.csr_num_layers(C.byref(d)) == len(specs)
        shape = (C.c_int32 * 4)()
        name = C.create_string_buffer(128)
        for i, (nm, co, ci, kh, kw) in enumerate(specs):
            assert lib.csr_layer_shape(C.byref(d), i, C.byref(shape), name, 128) == 0
            assert name.value.decode() == nm and tuple(shape) == (co, ci, kh, kw)


def test_argument_validation_without_gpu():
    from climsr_b200._lib import NetDesc, lib
    bad = NetDesc(4, 3, 64, 11, 16, 4)          # out_channels != 1
    assert lib.csr_num_layers(C.byref(bad)) == -2
    assert b"out_channels" in lib.csr_last_error()
    assert lib.csr_packed_weight_bytes(C.byref(bad)) == 0
    good = NetDesc(4, 1, 64, 11, 16, 4)
    assert lib.csr_packed_weight_bytes(C.byref(good)) > 4_000_000     # ~4.28 M params as bf16 + padding
    assert lib.csr_workspace_bytes(C.byref(good), 0, 8, 8) == 0
    ws = lib.csr_workspace_bytes(C.byref(good), 2, 16, 16)
    assert ws > 2 * 64 * 64 * 64 * 2 * 3
    assert lib.csr_set_option(999, 0) == -1
    assert lib.csr_plan_create(C.byref(good), 1, 8, 8, None, 0, None) == -1


def test_retired_option_keys_are_rejected():
    """Keys of the removed kernel variants and debug settings are unknown keys; 26 and 35 take only 0 / 1."""
    from climsr_b200._lib import lib
    for key in (2, 3, 5, 6, 7, 8, 9, 13, 14, 16, 20, 21, 22, 23, 24, 28, 29, 32):
        assert lib.csr_set_option(key, 0) == -1 and lib.csr_set_option(key, 1) == -1, key
    for key in (26, 35):
        assert lib.csr_set_option(key, 2) == -1 and lib.csr_set_option(key, -1) == -1, key
        assert lib.csr_set_option(key, 1) == 0, key                    # the default
    assert lib.csr_has_experiments() == 0


def test_no_cpu_fallback():
    import torch
    from climsr_b200 import CsrError
    from climsr_b200.models import ESRGANGenerator
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from climsr_b200._lib import lib
    assert lib.csr_device_check() != 0
    net = ESRGANGenerator(2, 1, 64, 1, 16).eval()
    with pytest.raises(CsrError):
        with torch.no_grad():
            net(torch.rand(1, 2, 8, 8), torch.rand(1, 1, 32, 32), torch.rand(1, 1, 32, 32))
