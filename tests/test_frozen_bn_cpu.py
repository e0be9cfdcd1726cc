"""CPU: the frozen-statistics entry points are exported and report errors through the C ABI without a GPU."""
from argus_b200 import _lib


def test_frozen_symbols_exported():
    lib = _lib.load()
    for name in ("argus_model_forward_frozen", "argus_bn_frozen_finish", "argus_relu_bits_mask_colsum",
                 "argus_stem_unpool_relu", "argus_pack_weight_scaled"):
        assert name in _lib.declared_symbols()
        assert hasattr(lib, name)


def test_model_forward_frozen_null_model():
    lib = _lib.load()
    status = lib.argus_model_forward_frozen(None, None, 0, 1, 64, 64, None, None)
    assert status != 0
    assert b"null model" in lib.argus_last_error_string()
