"""CPU: the input-gradient entry points are exported and report errors through the C ABI without a GPU."""
from argus_b200 import _lib


def test_input_grad_symbols_exported():
    lib = _lib.load()
    for name in ("argus_stem_dgrad", "argus_model_input_grad"):
        assert name in _lib.declared_symbols()
        assert hasattr(lib, name)


def test_model_input_grad_null_model():
    lib = _lib.load()
    status = lib.argus_model_input_grad(None, None, None)
    assert status != 0
    assert b"null model" in lib.argus_last_error_string()

