"""CPU: fine-tuning with frozen batch-norm statistics -- the staging entry point of the frozen forward is exported and
reports errors through the C ABI without a GPU; the TrainConfig switches default to the reference's behaviour."""
import dataclasses

from argus_b200 import _lib


def test_stage_input_frozen_exported():
    lib = _lib.load()
    assert "argus_model_stage_input_frozen_u8" in _lib.declared_symbols()
    assert hasattr(lib, "argus_model_stage_input_frozen_u8")


def test_stage_input_frozen_null_model():
    lib = _lib.load()
    status = lib.argus_model_stage_input_frozen_u8(None, None, None, None, None, 1, 64, 64, 0, None)
    assert status != 0
    assert b"null model" in lib.argus_last_error_string()


def test_train_config_defaults():
    from argus_b200.train import TrainConfig

    fields = {f.name: f.default for f in dataclasses.fields(TrainConfig)}
    assert fields["freeze_bn"] is False
    assert fields["init_model_path"] is None


def test_engine_default_is_training_mode_batch_norm():
    import inspect

    from argus_b200.engine import TrainEngine

    assert inspect.signature(TrainEngine).parameters["frozen_bn"].default is False
