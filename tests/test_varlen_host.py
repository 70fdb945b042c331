"""Ragged generator batches without a GPU: argument checks of mg_gen_forward_varlen / mg_gen_engine_forward_varlen (they
run before any CUDA call) and the Python layers' refusals."""
import ctypes
import warnings

import numpy as np
import pytest
import torch

from melgan_multi_b200 import engine

warnings.filterwarnings("ignore")

MG_ERR_INVALID_ARGUMENT = -1


def _call_varlen(B, T, lengths):
    L = engine.lib()
    dummy = ctypes.c_void_p(256)  # never dereferenced: the arguments are rejected first
    return L.mg_gen_forward_varlen(dummy, dummy, dummy, B, T, lengths, dummy, 1 << 40, None)


def _ints(*v):
    return (ctypes.c_int * len(v))(*v)


def test_varlen_exports_and_abi_version():
    L = engine.lib()
    assert hasattr(L, "mg_gen_forward_varlen") and hasattr(L, "mg_gen_engine_forward_varlen")
    assert L.mg_abi_version() == 2  # additive entry points


def test_varlen_rejects_null_lengths():
    assert _call_varlen(2, 8, None) == MG_ERR_INVALID_ARGUMENT
    assert "lengths" in engine.lib().mg_last_error_string().decode()


@pytest.mark.parametrize("bad, index", [((0, 8, 8), 0), ((8, 9, 8), 1), ((8, 8, -3), 2)])
def test_varlen_rejects_lengths_out_of_range_and_names_the_index(bad, index):
    assert _call_varlen(3, 8, _ints(*bad)) == MG_ERR_INVALID_ARGUMENT
    msg = engine.lib().mg_last_error_string().decode()
    assert "lengths[%d]" % index in msg, msg


def test_varlen_rejects_bad_shape_before_lengths():
    assert _call_varlen(0, 8, _ints(1)) == MG_ERR_INVALID_ARGUMENT
    assert _call_varlen(1, 0, _ints(1)) == MG_ERR_INVALID_ARGUMENT


def test_engine_varlen_rejects_bad_arguments():
    L = engine.lib()
    dummy = ctypes.c_void_p(256)
    assert L.mg_gen_engine_forward_varlen(None, dummy, dummy, 1, 4, _ints(4)) == MG_ERR_INVALID_ARGUMENT
    assert L.mg_gen_engine_forward_varlen(dummy, dummy, dummy, 2, 4, _ints(4, 5)) == MG_ERR_INVALID_ARGUMENT
    assert "lengths[1]" in L.mg_last_error_string().decode()
    assert L.mg_gen_engine_forward_varlen(dummy, dummy, dummy, 2, 4, None) == MG_ERR_INVALID_ARGUMENT


def test_lengths_array_accepts_list_tuple_tensor_and_checks_count():
    assert list(engine.lengths_array([3, 1, 2], 3)) == [3, 1, 2]
    assert list(engine.lengths_array((3, 1), 2)) == [3, 1]
    assert list(engine.lengths_array(torch.tensor([5, 4], dtype=torch.int64), 2)) == [5, 4]
    assert list(engine.lengths_array(np.array([7], np.int32), 1)) == [7]
    with pytest.raises(engine.EngineError):
        engine.lengths_array([1, 2], 3)
    with pytest.raises(engine.EngineError):
        engine.lengths_array(torch.tensor([1.0, 2.0]), 2)
    with pytest.raises(engine.EngineError):
        engine.lengths_array([1.5, 2.0], 2)


def test_generator_module_refuses_cpu_input_with_lengths():
    from melgan_multi_b200 import models
    g = models.Generator().eval()
    with torch.no_grad(), pytest.raises(engine.EngineError):
        g(torch.zeros(2, 80, 4), lengths=[4, 2])
