"""GPU: the same save_state / load_state round trip and reference interop as tests/test_state_mock.py, on the real device
layer (KV cache in HBM, the persistent token kernel writing it)."""
import pytest

from tests.test_state_mock import check_state_interop

pytestmark = pytest.mark.gpu


def test_state_round_trip_and_interop_with_reference_on_gpu(tmp_path):
    from fastllama_b200.build import lib_path

    check_state_interop(tmp_path, lib_path("pyfastllama.so"))
