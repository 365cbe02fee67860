"""CUDA twins of the later golden cases (their oracle twins run under `-m "not gpu"`): filter_map_test,
index_test / index_with_test, zset_sum, propagate_test, window bounded_memory."""
import pytest

import filter_map_cases as fc
import golden_cases as gc
import recursion_cases as rc

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", sorted(fc.CASES))
def test_cuda_filter_map(cuda, name):
    fc.run_filter_map_case(cuda, name)


@pytest.mark.parametrize("with_closure", [False, True], ids=["index", "index_with"])
def test_cuda_index(cuda, with_closure):
    fc.run_index_test(cuda, with_closure)


def test_cuda_neg_plus_and_sum_are_zero(cuda):
    fc.run_neg_plus_zero(cuda)
    fc.run_sum_zero(cuda)


def test_cuda_propagate_test(cuda):
    rc.run_propagate_test(cuda)


@pytest.mark.parametrize("name", sorted(gc.ORACLE_ONLY_CASES))
def test_cuda_late_golden(cuda, name):
    gc.ORACLE_ONLY_CASES[name](cuda)


def test_cuda_filter_map_circuit(cuda):
    fc.run_filter_map_circuit(cuda)


def test_cuda_sum_circuit(cuda):
    fc.run_sum_circuit(cuda)


def test_cuda_input_zset(cuda):
    fc.run_input_zset_test(cuda)
