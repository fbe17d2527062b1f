# -*- coding: utf-8 -*-
"""Every kernel instance of the reference's own suite (tests/test_kernels.py `kernels_to_test` + `test_stationary`):
(CPU) our oracle == the reference's compiled kernel_interface, bit for bit, values and hyper-gradients (what it returned
      is kept in tests/golden/reference_kernel_interface.npz);
(GPU) the CUDA build == the oracle, and the reference's finite-difference gradient check passes on the device path."""
import numpy as np
import pytest

from conftest import reference_kernel_list
from test_oracle_kernels import assert_equals_reference_binary

KERNELS = reference_kernel_list()
IDS = ["{0:02d}-{1}".format(i, type(k).__name__) for i, k in enumerate(KERNELS)]


def kernel_list_input(kernel):
    np.random.seed(123)
    return np.random.randn(20, kernel.ndim)


@pytest.mark.parametrize("kid,kernel", list(zip(IDS, KERNELS)), ids=IDS)
def test_oracle_equals_reference_binary(oracle, kid, kernel):
    from george_b200._spec import flatten
    t1 = kernel_list_input(kernel)
    spec = flatten(kernel)
    outs = [oracle.value_symmetric(spec, t1), oracle.value_general(spec, t1, t1[:1])]
    if kernel.full_size:
        which = np.ones(kernel.full_size, dtype=np.uint32)
        outs.append(oracle.gradient_general(spec, which, t1, t1[:3]))
    # input-coordinate gradients (kernel_interface.cpp:127-157)
    outs += [oracle.x_gradient_general(spec, 1, t1, t1[:3]), oracle.x_gradient_general(spec, 2, t1[:3], t1)]
    assert_equals_reference_binary("list", kid, outs)


def test_stationary_constructor_errors():
    from george_b200 import kernels
    with pytest.raises(ValueError):
        kernels.ExpSquaredKernel(metric=[1.0, 0.1, 10.0, 500], ndim=3)  # tests/test_kernels.py:117-118


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_device_values_gradients_and_fd(gpu, oracle, kernel):
    """reference tests/test_kernels.py:65-70 (test_kernel): FD check of the hyper-gradient, here on the CUDA path."""
    from george_b200._spec import flatten
    np.random.seed(123)
    t1 = np.random.randn(20, kernel.ndim)
    spec = flatten(kernel)
    np.testing.assert_allclose(kernel.get_value(t1), oracle.value_symmetric(spec, t1), rtol=1e-11, atol=1e-13)
    np.testing.assert_allclose(kernel.get_value(t1, t1[:1]), oracle.value_general(spec, t1, t1[:1]), rtol=1e-11, atol=1e-13)
    if kernel.full_size:
        which = np.ones(kernel.full_size, dtype=np.uint32)
        np.testing.assert_allclose(kernel.get_gradient(t1, t1[:3], include_frozen=True),
                                   oracle.gradient_general(spec, which, t1, t1[:3]), rtol=1e-10, atol=1e-12)
    if len(kernel):
        kernel.test_gradient(t1, eps=1.32e-6)
        kernel.test_gradient(t1, t1[:1], eps=1.32e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS, ids=IDS)
def test_device_x_gradients(gpu, oracle, kernel):
    """reference tests/test_kernels.py:73-80 (test_x_gradient_kernel) on the CUDA path, plus device == oracle."""
    from george_b200._spec import flatten
    np.random.seed(123)
    t1 = np.random.randn(20, kernel.ndim)
    spec = flatten(kernel)
    np.testing.assert_allclose(kernel.get_x1_gradient(t1, t1[:3]), oracle.x_gradient_general(spec, 1, t1, t1[:3]),
                               rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(kernel.get_x2_gradient(t1[:3], t1), oracle.x_gradient_general(spec, 2, t1[:3], t1),
                               rtol=1e-10, atol=1e-12)
    kernel.test_x1_gradient(t1, eps=1.32e-6)
    kernel.test_x1_gradient(t1, np.array(t1[:1]), eps=1.32e-6)
    kernel.test_x2_gradient(t1, eps=1.32e-6)
    kernel.test_x2_gradient(np.array(t1[:1]), t1, eps=1.32e-6)
