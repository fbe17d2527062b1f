# -*- coding: utf-8 -*-
"""
Generates tests/golden/reference_kernel_interface.npz: what the reference's own compiled kernel_interface.cpp
(oracle/_ref, `make -C oracle ref`) returns for the kernels of tests/conftest.py, driven with OUR kernel objects, on
the inputs of tests/test_oracle_kernels.py and tests/test_reference_kernel_list.py.  Those tests compare the CPU oracle
with it bit for bit, so they run on machines without the reference sources.

Per kernel the file keeps a SHA-256 digest of every output (tests/test_oracle_kernels.py:reference_digest) and a fixed,
seeded sample of SAMPLE values of the outputs laid end to end; the full arrays would not fit a small fixture.

Run from the repo root:   python tests/golden/make_golden_kernel_interface.py     (needs `make -C oracle ref`)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from conftest import make_kernels, reference_kernel_list  # noqa: E402
from test_oracle_kernels import GOLDEN_KI, kernel_zoo_inputs, reference_digest  # noqa: E402
from test_reference_kernel_list import IDS, kernel_list_input  # noqa: E402

SAMPLE = 32


def main():
    import oracle
    ref = oracle.reference_kernel_interface()
    assert ref is not None, "run `make -C oracle ref` first"
    rng = np.random.default_rng(0)
    out = {}

    def add(group, names, outputs):
        idx, val, sha = [], [], []
        for outs in outputs:
            flat = np.concatenate([np.ravel(a) for a in outs])
            assert not np.isnan(flat).any()  # so that equal digests mean np.array_equal
            i = np.sort(rng.choice(flat.size, SAMPLE, replace=False))
            idx.append(i)
            val.append(flat[i])
            sha.append(reference_digest(outs))
        out[group + "_names"] = np.array(names)
        out[group + "_idx"] = np.array(idx, dtype=np.int32)
        out[group + "_val"] = np.array(val)
        out[group + "_sha256"] = np.array(sha)

    # tests/test_oracle_kernels.py::test_oracle_equals_reference_binary
    names, outputs = [], []
    for name, kernel in make_kernels():
        x1, x2 = kernel_zoo_inputs(kernel)
        r = ref.KernelInterface(kernel)
        outs = [r.value_general(x1, x2), r.value_symmetric(x1), r.value_diagonal(x1[:19], x2)]
        if kernel.full_size:
            outs.append(r.gradient_general(np.ones(kernel.full_size, dtype=np.uint32), x1, x2))
        names.append(name)
        outputs.append(outs)
    add("zoo", names, outputs)

    # tests/test_reference_kernel_list.py::test_oracle_equals_reference_binary
    outputs = []
    for kernel in reference_kernel_list():
        t1 = kernel_list_input(kernel)
        r = ref.KernelInterface(kernel)
        outs = [r.value_symmetric(t1), r.value_general(t1, t1[:1])]
        if kernel.full_size:
            outs.append(r.gradient_general(np.ones(kernel.full_size, dtype=np.uint32), t1, t1[:3]))
        outs += [r.x1_gradient_general(t1, t1[:3]), r.x2_gradient_general(t1[:3], t1)]
        outputs.append(outs)
    add("list", IDS, outputs)

    np.savez_compressed(GOLDEN_KI, **out)
    print(GOLDEN_KI, os.path.getsize(GOLDEN_KI), "bytes")


if __name__ == "__main__":
    main()
