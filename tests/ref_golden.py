"""Stored outputs of the reference implementation's own CUDA kernels, for the comparisons in test_gpu_parity.py.

``tests/golden/ref_kernels/<case>.npz`` holds what the reference kernels computed on the seeded inputs below (written
by ``tests/golden/make_ref_kernels.py`` on a GPU).  An output of up to SAMPLE elements is stored whole; a larger one as
``<key>_shape`` and ``<key>`` = its values at ``positions(size, SAMPLE)``, sorted flat indices drawn by numpy's
RandomState(0), whose streams numpy keeps fixed across versions.  Inputs are regenerated from their seeds and checked
against a stored sample (``in_<key>``), so a change in torch's random streams shows up as an input mismatch, not as a
parity failure.
"""
import os

import numpy as np
import torch

DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels")
SAMPLE = 2048           # elements kept of an output
INPUT_SAMPLE = 256      # elements kept of an input


def randn(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).float()


# seeded inputs of each comparison (CPU tensors)
def correlation_inputs(shape):
    return randn(shape, 41), randn(shape, 42)


def correlation_grad_output(out_shape):
    return randn(out_shape, 43)


def resample_channelnorm_inputs():
    g = torch.Generator().manual_seed(44)
    img = torch.rand(2, 3, 32, 48, generator=g)
    flow = torch.randn(2, 2, 32, 48, generator=g) * 6
    go = torch.randn(2, 3, 32, 48, generator=g)
    x = torch.randn(2, 3, 32, 48, generator=g)
    gon = torch.randn(2, 1, 32, 48, generator=g)
    return img, flow, go, x, gon


def channelnorm_half_inputs(shape):
    return randn(shape, 35).half(), randn((shape[0], 1, shape[2], shape[3]), 36).half()


def case_name(op, shape):
    return "%s_%s" % (op, "x".join(str(s) for s in shape))


def _numpy(a):
    return a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)


def positions(size, n):
    return np.sort(np.random.RandomState(0).choice(size, n, replace=False))


def _stored(key, a, n):
    a = np.ascontiguousarray(_numpy(a))
    if a.size <= n:
        return {key: a}
    return {key: a.reshape(-1)[positions(a.size, n)], key + "_shape": np.array(a.shape)}


def save(case, inputs, outputs, out_dir=DIR):
    arrays = {}
    for k, v in inputs.items():
        arrays.update(_stored("in_" + k, v, INPUT_SAMPLE))
    for k, v in outputs.items():
        arrays.update(_stored(k, v, SAMPLE))
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, case + ".npz")
    np.savez_compressed(path, **arrays)
    return path


class Golden:
    def __init__(self, case):
        self.case = case
        self.z = np.load(os.path.join(DIR, case + ".npz"))

    def __getitem__(self, key):
        return self.z[key]

    def pick(self, key, a):
        """``a`` (a tensor or array shaped like the stored output ``key``) at the positions stored for ``key``."""
        a = _numpy(a)
        sampled = key + "_shape" in self.z
        shape = tuple(self.z[key + "_shape"]) if sampled else self.z[key].shape
        assert a.shape == shape, "%s/%s: shape %s vs %s" % (self.case, key, a.shape, shape)
        return a.reshape(-1)[positions(a.size, self.z[key].size)] if sampled else a

    def check_inputs(self, **inputs):
        for k, v in inputs.items():
            assert np.array_equal(self.pick("in_" + k, v), self.z["in_" + k]), \
                "%s: input %s is not the one the stored outputs were computed from" % (self.case, k)
