"""The public-data flavour of the field arithmetic on the GPU (k_fe_selftest ops 10..15: pub_mul, pub_sq, pub_add, pub_sub,
pub_neg, pub_pow2523 with their pending carries settled) compared bit for bit with the constant-time ops of the device
(0, 1, 2, 3, 8, 7) and with the host build of the same public functions, on the operands of test_fe_public.py that take
every rare path plus random ones."""
import numpy as np
import pytest

import test_fe_public as fp

pytestmark = pytest.mark.gpu

PAIRS = ((10, 0, 0), (11, 1, 1), (12, 2, 2), (13, 3, 3), (14, 8, 4), (15, 7, 6))    # (public op, constant-time op, host shim op)


def to_bytes(w):
    return np.ascontiguousarray(w, np.uint32).view(np.uint8).reshape(-1, 32)


def test_public_flavour_on_device(ed, tmp_path):
    host = fp.build_shim(str(tmp_path), "host")
    a_add, b_add = fp.crafted_pairs()
    rare = {op: fp.mul_operands(host, op, 4, seed=7 + op) for op in (0, 1)}
    rng = np.random.default_rng(3)
    for pub_op, ct_op, shim_op in PAIRS:
        if shim_op in (0, 1):
            a = np.concatenate([rare[shim_op][0], rng.integers(0, 1 << 32, (4000, 8), dtype=np.uint32)])
            b = np.concatenate([rare[shim_op][1], rng.integers(0, 1 << 32, (4000, 8), dtype=np.uint32)])
        elif shim_op == 6:
            a = b = a_add[:64]
        else:
            a, b = a_add, b_add
        got_pub = ed.fe_selftest(to_bytes(a), to_bytes(b), pub_op)
        got_ct = ed.fe_selftest(to_bytes(a), to_bytes(b), ct_op)
        _, want, pend = fp.run(host, shim_op, a, b)
        assert np.array_equal(np.asarray(got_pub), np.asarray(got_ct)), pub_op
        assert np.array_equal(np.asarray(got_pub), to_bytes(want)), pub_op
        if shim_op != 6:
            assert int(pend.sum()) >= 4, (pub_op, int(pend.sum()))
