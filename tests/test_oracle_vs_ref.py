"""Pin the oracle against the REFERENCE ITSELF: outputs of the unmodified reference host + native-CPU kernels
(oracle/Makefile `ref`), stored in tests/golden/native_cpu_ref.npz (re-record: ITB_RECORD_GOLDEN=1, see
tests/golden/store.py).  Covers every op the reference's native CPU backend implements within its valid domain
(SURVEY.md quirk q10: its Softmax ignores the axis, its MatMul is 2-D without trans/bias -- those are exercised only
inside that domain)."""
import numpy as np
import pytest

import oracle
from tests.golden.store import Golden, pick

gold = Golden("native_cpu_ref")


def run_op(*args, **kw):
    from oracle import ref  # only when recording: the reference built into oracle/_ref
    return ref.run_op(*args, **kw)


def rnd(shape, seed, scale=1.0):
    return (np.random.default_rng(seed).standard_normal(shape) * scale).astype(np.float32)


def test_matmul_2d():
    a, b = rnd((37, 53), 0), rnd((53, 29), 1)
    np.testing.assert_allclose(pick(oracle.matmul(a, b)), gold("matmul-37x53x29", lambda: run_op("MatMul", [a, b], [0, 0])),
                               rtol=2e-5, atol=2e-5)
    a, b = rnd((512, 512), 0), rnd((512, 512), 1)     # BASELINE config #1
    np.testing.assert_allclose(pick(oracle.matmul(a, b)), gold("matmul-512", lambda: run_op("MatMul", [a, b], [0, 0])),
                               rtol=1e-4, atol=5e-4)


@pytest.mark.parametrize("xs,ws,args", [((2, 6, 9, 9), (4, 6, 3, 3), (1, 1, 2, 1, 1, 2)),
                                        ((1, 3, 16, 16), (8, 3, 7, 7), (3, 3, 2, 2, 1, 1)),
                                        ((2, 8, 5, 5), (16, 8, 1, 1), (0, 0, 1, 1, 1, 1))])
def test_conv(xs, ws, args):
    x, w = rnd(xs, 2), rnd(ws, 3, 0.3)
    key = "conv-" + "x".join(map(str, xs + ws + args))
    np.testing.assert_allclose(pick(oracle.conv2d(x, w, *args)), gold(key, lambda: run_op("Conv", [x, w], args)),
                               rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("name,op", [("add", "Add"), ("sub", "Sub"), ("mul", "Mul"), ("div", "Div")])
def test_elementwise(name, op):
    a, b = rnd((2, 3, 4, 5), 4), rnd((2, 3, 4, 5), 5) + 3.0
    np.testing.assert_allclose(pick(oracle.binary(name, a, b)), gold("binary-" + name, lambda: run_op(op, [a, b])), rtol=1e-6, atol=0)
    b2 = rnd((1, 3, 1, 5), 6) + 3.0   # broadcast operand
    np.testing.assert_allclose(pick(oracle.binary(name, a, b2)), gold(f"binary-{name}-broadcast", lambda: run_op(op, [a, b2])),
                               rtol=1e-6, atol=0)


@pytest.mark.parametrize("name,op", [("relu", "Relu"), ("gelu", "Gelu"), ("silu", "Silu"), ("sigmoid", "Sigmoid"),
                                     ("tanh", "Tanh"), ("hardsigmoid", "HardSigmoid"), ("hardswish", "HardSwish"),
                                     ("abs", "Abs"), ("sqrt", "Sqrt"), ("erf", "Erf"), ("neg", "Neg")])
def test_unary(name, op):
    x = rnd((3, 7, 11), 7, 2.0)
    if name == "sqrt":
        x = np.abs(x)
    np.testing.assert_allclose(pick(oracle.unary(name, x)), gold("unary-" + name, lambda: run_op(op, [x])), rtol=2e-6, atol=2e-7)


def test_softmax_within_reference_domain():
    x = rnd((1, 40), 8, 2.0)   # the native kernel normalises over the whole tensor: equals axis=-1 for one row
    np.testing.assert_allclose(pick(oracle.softmax(x, -1)), gold("softmax", lambda: run_op("Softmax", [x], [1])),
                               rtol=2e-6, atol=1e-8)


def test_movement_bit_exact():
    x = rnd((2, 5, 3, 4), 9)
    for perm in [(0, 2, 1, 3), (3, 2, 1, 0), (1, 0, 3, 2)]:
        key = "transpose-" + "".join(map(str, perm))
        assert np.array_equal(pick(oracle.transpose(x, perm)), gold(key, lambda: run_op("Transpose", [x], perm)))
    parts = [rnd((2, 3, 4), 10), rnd((2, 1, 4), 11), rnd((2, 5, 4), 12)]
    assert np.array_equal(pick(oracle.concat(parts, 1)), gold("concat", lambda: run_op("Concat", parts, [1])))
    big = rnd((2, 10, 2, 1), 13)
    for i, o in enumerate(oracle.split(big, 1, 3)):
        assert np.array_equal(pick(o), gold(f"split-{i}", lambda: run_op("Split", [big], [1, 3], which_out=i)))
    assert np.array_equal(pick(oracle.reshape(x, (10, 12))), gold("reshape", lambda: run_op("Reshape", [x], [10, 12])))


@pytest.mark.parametrize("kind,op", [("max", "MaxPool"), ("avg", "AveragePool")])
def test_pooling(kind, op):
    x = rnd((2, 3, 9, 11), 14)
    if kind == "max":
        x = np.abs(x)  # the native-CPU max kernel seeds its running maximum with 0; cuDNN (-inf) is what we replace
    kdps = (3, 3, 1, 1, 1, 1, 2, 2)
    got = oracle.pool2d(kind, x, *kdps)
    if kind == "avg":
        # the native CPU kernel divides by the number of in-bounds taps; cuDNN (the CUDA path we replace) counts
        # padding (pooling.cc:88, quirk q9) -- compare on the interior where both agree
        refv = gold("avgpool-interior", lambda: run_op(op, [x], list(kdps) + [0])[:, :, 1:-1, 1:-1])
        np.testing.assert_allclose(pick(got[:, :, 1:-1, 1:-1]), refv, rtol=1e-6, atol=1e-6)
    else:
        assert np.array_equal(pick(got), gold("maxpool", lambda: run_op(op, [x], list(kdps) + [0])))
