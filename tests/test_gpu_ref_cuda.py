"""Pin against the REFERENCE's own CUDA kernels: the ops the reference's CPU backends cannot execute -- RMSNorm (no
reference test exists at all), RoPE, AttentionKVCache, Softmax with an axis, LayerNorm -- run through this repo's C-ABI
and compared with what the reference's launchers (oracle/Makefile `ref_cuda`) computed on a B200 from the same inputs,
stored in tests/golden/cuda_ref.npz (re-record on a B200: ITB_RECORD_GOLDEN=1, see tests/golden/store.py)."""
import ctypes

import numpy as np
import pytest

from tests.golden.store import Golden, pick

pytestmark = pytest.mark.gpu
F32, F16 = 1, 10
gold = Golden("cuda_ref")


def R():
    from oracle import ref_cuda  # only when recording: the reference's kernels built into oracle/_ref
    return ref_cuda.lib()


@pytest.fixture(scope="module")
def K():
    import tests.kernel_harness as K
    return K


def _t(a, dt=F32):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda().to(torch.float16 if dt == F16 else torch.float32)


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def _ulps16(a, b):
    def order(v):  # sign-magnitude bit pattern -> monotonic integer
        bits = v.astype(np.float16).view(np.int16).astype(np.int32)
        return np.where(bits < 0, -(bits & 0x7FFF), bits)
    return np.abs(order(a) - order(b))


@pytest.mark.parametrize("dt", [F32, F16])
@pytest.mark.parametrize("shape", [(16, 4096), (3, 256), (5, 1024)])
def test_rmsnorm_vs_reference_kernel(K, shape, dt):
    import torch
    rng = np.random.default_rng(1)
    x = rng.standard_normal(shape).astype(np.float32)
    w = (1 + 0.02 * rng.standard_normal(shape[-1])).astype(np.float32)
    xd, wd = _t(x, dt), _t(w, dt)

    def reference():
        yd = torch.empty_like(xd)
        assert R().ref_cuda_rmsnorm(dt, _p(xd), _p(wd), _p(yd), shape[0], shape[1]) == 0
        return yd.cpu().numpy()
    ref = gold(f"rmsnorm-{shape[0]}x{shape[1]}-dt{dt}", reference)
    got = pick(K.rms_norm(xd.float().cpu().numpy(), wd.float().cpu().numpy(), dt))
    if dt == F32:  # only the reduction order differs (block tree vs warp shuffles)
        np.testing.assert_allclose(got, ref, rtol=2e-6, atol=1e-7)
    else:
        assert _ulps16(got, ref).max() <= 1 and np.mean(got == ref) > 0.99


@pytest.mark.parametrize("dt", [F32, F16])
def test_rope_vs_reference_kernel_row0(K, dt):
    """The reference launch covers batch row 0 / token 0 only (quirk q2, rope.cu:84-85): that row is compared."""
    import torch
    rng = np.random.default_rng(2)
    x = rng.standard_normal((1, 1, 4096)).astype(np.float32)
    pos = np.array([[37]], np.int32)
    xd = _t(x, dt)

    def reference():
        yd = torch.zeros_like(xd)
        pd = torch.from_numpy(pos).cuda()
        assert R().ref_cuda_rope(dt, _p(pd), _p(xd), _p(yd), x.size, 4096, 128, 4096, 1) == 0
        return yd.cpu().numpy()
    ref = gold(f"rope-dt{dt}", reference)
    got = pick(K.rope(pos.astype(np.int64), xd.float().cpu().numpy(), dt))
    if dt == F32:  # the reference evaluates cos/sin in double precision of a float argument; ours in float
        np.testing.assert_allclose(got, ref, rtol=0, atol=2e-5)
    else:
        # both sides round cos / sin and the two products to fp16 and subtract; where the products nearly cancel a one-ulp
        # difference of a factor is many ulps of the small result, so the bound is absolute: 2 fp16 ulps of the operands
        scale = float(np.abs(xd.float().cpu().numpy()).max())
        assert np.abs(got - ref).max() <= 2 * 2.0 ** -10 * scale, (np.abs(got - ref).max(), np.mean(got == ref))
        assert np.mean(got == ref) > 0.5, np.mean(got == ref)


@pytest.mark.parametrize("B,H,S,pos", [(2, 4, 64, 37), (16, 32, 1024, 511), (1, 8, 256, 0)])
def test_attention_kvcache_vs_reference_kernel(K, B, H, S, pos):
    """fp32 (the only dtype the reference kernel has): output within fp32 attention tolerance (the reference does not subtract
    the row maximum, quirk q1), appended cache rows bit-exact, earlier rows untouched."""
    import torch
    rng = np.random.default_rng(3)
    kc = (0.5 * rng.standard_normal((B, H, S, 128))).astype(np.float32)
    vc = (0.5 * rng.standard_normal((B, H, S, 128))).astype(np.float32)
    q, k, v = [(0.5 * rng.standard_normal((B, H, 1, 128))).astype(np.float32) for _ in range(3)]

    def reference():
        kcd, vcd, qd, kd, vd = [_t(a) for a in (kc, vc, q, k, v)]
        od = torch.empty_like(qd)
        pd = torch.tensor([pos], dtype=torch.int32, device="cuda")
        tmp_o = torch.empty(B * H * (S // 8 + 8) * 128, device="cuda")
        tmp_s = torch.empty(B * H * (S // 8 + 8), device="cuda")
        assert R().ref_cuda_attention_kvcache(_p(kcd), _p(vcd), _p(qd), _p(kd), _p(vd), _p(pd), _p(od), B, H, S, 128,
                                              _p(tmp_o), _p(tmp_s)) == 0
        ref_k, ref_v = kcd.cpu().numpy(), vcd.cpu().numpy()
        assert np.array_equal(ref_k[:, :, :pos], kc[:, :, :pos]) and np.array_equal(ref_v[:, :, :pos], vc[:, :, :pos])
        return od.cpu().numpy(), ref_k[:, :, pos], ref_v[:, :, pos]
    ref, ref_krow, ref_vrow = gold(f"attention_kvcache-{B}x{H}x{S}-pos{pos}", reference)
    got, got_k, got_v = K.attention_kvcache(kc, vc, q, k, v, pos, F32, pos_np_dtype=np.int32)
    np.testing.assert_allclose(pick(got), ref, rtol=2e-5, atol=2e-6)
    assert np.array_equal(pick(got_k[:, :, pos]), ref_krow) and np.array_equal(pick(got_v[:, :, pos]), ref_vrow)
    assert np.array_equal(got_k[:, :, :pos], kc[:, :, :pos]) and np.array_equal(got_v[:, :, :pos], vc[:, :, :pos])


@pytest.mark.parametrize("dt", [F32, F16])
@pytest.mark.parametrize("shape,axis", [((1, 12, 128, 128), 3), ((4, 16, 8), 1), ((2, 1500), 1)])
def test_softmax_vs_reference_kernel(K, shape, axis, dt):
    import torch
    rng = np.random.default_rng(4)
    x = rng.standard_normal(shape).astype(np.float32)
    xd = _t(x, dt)

    def reference():
        yd = torch.empty_like(xd)
        stride = int(np.prod(shape[axis + 1:]))
        fn = R().ref_cuda_softmax_f32 if dt == F32 else R().ref_cuda_softmax_f16
        assert fn(_p(xd), _p(yd), x.size, shape[axis], stride) == 0
        return yd.cpu().numpy()
    ref = gold(f"softmax-{'x'.join(map(str, shape))}-axis{axis}-dt{dt}", reference)
    got = pick(K.softmax(xd.float().cpu().numpy(), axis, dt))
    if dt == F32:
        np.testing.assert_allclose(got, ref, rtol=3e-6, atol=1e-8)
    else:
        assert _ulps16(got, ref).max() <= 2


def test_layernorm_vs_reference_kernel(K):
    import torch
    rng = np.random.default_rng(5)
    x = rng.standard_normal((1, 128, 768)).astype(np.float32)
    s, b = (1 + 0.1 * rng.standard_normal(768)).astype(np.float32), (0.1 * rng.standard_normal(768)).astype(np.float32)

    def reference():
        xd, sd, bd = _t(x), _t(s), _t(b)
        yd = torch.empty_like(xd)
        assert R().ref_cuda_layernorm_f32(_p(xd), _p(sd), 1e-5, x.size, 768, 768, 1, _p(yd), _p(bd), 768) == 0
        with_bias = yd.cpu().numpy()
        assert R().ref_cuda_layernorm_f32(_p(xd), _p(sd), 1e-5, x.size, 768, 768, 1, _p(yd), None, 0) == 0
        return with_bias, yd.cpu().numpy()
    ref_bias, ref_nobias = gold("layernorm-1x128x768", reference)
    np.testing.assert_allclose(pick(K.layer_norm(x, s, b, 1e-5, -1, F32)), ref_bias, rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(pick(K.layer_norm(x, s, None, 1e-5, -1, F32)), ref_nobias, rtol=1e-5, atol=2e-6)
