"""-m gpu: W8A8 GEMM (SURVEY.md section 8 row f4; kernels/csrc/qgemm/w8a8/w8a8_gemm_cuda.cu) through the mirrored op
`omniserve_backend.qgemm_w8a8.w8a8_gemm_forward_cuda`, against the CPU oracle (INT32 accumulate bit-exact, fp16 tail
rounded once from the fp32 product) and the reference's own kernel rebuilt for sm_100 (oracle/_ref)."""
import numpy as np
import pytest
import torch

from tests.gpu_util import ref_module, reference_outputs, t

pytestmark = pytest.mark.gpu


def _inputs(M, N, K, seed):
    rng = np.random.default_rng(seed)
    a = rng.integers(-127, 128, (M, K), dtype=np.int8)
    w = rng.integers(-127, 128, (N, K), dtype=np.int8)
    ws = rng.uniform(0.002, 0.01, N).astype(np.float16)
    sa = rng.uniform(0.01, 0.05, M).astype(np.float16)
    return a, w, ws, sa


@pytest.mark.parametrize("M,N,K", [(1, 128, 128), (17, 256, 512), (64, 4096, 4096), (100, 1024, 2048), (300, 384, 1024),
                                   (1024, 6144, 4096), (64, 160, 256)])
def test_w8a8_gemm_vs_oracle_and_reference_kernel(M, N, K):
    from omniserve_b200.backend import qgemm_w8a8 as ours
    from oracle import w4a8 as ow
    a, w, ws, sa = _inputs(M, N, K, M + N + K)
    out = torch.full((M, N), float("nan"), dtype=torch.float16, device="cuda")
    args = [t(a), t(w), t(ws), t(sa)]
    ours.w8a8_gemm_forward_cuda(*args, out)
    torch.cuda.synchronize()
    _, ref = ow.gemm_w8a8(a, w, ws, sa)
    got = out.cpu().numpy()
    assert not np.isnan(got.astype(np.float32)).any()
    g32, r32 = got.astype(np.float32), ref.astype(np.float32)
    assert np.abs(g32 - r32).max() <= 1e-3 * np.abs(r32).max()
    assert (got == ref).mean() > 0.999
    rm = ref_module("qgemm_w8a8")
    if N % (256 if M > 128 else 64) == 0:   # the reference tiles N by 64 (M <= 128) / 256 without masking
        def run():
            o2 = torch.zeros((M, N), dtype=torch.float16, device="cuda")
            rm.w8a8_gemm_forward_cuda(*args, o2)
            torch.cuda.synchronize()
            return {"out": o2}
        r = reference_outputs(f"w8a8_{M}x{N}x{K}", rm is not None, run)
        a, b = r.pair("out", got)
        assert np.abs(a.astype(np.float32) - b.astype(np.float32)).max() <= 1e-3 * r.absmax("out")
        assert (a == b).mean() > 0.999


def test_w8a8_int32_accumulators_exact():
    """ws = sa = 1 and |acc| <= 2048: the fp16 output is the INT32 accumulator."""
    from omniserve_b200.backend import qgemm_w8a8 as ours
    rng = np.random.default_rng(3)
    M, N, K = 96, 512, 2048
    a = np.zeros((M, K), np.int8)
    for m in range(M):
        idx = rng.choice(K, 16, replace=False)
        a[m, idx] = rng.choice(np.array([-1, 1], np.int8), 16)
    w = rng.integers(-127, 128, (N, K), dtype=np.int8)
    want = (a.astype(np.int64) @ w.astype(np.int64).T).astype(np.int32)
    assert np.abs(want).max() <= 2048
    out = torch.empty((M, N), dtype=torch.float16, device="cuda")
    ours.w8a8_gemm_forward_cuda(t(a), t(w), t(np.ones(N, np.float16)), t(np.ones(M, np.float16)), out)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(out.cpu().numpy().astype(np.int32), want)


def test_w8a8_row_slice_output_view():
    from omniserve_b200.backend import qgemm_w8a8 as ours
    from oracle import w4a8 as ow
    a, w, ws, sa = _inputs(40, 256, 256, 9)
    buf = torch.full((40, 512), float("nan"), dtype=torch.float16, device="cuda")
    ours.w8a8_gemm_forward_cuda(t(a), t(w), t(ws), t(sa), buf[:, :256])
    torch.cuda.synchronize()
    _, ref = ow.gemm_w8a8(a, w, ws, sa)
    got = buf.cpu().numpy()
    assert np.isnan(got[:, 256:].astype(np.float32)).all()
    assert (got[:, :256] == ref).mean() > 0.999
