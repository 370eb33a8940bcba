"""The tcgen05 VQ kernel (vq2.cu) and the "auto" kernel choice against the exact FFMA kernel
and the C oracle.  Needs a B200: run with ``-m gpu``."""
import numpy as np
import pytest
import torch

from oracle import cref

pytestmark = pytest.mark.gpu

# The tcgen05 VQ kernel sums (e - z)^2 of one row in four fp32 partials (64 terms) and adds rows in double; the FFMA kernel and
# the oracle add every term in double.  Per-row relative error <= 16 * 2^-24 ~ 1e-6, random in sign across rows.
SSE_RTOL = 2e-6


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _inputs(N, K, kind, seed):
    rng = np.random.RandomState(seed)
    z = rng.standard_normal((N, 64)).astype(np.float32)
    if kind == "normal":
        E = rng.standard_normal((K, 64)).astype(np.float32)
    elif kind == "default":          # reference init: near-tie stress (SURVEY Q10)
        E = rng.uniform(-1.0 / K, 1.0 / K, size=(K, 64)).astype(np.float32)
        z *= np.float32(0.06)
    elif kind == "dups":             # heavily duplicated codebook: candidate-list overflow path
        base = rng.standard_normal((max(K // 32, 1), 64)).astype(np.float32)
        E = base[rng.randint(0, base.shape[0], size=K)]
    elif kind == "clustered":        # z sits on top of codes
        E = rng.standard_normal((K, 64)).astype(np.float32)
        z = E[rng.randint(0, K, size=N)] + 1e-4 * z
    elif kind == "nonfinite_z":
        E = rng.standard_normal((K, 64)).astype(np.float32)
        z[min(3, N - 1), 5] = np.nan
        z[min(70, N - 1), 9] = np.inf
    elif kind == "nonfinite_e":
        E = rng.standard_normal((K, 64)).astype(np.float32)
        E[K // 2, 3] = np.nan
    elif kind == "huge":
        E = (rng.standard_normal((K, 64)) * 1e15).astype(np.float32)
        z *= np.float32(1e15)
    return z, E


def _run(kernel, z, E):
    from vqvae_b200 import ops
    ops.set_vq_kernel(kernel)
    try:
        out = ops.vq_forward(_cuda(z), _cuda(E))
        torch.cuda.synchronize()
    finally:
        ops.set_vq_kernel("auto")
    return [t.cpu().numpy() for t in out]


CASES = [(1, 1, "normal"), (100, 37, "normal"), (128, 256, "normal"), (129, 257, "normal"),
         (1000, 512, "normal"), (1000, 512, "default"), (777, 512, "dups"), (600, 300, "clustered"),
         (3000, 1024, "normal"), (2000, 1000, "default"), (1500, 8192, "normal"),
         (400, 512, "nonfinite_z"), (400, 512, "nonfinite_e"), (300, 600, "huge"),
         (2000, 9000, "normal"), (2000, 9000, "default")]


@pytest.mark.parametrize("N,K,kind", CASES)
def test_tc_kernel_bit_exact_vs_exact_kernel_and_oracle(N, K, kind):
    """K <= 8192: the tcgen05 kernel, required.  K > 8192 is outside its domain: requiring it fails, and "auto"
    (what VQVAE.forward uses) runs the exact FFMA kernel."""
    z, E = _inputs(N, K, kind, N + K)
    o = cref.vq_rows(z, E)
    i_e, q_e, s_e, h_e = _run("exact", z, E)
    if K > 8192:
        with pytest.raises(RuntimeError, match="not supported"):
            _run("tc", z, E)
    i_t, q_t, s_t, h_t = _run("tc" if K <= 8192 else "auto", z, E)
    assert np.array_equal(i_e, o["idx"])
    assert np.array_equal(i_t, o["idx"]), int((i_t != o["idx"]).sum())
    assert np.array_equal(q_t, o["zq"], equal_nan=True)
    assert np.array_equal(h_t, o["hist"])
    np.testing.assert_allclose(s_t, s_e, rtol=SSE_RTOL, equal_nan=True)


@pytest.mark.parametrize("K,kind", [(512, "normal"), (512, "default"), (1024, "normal")])
def test_tc_kernel_large_n_matches_exact_kernel(K, kind):
    """BASELINE cfg4 scale (2^18 rows here): the selection bound must never drop the
    canonical winner -- identical indices, z_q and histogram to the exact kernel."""
    z, E = _inputs(1 << 18, K, kind, 7)
    i_e, q_e, s_e, h_e = _run("exact", z, E)
    i_t, q_t, s_t, h_t = _run("tc", z, E)
    assert np.array_equal(i_t, i_e), int((i_t != i_e).sum())
    assert np.array_equal(q_t, q_e)
    assert np.array_equal(h_t, h_e) and int(h_t.sum()) == 1 << 18
    np.testing.assert_allclose(s_t, s_e, rtol=SSE_RTOL)
    # oracle spot check on a slice
    o = cref.vq_rows(z[:4096], E)
    assert np.array_equal(i_t[:4096], o["idx"])


@pytest.mark.parametrize("N,K,D,kernel", [(5000, 512, 64, "auto"), (777, 1000, 64, "auto"), (640, 512, 64, "exact"), (300, 96, 32, "auto")])
def test_deferred_sse_reduction(N, K, D, kernel):
    """vqb_vq_forward_deferred_f32 + vqb_vq_reduce_sse_f32 (the reduction may run later / on a side stream)
    give exactly the outputs of vqb_vq_forward_f32, on the tcgen05 kernel and on the exact FFMA kernel."""
    from vqvae_b200 import ops
    rng = np.random.RandomState(N + K)
    z = torch.from_numpy(rng.standard_normal((N, D)).astype(np.float32)).cuda()
    E = torch.from_numpy((rng.standard_normal((K, D)) * 0.7).astype(np.float32)).cuda()
    ops.set_vq_kernel(kernel)
    try:
        i0, q0, s0, h0 = ops.vq_forward(z, E)
        i1, q1, s1, h1, ws = ops.vq_forward(z, E, defer=True)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            ops.vq_reduce_sse(ws, N, K, D, s1)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
    finally:
        ops.set_vq_kernel("auto")
    assert torch.equal(i0, i1) and torch.equal(q0, q1) and torch.equal(h0, h1)
    assert s0.item() == s1.item() and s0.item() > 0
