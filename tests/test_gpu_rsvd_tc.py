"""tcgen05 (3xTF32) rSVD passes vs FP64 NumPy (src/svd.py:52-60 products)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CASES = [(128, 64, 8), (256, 4096, 25), (512, 20001, 25), (100, 5003, 25), (700, 9000, 40), (1500, 3001, 25), (33, 257, 3)]


@pytest.mark.parametrize('m,n,r', CASES)
def test_sketch_and_xty_on_tensor_cores(cuda, m, n, r):
    import torch
    from gladsgp_b200 import ops
    rng = np.random.default_rng(m * 7 + r)
    X = (rng.standard_normal((m, n)) * rng.uniform(0.1, 3, size=(1, n))).astype(np.float32)
    Om = rng.standard_normal((r, n)).astype(np.float32)
    Yh = rng.standard_normal((m, r)).astype(np.float32)
    Xd, Od, Yd = (torch.as_tensor(a, device='cuda') for a in (X, Om, Yh))
    X64 = X.astype(np.float64)
    ref = X64 @ Om.astype(np.float64).T
    got = ops.rsvd_sketch_tc(Xd, Od).cpu().numpy()
    # FP32-level: the split keeps ~21 bits per product and chunk sums are added in round-to-nearest FP32
    assert np.abs(got - ref).max() <= 1e-6 * np.abs(ref).max()
    refb = Yh.astype(np.float64).T @ X64
    gotb = ops.rsvd_xty_tc(Xd, Yd).cpu().numpy()
    assert gotb.shape == (r, n)
    assert np.abs(gotb - refb).max() <= 1e-6 * np.abs(refb).max()
    # deterministic: same bits on a second call
    assert np.array_equal(got, ops.rsvd_sketch_tc(Xd, Od).cpu().numpy())
    assert np.array_equal(gotb, ops.rsvd_xty_tc(Xd, Yd).cpu().numpy())


def test_exact_on_tf32_representable_inputs(cuda):
    """Inputs that are exactly representable in TF32 with small integer values: every product and sum is exact."""
    import torch
    from gladsgp_b200 import ops
    rng = np.random.default_rng(0)
    m, n, r = 256, 2048, 25
    X = rng.integers(-8, 9, size=(m, n)).astype(np.float32)
    Om = rng.integers(-4, 5, size=(r, n)).astype(np.float32)
    Yh = rng.integers(-4, 5, size=(m, r)).astype(np.float32)
    Xd, Od, Yd = (torch.as_tensor(a, device='cuda') for a in (X, Om, Yh))
    assert np.array_equal(ops.rsvd_sketch_tc(Xd, Od).cpu().numpy(), (X.astype(np.int64) @ Om.astype(np.int64).T).astype(np.float32))
    assert np.array_equal(ops.rsvd_xty_tc(Xd, Yd).cpu().numpy(), (Yh.astype(np.int64).T @ X.astype(np.int64)).astype(np.float32))


def test_randomized_svd_large_m(cuda):
    """m > 1024 (cfg5-sized ensembles) goes through the tensor-core passes; compare with a dense SVD."""
    from gladsgp_b200 import svd
    rng = np.random.default_rng(3)
    m, n, p = 1300, 6000, 12
    U0, _ = np.linalg.qr(rng.standard_normal((m, p)))
    V0, _ = np.linalg.qr(rng.standard_normal((n, p)))
    s0 = np.linspace(50, 5, p)
    X = ((U0 * s0) @ V0.T + 1e-3 * rng.standard_normal((m, n))).astype(np.float32)
    np.random.seed(1)
    U, S, Vh = svd.randomized_svd(X, p, k=8, q=1)
    s_all = np.linalg.svd(X.astype(np.float64), compute_uv=False)
    np.testing.assert_allclose(S, s_all[:p], rtol=2e-4)
    rec = (U * S) @ Vh
    best = np.sqrt(np.sum(s_all[p:] ** 2))                      # error of the optimal rank-p approximation
    assert np.linalg.norm(rec - X) <= 1.02 * best


def test_sharded_rsvd_single_rank_equals_randomized_svd(cuda):
    """dist.randomized_svd_sharded on one rank (no process group) == svd.randomized_svd with the same test matrix."""
    import torch
    from gladsgp_b200 import svd, dist as gdist
    rng = np.random.default_rng(8)
    m, n, p = 96, 4001, 10
    X = (rng.standard_normal((m, 12)) @ rng.standard_normal((12, n)) + 0.01 * rng.standard_normal((m, n))).astype(np.float32)
    omega = rng.standard_normal((n, p)).astype(np.float32)
    U0, S0, Vh0 = svd.randomized_svd(X, p, k=0, q=1, omega=omega)
    U, S, Vh = gdist.randomized_svd_sharded(torch.as_tensor(X, device='cuda'), p, k=0, q=1, omega_slab=omega)
    np.testing.assert_array_equal(S.cpu().numpy(), S0)
    np.testing.assert_array_equal(U.cpu().numpy(), U0)
    np.testing.assert_array_equal(Vh.cpu().numpy(), Vh0)


def _misaligned(a):
    """Device copy of `a` whose base is 4 bytes past a 16-byte boundary (a view at storage offset 1)."""
    import torch
    buf = torch.empty(a.size + 1, dtype=torch.float32, device='cuda')
    buf[1:] = torch.as_tensor(a.reshape(-1), device='cuda')
    return buf[1:].view(a.shape)


@pytest.mark.parametrize('m,n,r', [(256, 4096, 25), (512, 20004, 25), (700, 9000, 40), (100, 5004, 25), (33, 260, 3)])
def test_sketch_kernel_per_alignment(cuda, m, n, r):
    """Row pitch a multiple of 16 bytes: aligned X and Omega^T take the TMA-fed kernel (fused hi products, raw hi tile), a
    4-byte misaligned Omega^T or X the register-staged kernel with scalar loads -- including ragged last chunks and row
    blocks (zero fill by the hardware instead of by predicated loads).  Each is at FP32 level against the float64
    product and deterministic, and the kernels agree with one another at the same level."""
    import torch
    from gladsgp_b200 import ops
    rng = np.random.default_rng(m + n)
    X = (rng.standard_normal((m, n)) * rng.uniform(0.1, 3, size=(1, n))).astype(np.float32)
    Om = rng.standard_normal((r, n)).astype(np.float32)
    Xd, Od = torch.as_tensor(X, device='cuda'), torch.as_tensor(Om, device='cuda')
    truth = X.astype(np.float64) @ Om.astype(np.float64).T
    scale = np.abs(truth).max()
    got = []
    for x, o in ((Xd, Od), (Xd, _misaligned(Om)), (_misaligned(X), Od)):
        y = ops.rsvd_sketch_tc(x, o).cpu().numpy()
        assert np.abs(y - truth).max() <= 1e-6 * scale
        assert np.array_equal(y, ops.rsvd_sketch_tc(x, o).cpu().numpy())
        got.append(y)
    for y in got[1:]:
        assert np.abs(y - got[0]).max() <= 2e-6 * scale


def test_sketch_beyond_int32_columns(cuda):
    """n >= 2^31 columns (past the int32 coordinates of a tensor map): the register-staged kernel with 16-byte loads.
    X = Omega^T = one row of values in {-1, 0, 1}, so every product and every partial sum is an exact integer and
    X Omega is the number of non-zeros."""
    import torch
    from gladsgp_b200 import ops
    n = (1 << 31) + 36
    g = torch.Generator(device='cuda'); g.manual_seed(5)
    X = torch.randint(-1, 2, (1, n), dtype=torch.float32, device='cuda', generator=g)
    nnz = int((X != 0).sum())
    assert ops.rsvd_sketch_tc(X, X).item() == np.float32(nnz)


@pytest.mark.parametrize('m,n,r', [(512, 20004, 25), (700, 9000, 40), (100, 5004, 25), (33, 260, 3), (256, 4096, 25),
                                   (512, 20032, 25), (300, 8224, 40), (70, 320, 5)])
def test_xty_against_float64(cuda, m, n, r):
    """Y^T X (register -> TMEM kernel) at FP32 level against the float64 product, deterministic."""
    import torch
    from gladsgp_b200 import ops
    rng = np.random.default_rng(m + n + 2)
    X = (rng.standard_normal((m, n)) * rng.uniform(0.1, 3, size=(1, n))).astype(np.float32)
    Yh = rng.standard_normal((m, r)).astype(np.float32)
    Xd, Yd = torch.as_tensor(X, device='cuda'), torch.as_tensor(Yh, device='cuda')
    truth = Yh.astype(np.float64).T @ X.astype(np.float64)
    got = ops.rsvd_xty_tc(Xd, Yd).cpu().numpy()
    assert got.shape == (r, n)
    assert np.abs(got - truth).max() <= 1e-6 * np.abs(truth).max()
    assert np.array_equal(got, ops.rsvd_xty_tc(Xd, Yd).cpu().numpy())


@pytest.mark.parametrize('m,n', [(512, 1460000), (1100, 1200004)])
def test_passes_at_full_ensemble_size_against_float64(cuda, m, n):
    """BASELINE.json cfg3 at full size (512 x 1.46 M float32, 3 GB) and an ensemble beyond 4 GB (byte offsets above 2^32): both
    passes against float64 products formed on the device in column chunks; inputs generated on the device."""
    import torch
    from gladsgp_b200 import ops
    r = 25
    g = torch.Generator(device='cuda'); g.manual_seed(m)
    X = torch.randn((m, n), dtype=torch.float32, device='cuda', generator=g)
    X *= torch.rand((1, n), dtype=torch.float32, device='cuda', generator=g) * 2.9 + 0.1
    Om = torch.randn((r, n), dtype=torch.float32, device='cuda', generator=g)
    Yh = torch.randn((m, r), dtype=torch.float32, device='cuda', generator=g)
    got = ops.rsvd_sketch_tc(X, Om).double()
    gotb = ops.rsvd_xty_tc(X, Yh)
    ref = torch.zeros((m, r), dtype=torch.float64, device='cuda')
    errb, scaleb = 0.0, 0.0
    step = 100000
    for c0 in range(0, n, step):
        Xc = X[:, c0:c0 + step].double()
        ref += Xc @ Om[:, c0:c0 + step].double().T
        rb = Yh.double().T @ Xc
        errb = max(errb, float((gotb[:, c0:c0 + step].double() - rb).abs().max()))
        scaleb = max(scaleb, float(rb.abs().max()))
    assert float((got - ref).abs().max()) <= 2e-6 * float(ref.abs().max())
    assert errb <= 1e-6 * scaleb
