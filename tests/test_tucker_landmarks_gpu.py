"""The Tucker entry points on raw MediaPipe landmarks (landmarks=True): the IPD normalisation of
FeatureExtractor.Read_Landmarks_and_Normalizing_using_IPD runs inside every kernel's read of X, and each call must give
the bits of the same call on the reference-normalised features.

The normalised twin of every raw input is the reference's own output (tests/golden/prepost_golden.npz: raw -> norm_X) or
oracle.mlp_oracle.ipd_normalize.  Rows 5 and 6 of the golden take the ipd == 0 branch (values near 1e5), so results are
compared as bit patterns, NaN-aware.
"""
import numpy as np
import pytest
import torch

from oracle import mlp_oracle

pytestmark = pytest.mark.gpu

KERNELS = ["auto", "thread_per_sample", "cta_per_sample", "warp_per_sample", "thread_per_sample_tmem", "tensor_core",
           "tensor_core_generic"]
T = 12


@pytest.fixture(scope="module")
def fitter(art, rows, cuda_lib):
    from nlml_hpe_b200.tucker import TuckerFitter
    return TuckerFitter(art["W"], *rows, device="cuda:0")


def _rows(g, n):
    """n raw rows [n,468,3] and their normalised twins [n,1404]: the golden's 96 faces, repeated."""
    idx = np.arange(n) % g["raw"].shape[0]
    return np.ascontiguousarray(g["raw"][idx]), np.ascontiguousarray(g["norm_X"][idx])


def _gpu(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _bits(x):
    a = x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    return a.view({4: np.uint32, 8: np.uint64}[a.dtype.itemsize])


def _same_bits(a, b):
    a, b = _bits(a), _bits(b)
    return a.shape == b.shape and np.array_equal(a, b)


def test_golden_twin_is_the_oracle_normalisation(prepost_golden):
    """The twin used below is what the oracle's float64 normalisation gives (the fixture itself is sound)."""
    g = prepost_golden
    assert _same_bits(mlp_oracle.ipd_normalize(g["raw"]), g["norm_X"])


@pytest.mark.parametrize("n", [1, 96, 2048, 4096 + 77])
@pytest.mark.parametrize("kernel", KERNELS)
def test_fit_landmarks_bit_exact(fitter, prepost_golden, kernel, n):
    """Both sides of the 1536-row tensor-core threshold and of the 4096-row projection-GEMM threshold."""
    raw, norm = _rows(prepost_golden, n)
    P_raw = fitter.fit(_gpu(raw), T, kernel=kernel, landmarks=True)
    P_norm = fitter.fit(_gpu(norm), T, kernel=kernel)
    assert _same_bits(P_raw, P_norm)


def test_fit_landmarks_flat_rows(fitter, prepost_golden):
    """[N,1404] raw rows are the same call as [N,468,3]."""
    raw, norm = _rows(prepost_golden, 300)
    ref = fitter.fit(_gpu(norm), T)
    assert _same_bits(fitter.fit(_gpu(raw.reshape(300, 1404)), T, landmarks=True), ref)
    assert _same_bits(fitter.fit(_gpu(raw), T, landmarks=True), ref)


@pytest.mark.parametrize("kernel", ["auto", "tensor_core", "thread_per_sample", "tensor_core_generic"])
def test_fit_landmarks_layout_paths(fitter, prepost_golden, kernel):
    """A view with a 16-byte aligned row pitch stays on the TMA projection; an odd column offset falls back to the
    in-kernel phase A.  Each equals the call on the normalised rows in the same layout (the two phase As round
    differently, so the twin must take the same one)."""
    n = 4096 + 77
    raw, norm = _rows(prepost_golden, n)

    def view(x, width, c0):
        buf = torch.zeros((n, width), device="cuda")
        buf[:, c0:c0 + 1404] = _gpu(x.reshape(n, 1404))
        return buf[:, c0:c0 + 1404]

    ref = fitter.fit(_gpu(norm), T, kernel=kernel)
    assert _same_bits(fitter.fit(view(raw, 1408, 0), T, kernel=kernel, landmarks=True), ref)
    assert _same_bits(fitter.fit(view(raw, 1408, 0), T, kernel=kernel, landmarks=True), fitter.fit(view(norm, 1408, 0), T, kernel=kernel))
    assert _same_bits(fitter.fit(view(raw, 1411, 3), T, kernel=kernel, landmarks=True), fitter.fit(view(norm, 1411, 3), T, kernel=kernel))


@pytest.mark.parametrize("n", [96, 4096 + 77])
def test_solve_landmarks_bit_exact(fitter, prepost_golden, n):
    raw, norm = _rows(prepost_golden, n)
    P_raw, ev_raw = fitter.solve(_gpu(raw), return_evals=True, landmarks=True)
    P_norm, ev_norm = fitter.solve(_gpu(norm), return_evals=True)
    assert _same_bits(P_raw, P_norm)
    assert torch.equal(ev_raw, ev_norm)


def test_powell_landmarks_bit_exact(fitter, prepost_golden):
    """x, fun and nfev of the reference's Powell search from raw landmarks equal those from the normalised features
    (and so, with the Powell kernel's bit identity, the reference's normalise-then-Test() chain)."""
    raw, norm = _rows(prepost_golden, 12)      # includes the two ipd == 0 faces (rows 5 and 6)
    x_raw, f_raw, n_raw = fitter.powell(_gpu(raw), return_info=True, landmarks=True)
    x_norm, f_norm, n_norm = fitter.powell(_gpu(norm), return_info=True)
    assert _same_bits(x_raw, x_norm)
    assert _same_bits(f_raw, f_norm)
    assert torch.equal(n_raw, n_norm)


@pytest.mark.parametrize("n", [96, 4096 + 77])
def test_host_variants_equal_device_calls(fitter, prepost_golden, n):
    raw, _ = _rows(prepost_golden, n)
    dev = fitter.fit(_gpu(raw), T, landmarks=True).cpu().numpy()
    assert _same_bits(fitter.fit_host(raw, T, landmarks=True), dev)
    assert _same_bits(fitter.fit_host(raw.reshape(n, 1404), T, landmarks=True), dev)
    dev_s = fitter.solve(_gpu(raw), landmarks=True).cpu().numpy()
    assert _same_bits(fitter.solve_host(raw, landmarks=True), dev_s)


def test_run_time_rank_path(art, cuda_lib):
    """Synthetic (8,5,5,5) core with F = 1404: the run-time-rank kernels (and their FP32 projection kernel) and the
    Powell fit on raw landmarks equal their twins.  Raw landmarks are built from synthetic features by a per-face
    scale and shift, as make_golden_prepost.py does."""
    from nlml_hpe_b200 import synthetic
    from nlml_hpe_b200.tucker import TuckerFitter
    ranks = (8, 5, 5, 5)
    G = synthetic.synthetic_core(ranks, 1404, seed=11, std=1.0)
    rws = [synthetic.synthetic_cos_params(r, 21 + i, base=art[f"optimized_{k}"][:3])
           for i, (r, k) in enumerate(zip(ranks[1:], ("yaw", "pitch", "roll")))]
    n = 200
    feats = synthetic.make_features(n, G, *rws, U_id=None, seed=3)
    rng = np.random.default_rng(8)
    raw = (feats.reshape(n, 468, 3).astype(np.float64) * rng.uniform(0.05, 0.3, (n, 1, 1))
           + rng.uniform(0.3, 0.7, (n, 1, 3))).astype(np.float32)
    norm = mlp_oracle.ipd_normalize(raw)
    fit = TuckerFitter(G, *rws, device="cuda:0")
    for kernel in ("auto", "cta_per_sample", "tensor_core_generic"):
        assert _same_bits(fit.fit(_gpu(raw), T, kernel=kernel, landmarks=True), fit.fit(_gpu(norm), T, kernel=kernel)), kernel
    assert _same_bits(fit.fit(_gpu(raw[:20]), T, landmarks=True), fit.fit(_gpu(norm[:20]), T))   # auto below 32 rows: CTA kernel
    assert _same_bits(fit.fit_host(raw, T, landmarks=True), fit.fit(_gpu(norm), T).cpu().numpy())
    x_raw, f_raw, n_raw = fit.powell(_gpu(raw[:2]), return_info=True, landmarks=True)
    x_norm, f_norm, n_norm = fit.powell(_gpu(norm[:2]), return_info=True)
    assert _same_bits(x_raw, x_norm) and _same_bits(f_raw, f_norm) and torch.equal(n_raw, n_norm)


def test_plan_without_landmark_263_is_rejected(art, rows, prepost_golden, cuda_lib):
    from nlml_hpe_b200 import _lib
    from nlml_hpe_b200.tucker import TuckerFitter
    small = TuckerFitter(np.ascontiguousarray(art["W"][..., :700]), *rows, device="cuda:0")
    raw, _ = _rows(prepost_golden, 8)
    X = _gpu(raw)
    for call in (lambda: small.fit(X, T, landmarks=True), lambda: small.solve(X, landmarks=True),
                 lambda: small.powell(X, landmarks=True), lambda: small.fit_host(raw, T, landmarks=True),
                 lambda: small.solve_host(raw, landmarks=True)):
        with pytest.raises(_lib.NlmlError, match="landmark 263"):
            call()
    small.fit(X.reshape(8, 1404), T)      # the feature entry points of the same plan are unaffected


def test_host_array_to_device_call_raises(fitter, prepost_golden):
    raw, _ = _rows(prepost_golden, 4)
    for call in (fitter.fit, fitter.solve, fitter.powell):
        with pytest.raises(TypeError):
            call(raw, landmarks=True)
        with pytest.raises(TypeError):
            call(torch.from_numpy(raw), landmarks=True)


@pytest.mark.parametrize("kernel,n", [("tensor_core", 4096 + 204), ("tensor_core", 130), ("thread_per_sample", 300),
                                      ("warp_per_sample", 40), ("cta_per_sample", 33), ("tensor_core_generic", 200)])
def test_output_and_input_guards(fitter, prepost_golden, kernel, n):
    """As tests/test_guard_gpu.py, for raw landmarks: fit() into a strided window of a NaN-filled buffer, from a strided
    window of a NaN-filled buffer (the nine per-row constants are read from the row, never from its neighbours), gives the
    contiguous call's bits and leaves the guards untouched."""
    raw, _ = _rows(prepost_golden, n)
    X = _gpu(raw.reshape(n, 1404))
    ref = fitter.fit(X, 6, kernel=kernel, landmarks=True).clone()
    big = torch.full((n + 2, 1408), float("nan"), device="cuda")
    big[1:n + 1, :1404] = X
    out = torch.full((n + 32, 12), float("nan"), device="cuda")
    view = out[16:16 + n, :8]
    fitter.fit(big[1:n + 1, :1404], 6, kernel=kernel, out=view, landmarks=True)
    torch.cuda.synchronize()
    assert _same_bits(view, ref)
    assert torch.isnan(out[:16]).all() and torch.isnan(out[16 + n:]).all() and torch.isnan(out[16:16 + n, 8:]).all()


def test_solve_and_powell_guards(fitter, prepost_golden):
    n = 4096 + 204
    raw, _ = _rows(prepost_golden, n)
    X = _gpu(raw.reshape(n, 1404))
    ref = fitter.solve(X, landmarks=True).clone()
    big = torch.full((n + 2, 1408), float("nan"), device="cuda")
    big[1:n + 1, :1404] = X
    out = torch.full((n + 32, 12), float("nan"), device="cuda")
    view = out[16:16 + n, :8]
    fitter.solve(big[1:n + 1, :1404], out=view, landmarks=True)
    torch.cuda.synchronize()
    assert _same_bits(view, ref)
    assert torch.isnan(out[:16]).all() and torch.isnan(out[16 + n:]).all() and torch.isnan(out[16:16 + n, 8:]).all()
    odd = torch.full((6, 1411), float("nan"), device="cuda")
    odd[1:5, 3:1407] = X[:4]
    assert _same_bits(fitter.powell(odd[1:5, 3:1407], landmarks=True), fitter.powell(X[:4], landmarks=True))
