"""The tensor-core rank-mu update (des_cma_rank_mu_tc) entry by entry, across the operand scales CMA-ES produces.

Coordinate j of y = B D z has scale sqrt(C_jj), which CMA-ES learns: on ill-conditioned problems the C_jj spread over
many decades, and the overall scale of C drifts.  The split-fp16 operands of the tensor-core kernel must hold every
coordinate to the same relative accuracy, and the norm-wise bars of test_gpu_cma.py cannot see that: the largest
coordinates dominate them.  The bar here is per entry,

    |got_ij - ref_ij| <= 1e-5 sqrt(A_ii A_jj),    A = sum_k |w_k| y_k y_k^T,

which Cauchy-Schwarz makes the natural size of entry (i, j), and which does not change when a coordinate is rescaled.
The CPU tests pin, with a numpy model of the operand split, that this bar tells a per-coordinate power-of-two scale from
no scale at all; the GPU tests hold the kernel to it against the fp64 restatement of the same fp32 inputs."""
import numpy as np
import pytest

from oracle import cma_oracle as cma

DEV = 'cuda:0'
TOL = 1e-5
SCALES = [1e-4, 1e-2, 1.0, 1e4, 1e6, 'spread']


def make_Y(rs, lam, n, scale):
    """randn [lam, n] in fp32, times `scale`, or ('spread') with columns scaled log-uniformly over [1e-3, 1e3] and
    n // 32 of them exactly zero."""
    Y = rs.randn(lam, n)
    if scale == 'spread':
        Y *= np.exp(rs.uniform(np.log(1e-3), np.log(1e3), n))
        Y[:, rs.choice(n, n // 32, replace=False)] = 0.0
    else:
        Y *= scale
    return Y.astype(np.float32)


def make_w(rs, n, lam, kind):
    """'pycma': the default recombination weights (the lower half zero; a single member weighs 1); 'active': signed
    weights as active CMA uses them; 'tiny': the default weights times 1e-8."""
    if kind == 'active':
        w = rs.rand(lam) / lam
        w[lam // 2:] *= -0.3
    else:
        w = cma.cma_constants(n, lam)['w'] if lam > 1 else np.ones(1)
        if kind == 'tiny':
            w = w * 1e-8
    return w.astype(np.float32)


def entrywise_error(got, ref, Y, w, keep=None):
    """max_ij |got_ij - ref_ij| / sqrt(A_ii A_jj) over the entries `keep` selects (all by default).  An exact entry counts
    0 (also where A_ii A_jj = 0); a non-finite error, or any error where A_ii A_jj = 0, counts inf."""
    got = np.asarray(got, dtype=np.float64)
    Y = np.asarray(Y, dtype=np.float64)
    d = np.sqrt((np.abs(np.asarray(w, dtype=np.float64))[:, None] * Y * Y).sum(axis=0))
    err = np.abs(got - ref)
    with np.errstate(divide='ignore', invalid='ignore'):
        r = np.where(err == 0, 0.0, err / np.outer(d, d))
    r[~np.isfinite(r)] = np.inf
    if keep is not None:
        r = r[keep]
    return float(r.max()) if r.size else 0.0


def both_norms(got, ref, tol=TOL):
    got = np.asarray(got, dtype=np.float64)
    assert np.linalg.norm(got - ref) <= tol * np.linalg.norm(ref)
    assert np.max(np.abs(got - ref)) <= tol * np.max(np.abs(ref))


def emulate_split(Y, w, scaled):
    """The kernel's arithmetic up to its accumulator: z_kj = fp32(sqrt|w_k| y_kj), optionally times 2^e_j with e_j putting
    max_k |z_kj| into [2^14, 2^15) (0 for a zero or non-finite column), split into hi = fp16(z) and lo = fp16(z - hi);
    the products hi.hi + lo.hi + hi.lo of Zs = diag(sign w) Z and Z summed in fp64, then times 2^-e_i 2^-e_j.  The fp32
    accumulation of the tensor cores is not modelled."""
    Y = np.asarray(Y, dtype=np.float32)
    w = np.asarray(w, dtype=np.float32)
    z = np.sqrt(np.abs(w))[:, None] * Y
    e = np.zeros(Y.shape[1], dtype=np.int64)
    if scaled:
        zmax = np.abs(z).max(axis=0)
        ok = np.isfinite(zmax) & (zmax > 0)
        e[ok] = np.minimum(15 - np.frexp(zmax[ok])[1], 126)          # zmax = f 2^E, f in [0.5, 1)
        z = z * np.exp2(e).astype(np.float32)                          # exact
    with np.errstate(over='ignore', invalid='ignore'):
        hi = z.astype(np.float16)
        lo = (z - hi.astype(np.float32)).astype(np.float16)
        hi, lo = hi.astype(np.float64), lo.astype(np.float64)
        s = np.where(w < 0, -1.0, 1.0)[:, None]
        D = (s * hi).T @ hi + (s * lo).T @ hi + (s * hi).T @ lo
        u = np.exp2(-e.astype(np.float64))
        return D * u[:, None] * u[None, :]


# ---- CPU: the bar separates the two operand schemes ------------------------------------------------------------------

@pytest.mark.parametrize('scale', [1.0, 1e-4, 1e6, 'spread'])
def test_entrywise_bar_tells_a_scaled_split_from_an_unscaled_one(scale):
    """n = 256, lambda = 1024, default weights.  Unscaled, the lo half of a small coordinate is an fp16 subnormal (a fixed
    2^-24 quantum) and the hi half of a large one overflows: the bar rejects that at Y * 1e-4, at Y * 1e6 and at a 1e6
    spread of column scales, and accepts the per-coordinate power-of-two scale everywhere.  On O(1) data both pass."""
    n, lam = 256, 1024
    rs = np.random.RandomState(7)
    Y = make_Y(rs, lam, n, scale)
    w = make_w(rs, n, lam, 'pycma')
    ref = cma.rank_mu_delta(Y.astype(np.float64), w.astype(np.float64))
    scaled = entrywise_error(emulate_split(Y, w, True), ref, Y, w)
    unscaled = entrywise_error(emulate_split(Y, w, False), ref, Y, w)
    assert scaled <= TOL, scaled
    if scale == 1.0:
        assert unscaled <= TOL, unscaled
    else:
        assert not unscaled <= TOL, unscaled


def test_entrywise_error_is_invariant_under_rescaling_a_coordinate():
    """Scaling coordinate j by 2^s scales row and column j of both got and ref by 2^s and the bar's d_j by 2^s."""
    rs = np.random.RandomState(3)
    Y = rs.randn(40, 9)
    w = rs.rand(40) - 0.3
    ref = cma.rank_mu_delta(Y, w)
    got = ref + 1e-6 * rs.randn(9, 9)
    got = 0.5 * (got + got.T)
    S = np.exp2(np.arange(-40, 41, 10))[None, :9]
    before = entrywise_error(got, ref, Y, w)
    after = entrywise_error(got * S * S.T, ref * S * S.T, Y * S, w)
    assert after == pytest.approx(before, rel=1e-12)


# ---- GPU: the kernel against the fp64 restatement of its fp32 inputs -------------------------------------------------

def check_rank_mu(Y, w, path, n, keep=None):
    """Full and packed output of `path` (None = the automatic choice) against the restatement, entry by entry and in both
    norms; packed tiles expanded through des_cma_cov_apply_packed equal the full matrix, which is exactly symmetric; the
    FFMA kernel meets the same bar.  `keep` restricts the comparison to the entries it selects (non-finite inputs)."""
    import torch
    from distributedes_b200 import ops
    Yt = torch.from_numpy(Y).to(DEV)
    wt = torch.from_numpy(w).to(DEV)
    Yr = np.where(np.isfinite(Y), Y, 0).astype(np.float64)            # the finite reference (keep excludes the rest)
    ref = cma.rank_mu_delta(Yr, w.astype(np.float64))
    full = ops.cma_rank_mu(Yt, wt, path=path)
    tiles = ops.cma_rank_mu_packed(Yt, wt, path=path)
    ffma = ops.cma_rank_mu(Yt, wt, path='ffma')
    C1 = torch.zeros((n, n), device=DEV)
    C2 = torch.zeros((n, n), device=DEV)
    ops.cma_cov_apply(C1, full, None, decay=0.0, c1=0.0, cmu=1.0)
    ops.cma_cov_apply_packed(C2, tiles, None, decay=0.0, c1=0.0, cmu=1.0)
    got = full.cpu().numpy()
    assert np.array_equal(got, got.T, equal_nan=True)                 # exactly symmetric
    assert torch.equal(torch.nan_to_num(C1), torch.nan_to_num(C2)) and torch.equal(C1.isnan(), C2.isnan())
    for name, out in (('tc', got), ('ffma', ffma.cpu().numpy())):
        err = entrywise_error(out, ref, Yr, w, keep)
        assert err <= TOL, (name, err)
        if keep is None:
            both_norms(out, ref)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize('scale,weights', [(s, 'pycma') for s in SCALES] + [('spread', 'active'), ('spread', 'tiny'),
                                                                         (1.0, 'tiny'), (1e4, 'active')])
def test_baseline_config_entrywise_over_scales(scale, weights):
    """BASELINE configs[4] (n = 4096, lambda = 1024) through the automatic dispatch, which takes the tensor cores."""
    from distributedes_b200 import ops
    n, lam = 4096, 1024
    assert n >= ops.CMA_TC_MIN_N
    rs = np.random.RandomState(4096)
    check_rank_mu(make_Y(rs, lam, n, scale), make_w(rs, n, lam, weights), None, n)


@pytest.mark.gpu
@pytest.mark.parametrize('scale', [1e-4, 1e6, 'spread'])
@pytest.mark.parametrize('weights', ['pycma', 'active', 'tiny'])
@pytest.mark.parametrize('lam', [1, 65, 129, 1024])
@pytest.mark.parametrize('n', [1, 33, 129, 255])
def test_forced_tensor_cores_at_small_and_ragged_shapes(n, lam, weights, scale):
    """path='tc' below the dispatch threshold: one partial output tile, ragged n; lambda padded to 1, 2, 3 and 16 k-stages of
    64 (an odd number splits unevenly between the two K-half accumulators)."""
    rs = np.random.RandomState(n * 10007 + lam)
    check_rank_mu(make_Y(rs, lam, n, scale), make_w(rs, n, lam, weights), 'tc', n)


@pytest.mark.gpu
@pytest.mark.parametrize('bad', [np.inf, -np.inf, np.nan])
@pytest.mark.parametrize('n,path', [(255, 'tc'), (2048, None)])
def test_a_non_finite_coordinate_stays_in_its_row_and_column(n, path, bad):
    """An inf or NaN in coordinate j of one member: every entry outside row and column j still meets the bar against the
    reference without it (a scale shared across coordinates would let it reach every entry), and entry (j, j) is not
    finite (the value is not silently dropped)."""
    lam = 129
    rs = np.random.RandomState(n)
    Y = make_Y(rs, lam, n, 'spread')
    w = make_w(rs, n, lam, 'pycma')
    j = n // 3
    Y[0, j] = bad                                                    # member 0 has the largest weight
    keep = np.ones((n, n), dtype=bool)
    keep[j, :] = keep[:, j] = False
    got = check_rank_mu(Y, w, path, n, keep)
    assert not np.isfinite(got[j, j])


@pytest.mark.gpu
def test_one_generation_at_an_ill_conditioned_covariance():
    """n = 2048 (tensor cores by the automatic dispatch), lambda = 512, from C = diag(d^2), B = I, D = d with d log-uniform over
    [1e-3, 1e3] (condition number 1e12) and m = 0: CMAEvolutionStrategy and the fp64 restatement tell() the same fp32
    solutions.  dC entry by entry, C entry by entry relative to sqrt(C_ii C_jj), and m, sigma, pc, ps as in
    test_gpu_cma.test_full_cma_generation_matches_restatement."""
    import torch
    from distributedes_b200.cma_es import CMAEvolutionStrategy
    n, lam = 2048, 512
    rs = np.random.RandomState(12)
    d = np.exp(rs.uniform(np.log(1e-3), np.log(1e3), n))
    es = CMAEvolutionStrategy(np.zeros(n), 1.0, lam, seed=5, device=DEV)
    ref = cma.CMAState(np.zeros(n), 1.0, lam)
    ref.C, ref.B, ref.D = np.diag(d * d), np.eye(n), d.copy()
    es.C = torch.diag(torch.from_numpy(d * d)).to(DEV, torch.float32).contiguous()
    es.B = torch.eye(n, dtype=torch.float64, device=DEV)
    es.D = torch.from_numpy(d).to(DEV)
    Xr = ref.ask(rs.randn(lam, n)).astype(np.float32)
    cost = cma.sphere(Xr)
    es.tell(torch.from_numpy(Xr).to(DEV), torch.from_numpy(cost))
    order = ref.tell(Xr.astype(np.float64), cost)
    Ysorted = Xr[order]                                              # m_old = 0, sigma = 1
    err = entrywise_error(es.dC.cpu().numpy(), ref.dC, Ysorted, ref.k['w'])
    assert err <= TOL, ('dC', err)
    dref = np.sqrt(np.diag(ref.C))
    Cerr = np.abs(es.C.cpu().numpy().astype(np.float64) - ref.C) / np.outer(dref, dref)
    assert Cerr.max() <= TOL, ('C', Cerr.max())
    assert np.linalg.norm(es.m.cpu().numpy() - ref.m) <= 1e-6 * np.linalg.norm(ref.m)
    assert abs(es.sigma - ref.sigma) <= 1e-6 * ref.sigma
    assert np.linalg.norm(es.pc.cpu().numpy() - ref.pc) <= 1e-6 * np.linalg.norm(ref.pc)
    assert np.linalg.norm(es.ps.cpu().numpy() - ref.ps) <= 1e-4 * np.linalg.norm(ref.ps)
