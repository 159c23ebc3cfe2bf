"""The full-size config-2 fixture (tests/golden/c2_logpdf.npz) is what the GPU test measures the grid kernels
against: pin it -- a few of its points recomputed with the oracle (bit for bit) and compared with the reference's own
_ParzenEstimator.log_pdf on the same 100 000-kernel estimator (1e-12; stored by tests/_reference_golden.py)."""
import numpy as np

from oracle import tpe_oracle as orc
from tests._reference_golden import recorded
from tests._util import load


def test_fixture_points_against_oracle_and_live_reference():
    g = load("c2_logpdf.npz")
    N, P = 100_000, 32
    rs = np.random.RandomState(0)
    X = rs.uniform(0, 1, (N, P))
    loss = ((X - 0.5) ** 2).sum(1)
    below, above = orc.split_trials(np.zeros(N, np.int8), np.stack([loss, np.zeros(N)], 1), orc.default_gamma(N))
    assert np.array_equal(below, g["below"])
    params = [orc.Param("float", 0.0, 1.0) for _ in range(P)]
    cfg = orc.Config(multivariate=True)
    pick = [0, 131, 255]
    x = g["x"][pick]
    ma = orc.build_mixture(X[above], params, cfg)
    mb = orc.build_mixture(X[below], params, cfg)
    assert np.array_equal(orc.mixture_log_pdf(ma, x), g["logg"][pick])
    assert np.array_equal(orc.mixture_log_pdf(mb, x), g["logl"][pick])

    def reference_log_pdf():
        import optuna
        from optuna.samplers._tpe.parzen_estimator import _ParzenEstimator, _ParzenEstimatorParameters
        from optuna.samplers._tpe.sampler import default_weights
        names = [f"x{j:02d}" for j in range(P)]
        space = {n: optuna.distributions.FloatDistribution(0.0, 1.0) for n in names}
        prm = _ParzenEstimatorParameters(prior_weight=1.0, consider_magic_clip=True, consider_endpoints=False,
                                         weights=default_weights, multivariate=True, categorical_distance_func={})
        pts = {n: x[:, j] for j, n in enumerate(names)}
        return [_ParzenEstimator({n: X[rows, j] for j, n in enumerate(names)}, space, prm).log_pdf(pts).tolist()
                for rows in (above, below)]

    logg, logl = recorded("test_fixture_points_against_oracle_and_live_reference/log_pdf", reference_log_pdf)
    np.testing.assert_allclose(logg, g["logg"][pick], rtol=0, atol=1e-12)
    np.testing.assert_allclose(logl, g["logl"][pick], rtol=0, atol=1e-12)
