"""The CA-CFAR threshold for non-coherently integrated surfaces (cfar_scale(pfa, N, looks=K), include/caf_b200.h,
DESIGN.md section 13): host arithmetic only, no GPU."""
import math

import numpy as np
import pytest

from caf_cookoff_b200 import api

GRID = [(1e-2, 1), (1e-3, 7), (1e-6, 20), (1e-6, 8320), (1e-9, 100), (0.5, 3), (1e-12, 50)]


def gamma_pfa(alpha, n, k):
    """P(v > alpha * mean) for v ~ Gamma(k) over the mean of n Gamma(k) cells, summed term by term in floats"""
    t = alpha / n
    m = n * k
    return sum(math.exp(math.lgamma(m + i) - math.lgamma(i + 1) - math.lgamma(m) + i * math.log(t) - (m + i) * math.log1p(t))
               for i in range(k))


@pytest.mark.parametrize("pfa,n", GRID)
def test_one_look_is_the_closed_form_bit_for_bit(pfa, n):
    want = n * (pfa ** (-1.0 / n) - 1.0)
    for got in (api.cfar_scale(pfa, n), api.cfar_scale(pfa, n, looks=1), api.cfar_scale(pfa, n, 1)):
        assert np.float64(got).view(np.uint64) == np.float64(want).view(np.uint64)


@pytest.mark.parametrize("pfa,n", GRID)
@pytest.mark.parametrize("looks", [2, 3, 4, 16, 64, 257])
def test_gamma_law_at_the_returned_scale_is_pfa(pfa, n, looks):
    alpha = api.cfar_scale(pfa, n, looks=looks)
    assert alpha > 0.0
    assert gamma_pfa(alpha, n, looks) == pytest.approx(pfa, rel=1e-9)
    assert math.exp(api.cfar_log_pfa(alpha, n, looks)) == pytest.approx(pfa, rel=1e-9)


def test_formula_against_numerical_integration():
    """N = 20, K = 4, alpha = 3: the sum equals P(v > t S), v ~ Gamma(K), S ~ Gamma(NK), by quadrature over S."""
    from scipy import integrate, special, stats
    n, k, alpha = 20, 4, 3.0
    t = alpha / n
    quad, _ = integrate.quad(lambda s: special.gammaincc(k, t * s) * stats.gamma.pdf(s, n * k), 0, np.inf, epsabs=0,
                             epsrel=1e-13, limit=400)
    assert gamma_pfa(alpha, n, k) == pytest.approx(3.6666e-3, rel=1e-4)
    assert math.exp(api.cfar_log_pfa(alpha, n, k)) == pytest.approx(quad, rel=1e-11)


@pytest.mark.parametrize("pfa,n", [(1e-6, 20), (1e-6, 8320), (1e-3, 100)])
def test_scale_decreases_as_looks_grow(pfa, n):
    alphas = [api.cfar_scale(pfa, n, looks=k) for k in (1, 2, 4, 8, 16, 64, 256)]
    assert all(a > b for a, b in zip(alphas, alphas[1:]))
    assert alphas[-1] > 1.0                     # the mean of the sum never clears a threshold at or below the mean


@pytest.mark.parametrize("n,k", [(16, 2), (24, 4), (40, 16), (10, 64)])
def test_monte_carlo_exceedance_rate(n, k):
    """Seeded draws of one Gamma(k) test cell and n Gamma(k) training cells (sums of k exponential cells): the share with
    v > alpha * mean lands within 15 % of Pfa = 1e-3."""
    pfa = 1e-3
    alpha = api.cfar_scale(pfa, n, looks=k)
    rng = np.random.default_rng(1000 * n + k)
    trials, hits = 2_000_000, 0
    for _ in range(trials // 200_000):
        v = rng.gamma(k, size=200_000)
        mean = rng.gamma(n * k, size=200_000) / n          # the sum of n Gamma(k) cells is Gamma(n k)
        hits += int(np.count_nonzero(v > alpha * mean))
    assert abs(hits / trials - pfa) <= 0.15 * pfa, hits / trials


def test_bad_arguments_raise():
    for pfa in (0.0, 1.0, -1e-3, 2.0, float("nan")):
        with pytest.raises(ValueError):
            api.cfar_scale(pfa, 20, looks=4)
    for n in (0, -3):
        with pytest.raises(ValueError):
            api.cfar_scale(1e-6, n, looks=4)
    for looks in (0, -1, 2.5):
        with pytest.raises(ValueError):
            api.cfar_scale(1e-6, 20, looks=looks)
