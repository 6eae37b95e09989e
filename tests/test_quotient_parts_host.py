"""The quotient by coset parts, as a big-integer model of what the part kernels compute (CPU only).

With n = 2^k and J = 2^(extended_k - k), extended row t = r + J*i is the point zeta * w_ext^r * w^i, so the extended coset is J
parts of n points.  The model below transforms each part with an n-point DFT (the twisted transform of ntt.cu), divides by the
per-part constant g_r^n - 1, and rebuilds the coefficients with a J-point inverse DFT per index (the recombination kernel).  It
must give exactly the oracle's full-coset coeff_to_extended / extended_to_coeff, for every number of kept pieces."""
import random

import pytest

from oracle import oracle as O
from oracle.pyref import R_MOD, ZETA, coeff_to_extended, dft, omega_for


def model_coeff_to_extended_part(coeffs, k, ext_k, part):
    g = ZETA * pow(omega_for(ext_k), part, R_MOD) % R_MOD
    return dft([c * pow(g, m, R_MOD) % R_MOD for m, c in enumerate(coeffs)], omega_for(k))


def model_extended_parts_to_coeff(parts, k, ext_k, n_pieces, divide_by_vanishing):
    n, J = 1 << k, 1 << (ext_k - k)
    w_inv, w_ext, w_j = pow(omega_for(k), -1, R_MOD), omega_for(ext_k), omega_for(ext_k - k)
    e = []
    for r, values in enumerate(parts):
        g = ZETA * pow(w_ext, r, R_MOD) % R_MOD
        scale = pow(n, -1, R_MOD)
        if divide_by_vanishing:
            scale = scale * pow(pow(g, n, R_MOD) - 1, -1, R_MOD) % R_MOD
        g_inv = pow(g, -1, R_MOD)
        e.append([x * scale % R_MOD * pow(g_inv, m, R_MOD) % R_MOD for m, x in enumerate(dft(values, w_inv))])
    zn_inv, j_inv = pow(pow(ZETA, n, R_MOD), -1, R_MOD), pow(J, -1, R_MOD)
    out = []
    for j in range(n_pieces):
        sc = pow(zn_inv, j, R_MOD) * j_inv % R_MOD
        out += [sc * sum(pow(w_j, (J - r) * j % J, R_MOD) * e[r][m] for r in range(J)) % R_MOD for m in range(n)]
    return out


CASES = [(k, log_j) for k in (2, 3, 4) for log_j in (0, 1, 2, 3)]


@pytest.mark.parametrize("k,log_j", CASES)
def test_parts_are_the_strided_slices_of_the_coset(k, log_j):
    rng = random.Random(100 * k + log_j)
    ext_k, J = k + log_j, 1 << log_j
    coeffs = [rng.randrange(R_MOD) for _ in range(1 << k)]
    full = coeff_to_extended(coeffs, k, ext_k)
    dom = O.EvaluationDomain(J + 1, k)  # quotient degree J: extended_k = k + log J
    assert dom.extended_k == ext_k
    assert O.frs_to_ints(dom.coeff_to_extended(O.frs_from_ints(coeffs))) == full
    for r in range(J):
        assert model_coeff_to_extended_part(coeffs, k, ext_k, r) == full[r::J]


@pytest.mark.parametrize("k,log_j", CASES)
def test_recombined_parts_give_the_oracles_extended_to_coeff(k, log_j):
    rng = random.Random(200 * k + log_j)
    n, ext_k, J = 1 << k, k + log_j, 1 << log_j
    h_ext = [rng.randrange(R_MOD) for _ in range(J * n)]
    dom = O.EvaluationDomain(J + 1, k)
    w_ext, zn = omega_for(ext_k), pow(ZETA, n, R_MOD)
    t_inv = [pow(zn * pow(w_ext, n * t, R_MOD) - 1, -1, R_MOD) for t in range(J)]  # divide_by_vanishing_poly, period J
    divided = [x * t_inv[t % J] % R_MOD for t, x in enumerate(h_ext)]
    want_plain = O.frs_to_ints(dom.extended_to_coeff(O.frs_from_ints(h_ext)))
    want_div = O.frs_to_ints(dom.extended_to_coeff(O.frs_from_ints(divided)))
    assert len(want_plain) == J * n
    parts = [h_ext[r::J] for r in range(J)]
    for n_pieces in range(1, J + 1):
        assert model_extended_parts_to_coeff(parts, k, ext_k, n_pieces, False) == want_plain[: n_pieces * n]
        assert model_extended_parts_to_coeff(parts, k, ext_k, n_pieces, True) == want_div[: n_pieces * n]


def test_vanishing_polynomial_is_constant_on_a_part():
    k, ext_k = 3, 5
    n, J = 1 << k, 1 << (ext_k - k)
    w, w_ext = omega_for(k), omega_for(ext_k)
    for r in range(J):
        g = ZETA * pow(w_ext, r, R_MOD) % R_MOD
        assert {pow(g * pow(w, i, R_MOD), n, R_MOD) for i in range(n)} == {pow(g, n, R_MOD)}
        for i in range(n):  # and row r + J*i of the extended coset is g * w^i
            assert g * pow(w, i, R_MOD) % R_MOD == ZETA * pow(w_ext, r + J * i, R_MOD) % R_MOD
