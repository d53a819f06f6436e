"""The parity tolerance helper (test_parity_gpu.flipped_fraction) on non-finite values: NaN and Inf must not pass as matches."""
import numpy as np

from test_parity_gpu import flipped_fraction


def test_flipped_fraction_counts_non_finite_mismatches():
    nan, inf = np.nan, np.inf
    want = np.array([[1.0, 2.0, 3.0]] * 8, dtype=np.float32)
    assert flipped_fraction(want, want) == 0.0
    got = want.copy()
    got[0, 0] = nan                   # NaN against finite
    got[1, 1] = inf                   # +Inf against finite
    got[2, 2] = 3.0 + 1e-3            # out of tolerance
    got[3, 0] = 1.0 + 1e-5            # within tolerance
    assert flipped_fraction(got, want) == 3 / 8
    assert flipped_fraction(want, got) == 3 / 8
    a = np.array([nan, inf, -inf, nan, inf, -inf, inf, 1.0], dtype=np.float32)[:, None]
    b = np.array([nan, inf, -inf, inf, nan, inf, -inf, -inf], dtype=np.float32)[:, None]
    # the same non-finite value matches; NaN against Inf, Inf of opposite sign and finite against -Inf do not
    assert flipped_fraction(a, b) == 5 / 8
    assert flipped_fraction(a[:3], b[:3]) == 0.0
