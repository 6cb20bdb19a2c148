"""The shock scenarios of tests/test_gpu_fast_path_window.py cross the fast path's rounding window, proved on the CPU from the
NumPy oracle's unrounded fields: a later change of defaults or seeds cannot quietly leave the GPU tests inside the window."""
import pytest

from kernel_sets import SCENARIOS, WIDE_WINDOW, WINDOW, window_crossings


@pytest.mark.parametrize("name", list(SCENARIOS))
def test_shock_crosses_the_rounding_window_with_finite_fields(name):
    below, above, wide, finite = window_crossings(name)
    print(f"{name}: {below} cover updates below -{WINDOW:g}, {above} at or above {WINDOW:g}")
    assert finite
    assert wide == 0        # inside the 16-bit window of the tile loops' rounding (the shocks test that path)
    if SCENARIOS[name]["crosses"]:
        assert below + above > 0


def test_wide_window_holds_the_default_regime():
    """The host-side bound of DESIGN.md section 2 at the default constants over the default luminosity range stays below
    WIDE_WINDOW - 1000: no reachable state of a default run leaves the tile loops' rounding window."""
    from kernel_sets import update_bound
    for L in (0.75, 1.0, 1.25, 1.5):
        assert update_bound(L) < WIDE_WINDOW - 1000.0, L


def test_each_window_edge_is_crossed():
    """Both edges are covered: the heat and cold shocks drop covers below the window, the upper-edge shock lifts them above."""
    assert window_crossings("cold_pulse")[0] > 1000 and window_crossings("heat_step")[0] > 100
    assert window_crossings("heat_graze")[0] > 0
    assert window_crossings("upper_edge")[1] > 100
