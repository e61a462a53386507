"""The rule that picks a recompute plan, without a GPU: the memory a new training plan may take under torch's caching
allocator and its per-process fraction, less the step's own allocations."""
from multi_modal_foundation_model_b200.engine import memory_for_plan, step_margin

GB = 1 << 30


def test_free_memory_bounds_when_the_fraction_is_loose():
    # 100 GB free of 180, 10 GB reserved of which 4 GB allocated: 100 GB + the 6 GB held unused
    assert memory_for_plan(100 * GB, 180 * GB, 10 * GB, 4 * GB, 1.0, 0) == 106 * GB


def test_fraction_bounds_when_it_is_tighter_than_free_memory():
    # fraction 0.25 of 180 GB = 45 GB, 10 GB of it reserved: 35 GB more, + 6 GB held unused
    assert memory_for_plan(100 * GB, 180 * GB, 10 * GB, 4 * GB, 0.25, 0) == 41 * GB
    # reserved beyond the fraction: only the unused part of what is held is left, less the excess
    assert memory_for_plan(100 * GB, 180 * GB, 50 * GB, 48 * GB, 0.25, 0) == -3 * GB


def test_margin_is_subtracted():
    assert memory_for_plan(100 * GB, 180 * GB, 0, 0, 1.0, 3 * GB) == 97 * GB


def test_margin_covers_moments_until_they_exist():
    flat = 400 << 20
    assert step_margin(5 << 20, flat, moments=False) == (5 << 20) + 3 * flat     # gradient copy + two moments
    assert step_margin(5 << 20, flat, moments=True) == (5 << 20) + flat          # gradient copy only


def test_fit_decision_at_the_boundary():
    avail = memory_for_plan(20 * GB, 180 * GB, 2 * GB, 2 * GB, 1.0, step_margin(GB, GB, False))
    assert avail == 16 * GB
    assert 16 * GB <= avail and not 16 * GB + 1 <= avail
