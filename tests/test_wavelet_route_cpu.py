"""The kernel route of one wavelet pass (``wats._resolve_route``) against a fake graph, without a GPU:
whether a pass runs on the SELL plan, the plan-free blocked kernel or neither, whether the step kernel
applies the flips' degree patches itself, whether it gets the pre-scaled first operand, and when the
pass counts in ``narrow_calls`` (the plan is built on a graph's second F = 1 pass)."""
import pytest

from efficient_gnn_b200.wats import _resolve_route


class FakeGraph:
    """What the route reads of a ``CsrGraph``.  As there, a weighted or unsorted graph never gets a plan,
    and a graph below the size thresholds gets one only when forced."""

    def __init__(self, n=1000, sorted_rows=True, weighted=False, large=True):
        self.n = n
        self.narrow_calls = 0
        self.sorted, self.weighted, self.large = sorted_rows, weighted, large
        self.plan = None
        self.builds = 0

    def rows_sorted(self):
        return self.sorted

    def has_sell_plan(self):
        return self.plan is not None

    def sell_plan(self, force=False):
        if self.plan is None and self.sorted and not self.weighted and (self.large or force):
            self.plan = object()            # stands for the egnn_sell_plan struct
            self.builds += 1
        return self.plan


def route(g, f=1, k=3, use_sell=None, differentiable=False, flips=False, default_signal=False):
    r = _resolve_route(g, f, k, use_sell, differentiable, flips, default_signal)
    return r.plan is not None, r.blocked, r.in_kernel, r.y0


def test_first_pass_blocked_then_the_plan():
    g = FakeGraph()
    assert route(g) == (False, 1, False, False)
    assert (g.narrow_calls, g.builds) == (1, 0)
    assert route(g) == (True, 0, False, False)
    assert route(g) == (True, 0, False, False)
    assert (g.narrow_calls, g.builds) == (3, 1)


def test_small_graph_stays_off_the_plan_unless_forced():
    g = FakeGraph(large=False)
    assert route(g) == (False, 1, False, False)
    assert route(g) == (False, 1, False, False)
    assert route(g, use_sell=True) == (True, 0, False, False)
    assert route(g) == (True, 0, False, False)        # built once, kept
    assert g.narrow_calls == 4


def test_use_sell_true_builds_the_plan_on_the_first_pass():
    g = FakeGraph()
    assert route(g, use_sell=True) == (True, 0, False, False)
    assert g.narrow_calls == 1


@pytest.mark.parametrize("use_sell", [False, "blocked"])
def test_use_sell_false_and_blocked_never_take_the_plan_or_count(use_sell):
    g = FakeGraph()
    route(g)
    route(g)                                          # the graph has its plan now
    assert g.narrow_calls == 2
    want_blocked = 2 if use_sell == "blocked" else 0
    assert route(g, use_sell=use_sell, flips=True, default_signal=True) == (False, want_blocked, False, False)
    assert route(g, f=8, use_sell=use_sell) == (False, 0, False, False)
    assert g.narrow_calls == 2


def test_blocked_forced_needs_sorted_rows():
    assert route(FakeGraph(sorted_rows=False), use_sell="blocked") == (False, 0, False, False)


@pytest.mark.parametrize("f", [2, 8, 64])
def test_wide_signals_take_neither_and_do_not_count(f):
    g = FakeGraph()
    route(g)
    route(g)
    assert route(g, f=f, default_signal=True, flips=True) == (False, 0, False, False)
    assert route(g, f=f, use_sell=True) == (False, 0, False, False)
    assert g.narrow_calls == 2


def test_order_zero_takes_neither_and_does_not_count():
    g = FakeGraph()
    route(g)
    route(g)
    assert route(g, k=0, flips=True, default_signal=True) == (False, 0, False, False)
    assert route(g, k=0, use_sell=True) == (False, 0, False, False)
    assert g.narrow_calls == 2


def test_unsorted_graph_gets_no_plan_and_no_blocked_kernel():
    g = FakeGraph(sorted_rows=False)
    for use_sell in (None, None, True):
        assert route(g, use_sell=use_sell, flips=True, default_signal=True) == (False, 0, False, False)
    assert (g.narrow_calls, g.builds) == (3, 0)


def test_weighted_graph_gets_no_plan_but_the_blocked_kernel_when_sorted():
    # the blocked kernel has a weighted instantiation; the SELL plan stores no values
    g = FakeGraph(weighted=True)
    for use_sell in (None, None, True):
        assert route(g, use_sell=use_sell, flips=True, default_signal=True) == (False, 1, False, False)
    assert (g.narrow_calls, g.builds) == (3, 0)


def test_flips_patch_in_the_kernel_on_the_plan_unless_differentiable():
    g = FakeGraph()
    assert route(g, flips=True) == (False, 1, False, False)          # first pass: host patches
    assert route(g, flips=True) == (True, 0, True, False)
    assert route(g, flips=True, differentiable=True) == (True, 0, False, False)
    assert route(g, flips=False) == (True, 0, False, False)
    assert g.narrow_calls == 4


def test_first_operand_handed_over_on_the_plan_for_the_default_signal():
    g = FakeGraph()
    assert route(g, default_signal=True) == (False, 1, False, False)
    assert route(g, default_signal=True) == (True, 0, False, True)
    assert route(g, default_signal=True, flips=True) == (True, 0, True, True)
    assert route(g, default_signal=True, flips=True, differentiable=True) == (True, 0, False, True)
    assert route(g, default_signal=False) == (True, 0, False, False)


def test_counter_bumped_once_per_pass():
    g = FakeGraph()
    for i in range(1, 6):
        route(g, flips=bool(i % 2), differentiable=i == 3, default_signal=i > 2)
        assert g.narrow_calls == i
