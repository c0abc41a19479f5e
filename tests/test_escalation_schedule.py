"""Pop budgets by work position (pdmpc_escalation_budgets): under the default escalation threshold the searches that
start late in the work order get fewer pops on the tile shapes before the CTA shape runs them again.  A CPU test of the
budget function and a GPU test that predicts the escalated set from pop counts and work positions."""
import numpy as np
import pytest

from oracle import oracle_py, parity
from pdmpc_b200 import capi

from helpers import road_records


@pytest.fixture
def default_schedule(monkeypatch):
    for k in ("PDMPC_ESC_MIN", "PDMPC_ESC_SLOPE"):
        monkeypatch.delenv(k, raising=False)


@pytest.mark.parametrize("n", [56000, 168000, 358400])
def test_budget_by_position(built, default_schedule, n):
    pos = np.arange(n, dtype=np.int32)
    b = capi.escalation_budgets(n, pos)
    p_max = 4096 if n >= 300000 else 3072 if n >= 120000 else 2560   # the uniform threshold of the size
    assert b.max() <= p_max
    assert np.all(np.diff(b) <= 0)                       # never more pops for a later start
    assert b[-1] == 1024 and b[n - 7104] < 1250          # the last searches get a reduced budget, never none
    if n >= 300000:
        assert b[n // 4] == p_max                        # the first quarter of a large batch keeps the full budget
    # the same function at any position subset
    sel = np.array([n - 1, 0, n // 3, n - 7104], dtype=np.int32)
    assert capi.escalation_budgets(n, sel).tolist() == b[sel].tolist()


def test_budget_experiment_variables(built, monkeypatch):
    monkeypatch.setenv("PDMPC_ESC_MIN", "100")
    monkeypatch.setenv("PDMPC_ESC_SLOPE", "10")
    n = 56000
    b = capi.escalation_budgets(n, [0, n - 20000, n - 1000, n - 1])
    assert b.tolist() == [2560, 2100, 200, 100]          # min(P_max, P_min + (n - p) // S)
    monkeypatch.setenv("PDMPC_ESC_SLOPE", "0")
    assert capi.escalation_budgets(n, [0, n - 1]).tolist() == [2560, 2560]


def test_budget_rejects_bad_positions(built):
    for pos in ([-1], [10]):
        with pytest.raises(capi.PdmpcError):
            capi.escalation_budgets(10, pos)


def heavy_first(batch, Hp, s0, s1):
    """The library's work order of searches [s0, s1): most obstacle polygons first, stable."""
    sp = batch.slot_ptr.astype(np.int64)
    idx = np.arange(s0, s1)
    key = sp[(idx + 1) * (Hp + 1)] - sp[idx * (Hp + 1)]
    return idx[np.argsort(-key, kind="stable")]


@pytest.mark.gpu
def test_escalated_set_follows_the_work_position(planner, monkeypatch):
    """With a steep schedule most late searches go over their budget: the CTA shape runs exactly the predicted set
    (a search is given up after budget(p) pops unless that pop was its goal), staged and pipelined (where positions
    count in the whole batch, not in the chunk), with the outputs of the oracle and of the launch without escalation."""
    mpa, batch = road_records("triple_speed", 8)
    planner.upload_mpa(mpa)
    n, Hp = batch.n, mpa.Hp
    ref = oracle_py.plan_batch(mpa, batch, 4, hash_valid_pops_only=True)
    pops = ref.n_pops.astype(np.int64)
    exh = ref.is_exhausted != 0
    monkeypatch.setenv("PDMPC_ESC_MIN", "8")
    monkeypatch.setenv("PDMPC_ESC_SLOPE", "1")
    budget = capi.escalation_budgets(n, np.arange(n, dtype=np.int32)).astype(np.int64)
    assert budget[0] > budget[-1]

    def expected(order):
        bs = np.empty(n, dtype=np.int64)
        bs[order] = budget                               # budget of each search by its work position
        return int(((pops > bs) | ((pops == bs) & exh)).sum())

    try:
        planner.set_cta_queue(True)
        planner.set_variant(2)
        planner.set_escalation(0)
        off = planner.plan_batch(batch, raise_on_search_error=False)
        parity.compare(off, ref)
        planner.set_escalation(-1)
        for short in (-1, 10):                           # one master per CTA / several masters
            planner.set_escalation(-1, short)
            planner.set_pipeline_chunks(1)
            dev = planner.plan_batch(batch, raise_on_search_error=False)
            st = planner.stats()
            parity.compare(dev, ref)
            parity.compare(dev, off)
            want = expected(heavy_first(batch, Hp, 0, n))
            assert 0 < want < n and st.escalated == want, (st.escalated, want)
            planner.set_pipeline_chunks(3)
            dev = planner.plan_batch(batch, raise_on_search_error=False)
            st = planner.stats()
            parity.compare(dev, ref)
            bnd = capi.pipeline_bounds(n, 3)
            order = np.concatenate([heavy_first(batch, Hp, bnd[c], bnd[c + 1]) for c in range(len(bnd) - 1)])
            assert st.escalated == expected(order), (st.escalated, expected(order))
    finally:
        planner.set_variant(0)
        planner.set_pipeline_chunks(0)
        planner.set_cta_queue(False)
        planner.set_escalation(-1)
