"""GPU: the time-sliced team build of K3 (between one and two chains per SM, csrc/k3_team.cuh k3_team_slot_kernel).

A slice ends by the clock, so where a chain is cut and which chains share an SM change from run to run.  None of it may
show: with slices of a few tens of microseconds (hundreds of cuts per launch), records, final states and event counters
must be those of the compact build (loop_variant 2), bit for bit.
"""
import numpy as np
import pytest

from conftest import golden_input
from oracle import literate_oracle as O
from literate_b200 import engine as E, synth

pytestmark = pytest.mark.gpu

TINY_SLICE_US = "20"
RAGGED = [(1, 0), (7, 1), (1025, 5), (3000, 0), (64, 3), (4096, 100), (5, 1), (2047, 64)]


@pytest.fixture(scope="module")
def tables(device):
    ts, te = synth.syn_int(200_000, 3)
    st = device.bin_stats(ts, te, only_dead=True)
    return {m: E.Dataset(device, st, m, float(ts.min()), float(te.max())) for m in (0, 1, 2, 3)}


def _sliced(device, monkeypatch, n_chains):
    """The automatic build of a population between one and two chains per SM, with at least one SM in eight left to a
    single chain, is the sliced one."""
    sm = device.sm_count
    if not sm < n_chains <= 2 * sm - sm // 8:
        pytest.skip("%d chains are not in the sliced range on %d SMs" % (n_chains, sm))
    monkeypatch.delenv("LR_TEAM_W", raising=False)
    monkeypatch.setenv("LR_TEAM_SLICE_US", TINY_SLICE_US)


def _same(a, b, runs, key):
    for k, (n, s) in enumerate(runs):
        ra, rb = a.run(n, s), b.run(n, s)
        if s:
            assert np.array_equal(ra, rb), (key, k, n, s)
        assert np.array_equal(a.state(), b.state()), (key, k, n)
    assert np.array_equal(a.counters(), b.counters()), key


@pytest.mark.parametrize("nobail", [0, 1])
@pytest.mark.parametrize("n_chains", [149, 200, 256, 278])
def test_sliced_teams_give_the_compact_chains(device, tables, monkeypatch, n_chains, nobail):
    _sliced(device, monkeypatch, n_chains)
    monkeypatch.setenv("LR_TEAM_NOBAIL", str(nobail))
    ds = tables[0]
    a = E.Chains(ds, n_chains, 31, E.default_config(0, loop_variant=2))
    b = E.Chains(ds, n_chains, 31, E.default_config(0, loop_variant=0))
    l0 = device.kernel_launches
    _same(a, b, [(6000, 250)], (n_chains, nobail))
    assert device.kernel_launches - l0 > 20          # the run was cut into slices
    _same(a, b, RAGGED, (n_chains, nobail))
    t = b.team_stats().sum(0)
    assert t[4] > 0                                  # teams did run


def test_sliced_teams_with_hand_over(device, monkeypatch):
    """A small table (40 % of the iterations change the state): teams hand their chains over inside a slice."""
    _sliced(device, monkeypatch, 200)
    monkeypatch.delenv("LR_TEAM_NOBAIL", raising=False)
    lin = O.read_lineages(golden_input("example_dataTAD.txt"))
    st = device.bin_stats(lin.ts, lin.te, end_time=lin.end_time)
    ds = E.Dataset(device, st, 0, lin.start_time, lin.end_time)
    a = E.Chains(ds, 200, 8, E.default_config(0, loop_variant=2))
    b = E.Chains(ds, 200, 8, E.default_config(0, loop_variant=0))
    _same(a, b, [(20000, 500)] + RAGGED, "hand-over")
    assert b.team_stats()[:, 5].sum() > 0            # hand-overs did happen


@pytest.mark.parametrize("model", [0, 1, 2, 3])
def test_sliced_teams_every_likelihood_model(device, tables, monkeypatch, model):
    _sliced(device, monkeypatch, 256)
    monkeypatch.delenv("LR_TEAM_NOBAIL", raising=False)
    ds = tables[model]
    a = E.Chains(ds, 256, 5 + model, E.default_config(model, loop_variant=2))
    b = E.Chains(ds, 256, 5 + model, E.default_config(model, loop_variant=0))
    _same(a, b, [(5000, 100), (333, 7)], model)


def test_sliced_teams_chains_with_different_counters(device, tables, monkeypatch):
    """Chains set to different iteration counters: every chain runs n_iter from its own counter, across slices."""
    _sliced(device, monkeypatch, 256)
    monkeypatch.delenv("LR_TEAM_NOBAIL", raising=False)
    ds = tables[0]
    c = E.Chains(ds, 256, 12, E.default_config(0, loop_variant=2))
    c.run(3000)
    snap = c.state()
    a = E.Chains(ds, 256, 12, E.default_config(0, loop_variant=2))
    b = E.Chains(ds, 256, 12, E.default_config(0, loop_variant=4))
    snap[:, E.REC_IT] += 37 * (np.arange(256) % 29)
    a.set_state(snap); b.set_state(snap)
    _same(a, b, [(4000, 0), (1, 0), (2500, 0)], "set_state")
    assert np.array_equal(a.state()[:, E.REC_IT], snap[:, E.REC_IT] + 6501)
