"""CPU: the tempering flags of the TrendRate and DDRate command lines (-temper, -swap_every, -temper_delta), as those of
literate_b200.forward.  -temper is checked before any device is touched."""
import pytest

from literate_b200 import ddrate as DD
from literate_b200 import library as L
from literate_b200 import trend as TR


@pytest.mark.parametrize("mod", [TR, DD])
def test_defaults_leave_behaviour_unchanged(mod):
    a = mod.build_parser().parse_args([])
    assert (a.temper, a.swap_every, a.temper_delta) == (1, 1000, 0.1)
    a = mod.build_parser().parse_args(["-temper", "8", "-swap_every", "50", "-temper_delta", "0.3"])
    assert (a.temper, a.swap_every, a.temper_delta) == (8, 50, 0.3)


@pytest.mark.parametrize("mod", [TR, DD])
@pytest.mark.parametrize("T", [0, 33, -1])
def test_temper_outside_one_to_thirty_two_is_refused(mod, T):
    a = mod.build_parser().parse_args(["-d", "missing.tsv", "-seed", "1", "-temper", str(T)])
    with pytest.raises(SystemExit, match="-temper must be 1..32"):
        L.seed_and_chains(a, 1)
    with pytest.raises(SystemExit, match="-temper must be 1..32"):
        mod.run(a, device=object())                             # refused before the table is read or a device is used


def test_ladders_of_logged_chains():
    """Logged chain k of a rank holding [c0, c0 + n) is the ladder of device chains [k T, (k + 1) T), all on table k % n_tab."""
    a = TR.build_parser().parse_args(["-temper", "3", "-temper_delta", "0.5"])
    c0, n, rep, beta = L.ladders(a, 2, 3, 2)
    assert (c0, n) == (6, 9)
    assert rep.tolist() == [0, 0, 0, 1, 1, 1, 0, 0, 0]
    assert beta.tolist() == [1.0, 1 / 1.5, 0.5] * 3
    a = TR.build_parser().parse_args([])
    c0, n, rep, beta = L.ladders(a, 2, 3, 2)
    assert (c0, n, rep.tolist(), beta) == (2, 3, [0, 1, 0], None)
