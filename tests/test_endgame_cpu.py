"""The endgame solver without a GPU: the CPU reference's win/draw/loss against the alpha-beta oracle's exact root values,
argument validation of the library entry points and of the Python API, and a relabel that solves nothing."""
import numpy as np
import pytest
import torch

import alphabeta_oracle as ABO
import oracle as O
import wld_oracle as WO
from alphazero_othello_b200 import _lib, endgame
from alphazero_othello_b200.alphabeta import NONE
from test_alphabeta_cpu import forced_pass_positions, random_positions


def _exact_sign(s, pl):
    """The sign of the best exact root value of the alpha-beta oracle."""
    v, _, _ = ABO.alphabeta(s, pl, 1, int((s == 0).sum()))
    best = int(v[v != NONE].max())
    return (best > 0) - (best < 0)


def test_oracle_wld_is_the_sign_of_the_exact_root_value():
    pos = random_positions(500, 520, (1, 11)) + forced_pass_positions(501, 30)
    pos = [p for p in pos if (p[0] == 0).sum() <= 11]
    assert len(pos) >= 500
    seen = set()
    for s, pl in pos:
        w, nodes = WO.wld(s, pl)
        assert w == _exact_sign(s, pl), (s, pl)
        assert nodes >= 2
        seen.add(w)
    assert seen == {-1, 0, 1}
    g = O.OracleGame()
    assert sum(g.get_valid_moves(s, pl)[64] == 1 for s, pl in pos) >= 20


def test_oracle_wld_of_terminal_roots_is_the_sign_of_the_disc_difference():
    g, rng, term = O.OracleGame(), np.random.default_rng(502), []
    while len(term) < 30:
        s, pl = g.get_initial_state(), 1
        while not g.get_value_and_terminated(s, 0, pl)[1]:
            s = g.get_next_state(s, int(rng.choice(np.nonzero(g.get_valid_moves(s, pl))[0])), pl)
            pl = -pl
        term.append((s, pl))
    for pl in (1, -1):  # one colour wiped out with empty squares left
        s = np.full(64, pl, np.int8)
        s[:13] = 0
        term += [(s.reshape(8, 8), pl), (s.reshape(8, 8), -pl)]
    for s, pl in term:
        d = int((s == pl).sum()) - int((s == -pl).sum())
        assert WO.wld(s, pl) == ((d > 0) - (d < 0), 1)


def test_argument_validation_without_device():
    L = _lib.lib()
    E, cap = _lib.OTH_E_ARG, _lib.SOLVE_MAX_EMPTIES
    assert _lib.WLD_UNSOLVED not in (-1, 0, 1)
    for fn, tail in ((L.oth_solve_wld, (None, None, None)), (L.oth_host_solve_wld, (None, None))):
        assert fn(None, None, 1, cap + 1, *tail) == E     # max_empties above the cap
        assert fn(None, None, 1, -1, *tail) == E
        assert fn(None, None, -1, cap, *tail) == E        # n < 0
        assert fn(None, None, 1, cap, *tail) == E         # missing buffers
        assert fn(None, None, 0, cap, *tail) == _lib.OTH_OK
        assert fn(None, None, 0, 0, *tail) == _lib.OTH_OK


def test_python_argument_errors():
    own = torch.zeros(4, dtype=torch.int64)
    with pytest.raises(ValueError):
        endgame.solve_wld(own, own)                       # not on a CUDA device
    with pytest.raises(ValueError):
        endgame.solve_wld(own, own.to(torch.int32))
    with pytest.raises(ValueError):
        endgame.solve_wld(own, own[:3])
    out = {"boards": torch.zeros((3, 2), dtype=torch.int64), "values": torch.tensor([0.25, -0.5, 1.0], dtype=torch.float64)}
    for bad in (-1, endgame.MAX_EMPTIES + 1):
        with pytest.raises(ValueError):
            endgame.relabel(out, bad)
    with pytest.raises(ValueError):
        from alphazero_othello_b200.self_play_worker import collect_self_play_games
        collect_self_play_games(None, {}, 1, solve_empties=endgame.MAX_EMPTIES + 1)


def test_relabel_with_zero_empties_solves_nothing_and_needs_no_device():
    out = {"boards": torch.tensor([[1, 2], [3, 4]], dtype=torch.int64), "values": torch.tensor([0.3, -0.7], dtype=torch.float64),
           "meta": torch.tensor([5, 6])}
    r = endgame.relabel(out, 0)
    assert r is not out and set(r) == set(out) | {"solved"}
    assert r["values"] is out["values"] and r["meta"] is out["meta"] and r["boards"] is out["boards"]
    assert r["solved"].dtype == torch.bool and not r["solved"].any() and r["solved"].device == out["values"].device
