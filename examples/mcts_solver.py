"""Solving thousands of TwixT endgames at once with the batched MCTS-Solver (BatchedMCTS(..., solve=True)).

B roots at n = 8, each a few plies (2..6) before the end of a seeded random game, are searched with open_spiel's
MCTSBot(solve=True) search: UCT with R random rollouts per leaf, plus the solver's proof pass.  A tree whose root is
proven stops searching.  The script prints how many roots were proven as wins, losses and draws for the player to
move, and the mean number of simulations the trees used.

    python examples/mcts_solver.py [roots] [simulations]
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from twixt_for_open_spiel_b200 import TwixTBatch  # noqa: E402
from twixt_for_open_spiel_b200.mcts import BatchedMCTS  # noqa: E402


def endgame_roots(batch: TwixTBatch, first: int, count: int, backs=(2, 3, 4, 5, 6)):
    """Envs [first, first + count) become positions backs[t % len(backs)] plies before the end of a seeded random
    game: one traced playout, then a replay of all but its last plies."""
    batch.reset(first, count)
    _, lengths, actions = batch.playout(first, count, trace=True)
    batch.reset(first, count)
    back = np.asarray(backs, dtype=np.int32)[np.arange(count) % len(backs)]
    batch.replay(actions.T.astype(np.int32), first, lengths=np.maximum(lengths - back, 0))


def main():
    roots = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
    sims = int(sys.argv[2]) if len(sys.argv) > 2 else 400
    n = 8
    batch = TwixTBatch(n, roots, 0, seed=5)
    endgame_roots(batch, 0, roots)
    player = batch.current_player(0, roots).astype(np.int64)

    search = BatchedMCTS(batch, roots, sims, n_rollouts=2, uct_c=2.0, solve=True)
    search.begin(0, roots)
    search.run(sims)
    proven, returns, edge_values, simulations = search.solver_stats()
    best = search.best()

    value = returns[np.arange(roots), np.clip(player, 0, 1)]  # for the player to move at the root
    p = proven == 1
    print("%d endgame roots at n = %d, %d simulations each, solve=True" % (roots, n, sims))
    print("proven: %d (%.1f %%): %d wins, %d losses, %d draws for the player to move" % (
        p.sum(), 100.0 * p.mean(), (p & (value > 0)).sum(), (p & (value < 0)).sum(), (p & (value == 0)).sum()))
    print("unproven: %d" % (~p).sum())
    print("mean simulations used: %.1f (proven roots %.1f)" % (
        simulations.mean(), simulations[p].mean() if p.any() else float("nan")))
    for t in range(4):
        a = int(best[t])
        moves = "" if a < 0 else " best %s%d (proven value %s)" % (
            chr(ord("a") + a // n), n - a % n, "?" if edge_values[t, a] == -128 else "%+d" % edge_values[t, a])
        print("root %d: %s after %d simulations%s" % (
            t, "proven %+d" % value[t] if p[t] else "unproven", simulations[t], moves))
    search.close()
    batch.close()


if __name__ == "__main__":
    main()
