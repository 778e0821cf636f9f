"""Thousands of MCTS searches at once on the device (twixt_for_open_spiel_b200/mcts.py).

Part 1: 4 096 roots at n = 12 (each a few random plies into a game), every one searched with open_spiel's UCT
MCTS and R = 4 random rollouts per leaf; the best move of the first roots is printed.

Part 2, AlphaZero-style: the leaves are evaluated by a (stand-in) value head instead of rollouts.  Each
simulation is `select` (leaves -> batch envs) -> the obs + mask producer on those envs -> the value head ->
`backup`, all on the device.

    python examples/mcts_search.py [simulations]
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from twixt_for_open_spiel_b200 import TwixTBatch  # noqa: E402
from twixt_for_open_spiel_b200.mcts import BatchedMCTS  # noqa: E402
from twixt_for_open_spiel_b200.producer import ObservationMaskProducer  # noqa: E402


def main():
    sims = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    n, roots = 12, 4096
    batch = TwixTBatch(n, 2 * roots, 0, seed=1)   # envs [0, roots) hold the roots, [roots, 2*roots) the leaves
    batch.playout(0, roots, max_plies=6, want_returns=False, want_lengths=False)

    # -- 1. built-in rollout evaluator -------------------------------------------------------------------------
    search = BatchedMCTS(batch, roots, sims, n_rollouts=4, uct_c=2.0)
    search.begin(0, roots)
    search.run(sims)
    visits, value_sums, best = search.root_stats()
    for t in range(4):
        a = int(best[t])
        x, y = divmod(a, n)
        print("root %d: best %s%d  visits %d  mean value %+.3f" % (
            t, chr(ord("a") + x), n - y, visits[t, a], value_sums[t, a] / max(1, visits[t, a])))

    # -- 2. stepwise form with a value network -------------------------------------------------------------------
    dev = torch.device("cuda:0")
    batch.use_torch_stream()
    producer = ObservationMaskProducer(batch, max_count=roots)
    value_head = torch.nn.Sequential(torch.nn.Flatten(), torch.nn.Linear(12 * n * (n - 2), 1), torch.nn.Tanh()).to(dev)
    status = torch.zeros(roots, dtype=torch.int32, device=dev)
    az = BatchedMCTS(batch, roots, sims)
    az.begin(0, roots)
    with torch.no_grad():
        for _ in range(sims):
            az.select(roots, out_status=status)         # leaf of tree t -> env roots + t
            obs, _ = producer.produce(roots, roots)
            v = value_head(obs).squeeze(1)              # value for red; terminal leaves are scored by the search
            az.backup(torch.stack([v, -v], dim=1).float().contiguous())
    best_dev = torch.zeros(roots, dtype=torch.int32, device=dev)
    az.root_stats(out_best=best_dev)
    print("value-head search: best moves of roots 0..7:", best_dev[:8].tolist())
    az.close()
    search.close()
    batch.close()


if __name__ == "__main__":
    main()
