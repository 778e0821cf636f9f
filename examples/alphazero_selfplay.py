"""AlphaZero self-play with the device PUCT search (twixt_for_open_spiel_b200/mcts.py, selection="puct").

The loop open_spiel's alpha_zero actor runs (MCTSBot with AlphaZeroEvaluator, child_selection_fn = puct_value,
solve = False, dirichlet_noise = (epsilon, alpha)), for B games at once, with a small random-init policy/value
net.  Each move:
  1. `begin` copies the B game envs as the roots;
  2. every simulation is `select` (leaves -> envs [B, 2B)) -> the obs + mask producer on the leaf envs -> the net
     -> a masked softmax (priors) -> `current_player` to orient the value as [v, -v] / [-v, v] -> Dirichlet
     noise on simulation 0, whose leaf is always the root -> `backup(values, priors)`;
  3. `root_stats` gives the policy target, visits^(1/temperature) normalised;
  4. the move is sampled from it before `temperature_drop` moves, and is the best child after;
  5. one `apply` moves every game, with -1 for the finished ones.
Everything stays on the device; per move only the count of running games, which the loop prints, crosses the
bus.  The trajectories (obs, mask, policy target, player, action per move) and the final returns are copied to
the host at the end.

leaves_per_step=K > 1 searches K leaves per tree in each step with virtual loss (BatchedMCTS): the leaf envs are
[B, B + B*K), row g*K + j being descent j of game g, so each network call evaluates B*K leaves and a move takes
sims / K calls.  Every descent of the first step stops at the root, which takes the priors of row g*K + 0: the
Dirichlet noise goes into those rows.

reuse_tree=True keeps each game's tree between moves (BatchedMCTS.advance): `begin` runs once, and after each
`apply` the played move's subtree becomes the new root with its statistics (at most sims + 1 nodes of a search
holding 2*sims), so every move still runs sims new simulations on top of what the last search spent there.  The
root Dirichlet noise then reaches a kept root through `set_root_priors`; a root the advance left without
statistics (ROOT_FRESH) is expanded by the first backup as after `begin`, so the noise goes into its row g*K + 0
there, masked on the device.

    python examples/alphazero_selfplay.py [board_size] [games] [simulations] [leaves_per_step] [reuse_tree]
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from twixt_for_open_spiel_b200 import TwixTBatch  # noqa: E402
from twixt_for_open_spiel_b200.mcts import ROOT_FRESH, BatchedMCTS, add_dirichlet_noise  # noqa: E402
from twixt_for_open_spiel_b200.producer import ObservationMaskProducer  # noqa: E402


class PolicyValueNet(torch.nn.Module):
    """A small convolutional policy/value net: logits [B, n*n] and a value in [-1, 1] for the player to move."""

    def __init__(self, n: int, width: int = 32):
        super().__init__()
        self.trunk = torch.nn.Sequential(torch.nn.Conv2d(12, width, 3, padding=1), torch.nn.ReLU(),
                                         torch.nn.Conv2d(width, width, 3, padding=1), torch.nn.ReLU(),
                                         torch.nn.Flatten())
        self.policy = torch.nn.Linear(width * n * (n - 2), n * n)
        self.value = torch.nn.Sequential(torch.nn.Linear(width * n * (n - 2), 1), torch.nn.Tanh())

    def forward(self, obs):
        h = self.trunk(obs)
        return self.policy(h), self.value(h).squeeze(1)


def masked_softmax(logits, legal):
    return torch.softmax(logits.float().masked_fill(~legal, float("-inf")), dim=1).nan_to_num(0.0)


def self_play(n=8, games=64, sims=50, temperature=1.0, temperature_drop=10, uct_c=2.0, dirichlet_epsilon=0.25,
              dirichlet_alpha=1.0, seed=0, net=None, verbose=True, leaves_per_step=1, virtual_loss=1.0,
              reuse_tree=False):
    """Plays `games` games to the end.  Returns (trajectories, returns [games, 2]); trajectories[g] is a list of
    per-move dicts with obs [12, n, n-2], mask [n*n], policy [n*n], player and action.  sims must be a multiple
    of leaves_per_step.  reuse_tree=True keeps the played move's subtree between moves (see the module text)."""
    K = int(leaves_per_step)
    if sims % K:
        raise ValueError("sims = %d is not a multiple of leaves_per_step = %d" % (sims, K))
    torch.manual_seed(seed)
    dev = torch.device("cuda:0")
    rows = games * K
    batch = TwixTBatch(n, games + rows, 0, seed)  # envs [0, games) are the games, [games, games + games*K) the leaves
    batch.use_torch_stream()
    producer = ObservationMaskProducer(batch, max_count=rows)
    if net is None:
        net = PolicyValueNet(n).to(dev).eval()
    capacity = 2 * sims if reuse_tree else sims
    search = BatchedMCTS(batch, games, capacity, uct_c=uct_c, selection="puct", leaves_per_step=K,
                         virtual_loss=virtual_loss)
    fresh = torch.ones(games, dtype=torch.bool, device=dev)  # roots without statistics (all of them at begin)
    status = torch.zeros(games, dtype=torch.int32, device=dev)
    player = torch.zeros(rows, dtype=torch.int8, device=dev)
    root_player = torch.zeros(games, dtype=torch.int8, device=dev)
    done = torch.zeros(games, dtype=torch.uint8, device=dev)
    visits = torch.zeros((games, n * n), dtype=torch.int32, device=dev)
    best = torch.zeros(games, dtype=torch.int32, device=dev)
    history = []  # per move: (obs, mask, policy, player, action, live) on the device
    move = 0
    with torch.no_grad():
        while True:
            batch.is_terminal(0, games, out=done)
            live = done == 0
            running = int(live.sum().item())
            if verbose:
                print("move %3d: %d games running" % (move, running))
            if running == 0:
                break
            root_obs, root_mask = producer.produce(0, games)
            root_obs, root_mask = root_obs.clone(), root_mask.clone()
            batch.current_player(0, games, out=root_player)
            if not reuse_tree:
                search.begin(0, games)
            elif move == 0:
                search.begin(0, games)
            else:  # kept roots take their noise now; fresh ones at the first backup below
                root_legal = root_mask.bool()
                root_priors = masked_softmax(net(root_obs)[0], root_legal)
                search.set_root_priors(add_dirichlet_noise(root_priors, root_legal, dirichlet_epsilon,
                                                           dirichlet_alpha).contiguous())
            for k in range(sims // K):
                search.select(games)
                obs, mask = producer.produce(games, rows)
                legal = mask.bool()
                logits, v = net(obs)
                priors = masked_softmax(logits, legal)
                if k == 0:
                    if K == 1 and not reuse_tree:
                        priors = add_dirichlet_noise(priors, legal, dirichlet_epsilon, dirichlet_alpha)
                    else:  # the root rows g*K + 0, and with reuse_tree only where the root is fresh
                        noisy = add_dirichlet_noise(priors[::K], legal[::K], dirichlet_epsilon, dirichlet_alpha)
                        priors[::K] = torch.where(fresh[:, None], noisy, priors[::K])
                batch.current_player(games, rows, out=player)
                v = torch.where(player == 1, -v, v).float()
                search.backup(torch.stack([v, -v], dim=1).contiguous(), priors.contiguous())
            search.root_stats(out_visits=visits, out_best=best)
            policy = visits.double() ** (1.0 / temperature)
            policy = (policy / policy.sum(1, keepdim=True).clamp_min(1e-300)).float()
            if move < temperature_drop:
                sampled = torch.multinomial(torch.where(live[:, None], policy, torch.ones_like(policy)), 1)
                action = sampled.squeeze(1).int()
            else:
                action = best.clone()
            action = torch.where(live, action, torch.full_like(action, -1)).contiguous()
            history.append((root_obs, root_mask, policy, root_player.clone(), action, live))
            batch.apply(action, 0)
            if reuse_tree:
                search.advance(action, sims + 1, out_status=status)
                fresh = status == ROOT_FRESH
            move += 1
    returns = batch.returns(0, games)
    trajectories = [[] for _ in range(games)]
    for obs, mask, policy, pl, action, live in history:
        obs, mask, policy, pl, action, live = (x.cpu().numpy() for x in (obs, mask, policy, pl, action, live))
        for g in np.nonzero(live)[0]:
            trajectories[g].append({"obs": obs[g], "mask": mask[g], "policy": policy[g], "player": int(pl[g]),
                                    "action": int(action[g])})
    search.close()
    batch.close()
    return trajectories, returns


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 8
    games = int(sys.argv[2]) if len(sys.argv) > 2 else 256
    sims = int(sys.argv[3]) if len(sys.argv) > 3 else 100
    leaves = int(sys.argv[4]) if len(sys.argv) > 4 else 1
    reuse = len(sys.argv) > 5 and sys.argv[5] not in ("0", "false", "False")
    trajectories, returns = self_play(n, games, sims, leaves_per_step=leaves, reuse_tree=reuse)
    lengths = [len(t) for t in trajectories]
    print("%d games at n = %d, %d simulations per move: mean length %.1f, red wins %d, blue wins %d, draws %d" % (
        games, n, sims, float(np.mean(lengths)), int((returns[:, 0] > 0).sum()), int((returns[:, 1] > 0).sum()),
        int((returns[:, 0] == 0).sum())))


if __name__ == "__main__":
    main()
