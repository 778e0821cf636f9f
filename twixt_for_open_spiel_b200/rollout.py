"""Batched MCTS leaf evaluation by random rollouts (SURVEY 8f row 3).

Upstream `mcts_example --rollout_count=R` evaluates ONE leaf at a time with
`RandomRolloutEvaluator`: R times { leaf.Clone(); play uniformly random legal
moves to the end; Returns() } and averages; its prior is uniform over
LegalActions().  Here B leaves are evaluated at once: their records are copied
R times inside a scratch batch (device-side clone) and all B*R games are played
by ONE launch of the fused playout kernel; the host only sees [B, 2] mean
returns.  The tree itself stays on the host, as in open_spiel; `mcts.py` runs whole searches with the
trees on the device.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np

from .batch import TwixTBatch
from .spiel import TwixTGame, TwixTState


class BatchedRolloutEvaluator:
    def __init__(self, board_size: int, n_rollouts: int = 4, max_leaves: int = 4096, device: int = 0,
                 seed: int = 0):
        if n_rollouts < 1 or max_leaves < 1:
            raise ValueError("n_rollouts and max_leaves must be positive")
        self.board_size = board_size
        self.n_rollouts = n_rollouts
        self.max_leaves = max_leaves
        # slots [0, max_leaves) hold the leaves, the rest their rollout copies
        self._batch = TwixTBatch(board_size, max_leaves * (1 + n_rollouts), device, seed)
        self._calls = 0

    @property
    def batch(self) -> TwixTBatch:
        return self._batch

    def stream_ids(self, num_leaves: int, call: Optional[int] = None) -> np.ndarray:
        """Philox stream of rollout r of leaf i in evaluation call c: (c * max_leaves + i) * R + r."""
        c = self._calls if call is None else call
        base = (np.uint64(c) * np.uint64(self.max_leaves) + np.arange(num_leaves, dtype=np.uint64))
        return (base[:, None] * np.uint64(self.n_rollouts) + np.arange(self.n_rollouts, dtype=np.uint64)).reshape(-1)

    def evaluate_records(self, records: np.ndarray, max_plies: Optional[int] = None) -> np.ndarray:
        """records: [B, record_words] uint32 leaf states -> [B, 2] float32 mean returns over the rollouts."""
        records = np.ascontiguousarray(records, dtype=np.uint32).reshape(-1, self._batch.record_words)
        num = records.shape[0]
        if num > self.max_leaves:
            raise ValueError("%d leaves > max_leaves %d" % (num, self.max_leaves))
        b, r = self._batch, self.n_rollouts
        b.import_state(records, 0)
        src = np.repeat(np.arange(num, dtype=np.int64), r)
        b.clone_gather(src, self.max_leaves)
        rets, _, _ = b.playout(self.max_leaves, num * r, max_plies=max_plies, stream_ids=self.stream_ids(num),
                               want_lengths=False)
        self._calls += 1
        return rets.reshape(num, r, 2).mean(axis=1, dtype=np.float64).astype(np.float32)

    def evaluate_slots(self, num_leaves: int, max_plies: Optional[int] = None) -> np.ndarray:
        """Device-resident form: the leaves already live in slots [0, num_leaves) of `self.batch` (put there by
        twixt_apply / twixt_replay / twixt_clone_from on the device), so nothing but the [B, 2] means crosses
        the bus: clone x R on the device, one playout launch, the mean over the rollouts on the device."""
        import torch
        if num_leaves > self.max_leaves:
            raise ValueError("%d leaves > max_leaves %d" % (num_leaves, self.max_leaves))
        b, r = self._batch, self.n_rollouts
        dev = torch.device("cuda", b.device)
        if getattr(self, "_dev_src", None) is None:
            b.use_torch_stream()
            self._dev_src = torch.arange(self.max_leaves, dtype=torch.int64, device=dev).repeat_interleave(r)
            self._dev_rets = torch.empty((self.max_leaves * r, 2), dtype=torch.float32, device=dev)
            self._dev_ids = torch.empty(self.max_leaves * r, dtype=torch.int64, device=dev)
        n = num_leaves * r
        self._dev_ids[:n] = torch.arange(n, dtype=torch.int64, device=dev) + self._calls * self.max_leaves * r
        b.clone_gather(self._dev_src[:n], self.max_leaves)
        b.playout(self.max_leaves, n, max_plies=max_plies, stream_ids=self._dev_ids[:n],
                  out_returns=self._dev_rets[:n], want_lengths=False)
        self._calls += 1
        return self._dev_rets[:n].view(num_leaves, r, 2).double().mean(dim=1).float().cpu().numpy()

    def evaluate(self, states: Sequence[TwixTState]) -> np.ndarray:
        """RandomRolloutEvaluator::Evaluate for a list of adapter states."""
        return self.evaluate_records(np.stack([s.export_record() for s in states]))

    @staticmethod
    def prior(state: TwixTState) -> List[Tuple[int, float]]:
        """RandomRolloutEvaluator::Prior: uniform over the legal actions."""
        legal = state.legal_actions()
        return [(a, 1.0 / len(legal)) for a in legal]

    def close(self):
        self._batch.close()
