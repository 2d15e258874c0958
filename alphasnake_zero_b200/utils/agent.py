"""Agent -- mirror of code/utils/agent.py:7-147 (root search driver).  The epoch / depth loops, the Q cache and the
in-tree policy (MCTSAgent, agent.py:149-223, and MCTSMPGameRunner, mp_game_runner.py:79-115) run as CUDA kernels
inside the Engine; this class keeps the reference's constructor, `make_moves(games, ids)`, `records` / `values`
and `clear()`."""
import random

import numpy as np
import torch


class DeviceRecords:
    """Sequence view of one column of the engine's device-resident record store: `len()`, integer indexing (one record is
    copied to the host) and iteration, which is all alpha_snake_zero_trainer.py:64-75 does with Agent.records / values.
    Bulk consumers use Agent.sample_training_batch (one gather kernel, nothing goes through the host)."""

    def __init__(self, agent, column):
        self._agent, self._column = agent, column

    def __len__(self):
        eng = self._agent._engine
        return 0 if eng is None or not self._agent._records_on else eng.records_count()

    def __getitem__(self, i):
        n = len(self)
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(n))]
        if i < 0:
            i += n
        if not 0 <= i < n:
            raise IndexError(i)
        return self._agent._engine.records_views()[self._column][i].cpu().numpy()

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    def __eq__(self, other):
        """list semantics for callers that compare with a list (e.g. `agent.records == []` after clear())"""
        try:
            if len(other) != len(self):
                return False
        except TypeError:
            return NotImplemented
        return all(np.array_equal(a, b) for a, b in zip(self, other))

    __hash__ = None


class Agent:

    def __init__(self, nnet, softmax_base=100, training=False, max_MCTS_depth=8, max_MCTS_breadth=128, records_capacity=None,
                 host_records=False):
        """records_capacity (extension): initial rows of the device-resident record store when training (default: 32 root turns
        x games x snakes; it doubles when full); host_records=True keeps the reference's two host lists instead (one plane copy per record)."""
        self.nnet = nnet
        self.softmax_base = softmax_base
        self.training = training
        self.max_MCTS_depth = max_MCTS_depth
        self.max_MCTS_breadth = max_MCTS_breadth
        self._engine = None
        self._records_on = False
        self._records_capacity = records_capacity
        self._host_records = host_records
        # record data for training (agent.py:21-23)
        if training:
            if host_records:
                self.records = []
                self.values = []
            else:
                self.records = DeviceRecords(self, 0)
                self.values = DeviceRecords(self, 1)

    def make_moves(self, games, ids):
        eng = getattr(games, "engine", None)
        if eng is None:
            raise TypeError("Agent.make_moves needs the games of an engine-backed MPGameRunner (no CPU path)")
        self._engine = eng
        value_fn, native = self.search_values()
        q, mv = eng.search(value_fn=value_fn, net=native)
        mvh = mv.cpu().numpy()                         # the only per-turn device -> host traffic: G x 8 bytes of moves
        moves = [int(mvh[g, s]) for g, s in ids]
        if any(m > 2 for m in moves):      # a live snake without a searched row: never hand an arbitrary direction to the tic
            from .._lib import AszError
            raise AszError("search returned no move for a live snake (ids do not match the engine's live snakes)")
        if self.training and not self._host_records:
            # agent.py:93-97: root states and their Q rows (snapshots; the reference stores aliases, SURVEY.md D-17) go into
            # the engine's device-resident store: one encode launch + one gather of the Q rows, nothing through the host
            if not self._records_on:
                cap = self._records_capacity or 32 * eng.G * eng.S
                eng.records_enable(cap)
                self._records_on = True
            eng.records_append()
        elif self.training:
            qh = q.cpu().numpy()
            planes, rows = eng.encode_rows()
            row_of = {(int(r) // 8, int(r) % 8): i for i, r in enumerate(rows)}
            ph = planes.cpu().numpy()
            for g, s in ids:
                self.records.append(ph[row_of[(g, s)]])
                self.values.append(qh[g, s].copy())
        return moves

    def search_values(self):
        """(value_fn, native network) of Engine.search for this agent's network: both None for no network or a StubNet (the
        engine's stub value function)."""
        if self.nnet is None or getattr(self.nnet, "is_stub", False):
            return None, None
        if getattr(self.nnet, "backend", "native") == "torch":
            return self.nnet.v_device, None            # explicit PyTorch reference network: Python-driven loop
        return None, self.nnet._get_native()           # product path: the whole root turn in one native call

    # agent.py:114-122 (host restatement for callers that use it directly)
    def softermax(self, z):
        z = np.asarray(z, dtype=np.float32)
        with np.errstate(divide="ignore"):
            normalized = np.power(np.float32(self.softmax_base), np.arctanh(z)).astype(np.float32)
        sigma = np.float32(0)
        for n in normalized:
            sigma = np.float32(sigma + n)
        if sigma == 0.0:
            return np.array([1.0 / 3.0] * 3, dtype=np.float32)
        return normalized / sigma

    # agent.py:124-137
    def argmaxs(self, Z):
        out = [-1] * len(Z)
        for i in range(len(Z)):
            if Z[i][0] > Z[i][1]:
                out[i] = 0 if Z[i][0] > Z[i][2] else 2
            else:
                out[i] = 1 if Z[i][1] > Z[i][2] else 2
        return out

    def sample_training_batch(self, batch_size=2048, max_batches=5, mirror=True, rng=random):
        """alpha_snake_zero_trainer.py:62-77: up to max_batches x batch_size records drawn without replacement (the whole set
        when there are fewer than batch_size), then the mirrored copies (:93-100).  Returns (X, V, batch_size): device tensors
        [m, N, N, 3] / [m, 3] and the batch size the trainer passes to AlphaNNet.train."""
        n_rec = len(self.records)
        batches = min(max_batches, n_rec // batch_size)
        samples = batch_size * batches
        if samples > n_rec or samples == 0:       # :67-69 (fewer records than one batch: everything, as one batch)
            batch_size = n_rec
            samples = batch_size
        idx = rng.sample(range(n_rec), samples)   # :70
        if self._host_records:
            X = np.array([self.records[i] for i in idx], np.float32)
            V = np.array([self.values[i] for i in idx], np.float32)
            if mirror:
                X = np.concatenate([X, np.flip(X, axis=2)])
                V = np.concatenate([V, np.flip(V, axis=1)])
            dev = self.nnet.device if hasattr(self.nnet, "device") else "cuda"
            return torch.from_numpy(np.ascontiguousarray(X)).to(dev), torch.from_numpy(np.ascontiguousarray(V)).to(dev), batch_size
        X, V = self._engine.records_gather(idx, mirror=mirror)
        return X, V, batch_size

    # agent.py:140-147
    def clear(self):
        if self._engine is not None:
            self._engine.search_clear()
            if self._records_on:
                self._engine.records_clear()
        if self.training and self._host_records:
            self.records = []
            self.values = []


class StubNet:
    """deterministic value function evaluated inside the engine (value from the plane key + obstacle mask)."""
    is_stub = True
