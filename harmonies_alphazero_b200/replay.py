"""GPU-resident replay ring (SURVEY.md §8 f2): the consumer side of self-play.

The reference keeps a ``deque(maxlen)`` of CPU tensor 4-tuples (6,064 B per example) that is
pickled whole every iteration (buffer.py:7-67, trainer.py:127,146-153,250-254).  Here the
examples stay packed on the device — 128 B state + 143 x int16 visit counts + z = 418 B — and
a training batch is produced on the fly by hz_encode: no H2D copy and no DataLoader on the
training path.  ``to_reference_buffer`` exports the reference's exact structure so that
``buffer.save_buffer`` / ``ReplayBufferDataset`` keep working.
"""

from collections import deque

import torch

from . import batched as hb


class ReplayRing:
    def __init__(self, capacity, device="cuda"):
        self.capacity, self.device = int(capacity), torch.device(device)
        self.states = torch.zeros((self.capacity, 32), dtype=torch.int32, device=self.device)
        self.visits = torch.zeros((self.capacity, 143), dtype=torch.int16, device=self.device)
        self.z = torch.zeros(self.capacity, dtype=torch.float32, device=self.device)
        self.size = 0      # valid examples
        self.head = 0      # next write position (oldest example once full) — deque(maxlen) semantics

    def __len__(self):
        return self.size

    def extend(self, traj):
        """Append a Trajectories set; the oldest examples are overwritten when full
        (``deque.extend`` with ``maxlen``, trainer.py:127)."""
        n = len(traj)
        if n == 0:
            return
        S, V, Z = traj.states.to(self.device), traj.visits.to(self.device), traj.z.to(self.device)
        if n >= self.capacity:                      # only the newest `capacity` examples survive
            S, V, Z, n = S[-self.capacity:], V[-self.capacity:], Z[-self.capacity:], self.capacity
        idx = (self.head + torch.arange(n, device=self.device)) % self.capacity
        self.states[idx], self.visits[idx], self.z[idx] = S, V, Z
        self.head = (self.head + n) % self.capacity
        self.size = min(self.capacity, self.size + n)

    def _ordered_index(self):
        """indices oldest -> newest (the iteration order of the reference's deque)"""
        if self.size < self.capacity:
            return torch.arange(self.size, device=self.device)
        return (self.head + torch.arange(self.capacity, device=self.device)) % self.capacity

    def sample(self, batch_size, generator=None, dtype=torch.float32, augment=None):
        """A training batch (board [B,38,5,7], global [B,42], pi [B,143], z [B,1]) on the
        device: uniform sampling with replacement + hz_encode of the packed states.
        augment: None, "board" or "full": every row is mapped by its own uniform group element g
        (drawn from ``generator`` after the indices): encode(T_g(state)), T_g(visits) normalised, z."""
        if self.size == 0:
            raise ValueError("replay ring is empty")
        idx = torch.randint(0, self.size, (batch_size,), device=self.device, generator=generator)
        if self.size == self.capacity:
            idx = (self.head + idx) % self.capacity
        return self._batch(idx, dtype, self._elements(idx.numel(), augment, generator))

    def _elements(self, n, augment, generator):
        if augment is None:                      # no draw: the generator advances exactly as without augmentation
            return None
        from .symmetry import random_elements

        return random_elements(n, augment, device=self.device, generator=generator)

    def _batch(self, idx, dtype=torch.float32, sym=None):
        states, visits = self.states[idx].contiguous(), self.visits[idx]
        if sym is not None:
            from .symmetry import transform_actions, transform_states

            visits = transform_actions(visits.contiguous(), sym, states)
            transform_states(states, sym, out=states)
        board, glob = hb.encode(states, dtype=dtype)
        v = visits.to(torch.float64)
        pi = (v / v.sum(dim=1, keepdim=True).clamp_min(1)).to(torch.float32)      # trainer.py:535
        return board, glob, pi, self.z[idx].view(-1, 1)

    def epoch(self, batch_size, shuffle=True, generator=None, augment=None):
        """Iterate once over the whole buffer in batches (DataLoader(ReplayBufferDataset(...),
        shuffle=True), trainer.py:146-153).  augment: as for ``sample`` (one element per row and batch)."""
        order = self._ordered_index()
        if shuffle:
            order = order[torch.randperm(order.numel(), device=self.device, generator=generator)]
        for i in range(0, order.numel(), batch_size):
            part = order[i:i + batch_size]
            yield self._batch(part, sym=self._elements(part.numel(), augment, generator))

    def to_reference_buffer(self):
        """deque(maxlen=capacity) of (board, global, pi, z) CPU tensors, oldest first — the
        object buffer.save_buffer pickles and ReplayBufferDataset wraps (buffer.py:7-67)."""
        out = deque(maxlen=self.capacity)
        order = self._ordered_index()
        for i in range(0, order.numel(), 8192):
            fields = [t.cpu().numpy() for t in self._batch(order[i:i + 8192])]
            # every tensor owns its storage (a view would pull its whole batch into the pickle)
            out.extend(tuple(torch.from_numpy(f[k].copy()) for f in fields) for k in range(fields[0].shape[0]))
        return out

    def state_dict(self):
        order = self._ordered_index()
        return {"states": self.states[order].cpu(), "visits": self.visits[order].cpu(), "z": self.z[order].cpu(),
                "capacity": self.capacity}

    def load_state_dict(self, sd):
        n = min(self.capacity, sd["states"].shape[0])
        self.states[:n] = sd["states"][-n:].to(self.device)
        self.visits[:n] = sd["visits"][-n:].to(self.device)
        self.z[:n] = sd["z"][-n:].to(self.device)
        self.size, self.head = n, n % self.capacity
