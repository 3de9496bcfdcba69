"""CPU ORACLE for the observation normaliser — test infrastructure, NOT product code.

Restates RLlib's ``MeanStdFilter`` / ``RunningStat`` (third party; ray is unpinned in the reference's
requirements.txt:15 and not installable here, so this is written from the published algorithm -- Welford's
recurrence, ``var = S / (n - 1)`` for n > 1 else ``mean ** 2``, ``(x - mean) / (std + 1e-8)``, clip -- PARITY UNPINNED
vs RLlib).  ``SequentialFilter`` is the reference-style filter (one observation at a time, statistics updated before the
observation is normalised); ``BatchSyncFilter`` is the semantics of pnr_filter_apply / pnr_filter_sync (statistics
pushed per batch, normalisation with the statistics of the last synchronisation).  Both take RLlib's ``demean`` / ``destd``
flags: the mean is subtracted only if ``demean``, the result divided by ``std + 1e-8`` only if ``destd``; the running
statistics are kept either way."""
from __future__ import annotations

import numpy as np


class RunningStat:
    def __init__(self, dim):
        self.n, self.M, self.S = 0, np.zeros(dim), np.zeros(dim)

    def push(self, x):
        x = np.asarray(x, np.float64)
        self.n += 1
        if self.n == 1:
            self.M = x.copy()
        else:
            delta = x - self.M
            self.M = self.M + delta / self.n
            self.S = self.S + delta * delta * (self.n - 1) / self.n

    @property
    def var(self):
        return self.S / (self.n - 1) if self.n > 1 else np.square(self.M)

    @property
    def std(self):
        return np.sqrt(self.var)


class SequentialFilter:
    def __init__(self, dim, clip=10.0, demean=True, destd=True):
        self.rs, self.clip, self.demean, self.destd = RunningStat(dim), clip, demean, destd

    def __call__(self, x, update=True):
        x = np.asarray(x, np.float64)
        if update:
            self.rs.push(x)
        y = x - self.rs.M if self.demean else x
        if self.destd:
            y = y / (self.rs.std + 1e-8)
        return np.clip(y, -self.clip, self.clip)


class BatchSyncFilter:
    def __init__(self, dim, clip=10.0, demean=True, destd=True):
        self.rs, self.clip, self.demean, self.destd = RunningStat(dim), clip, demean, destd
        # before the first synchronisation nothing has been pushed: the filter is the identity (mean 0, scale 1), as an
        # RLlib filter that has seen no sample never normalises anything
        self.applied_mean, self.applied_std = np.zeros(dim), np.ones(dim) - 1e-8
        self.pending = []

    def __call__(self, batch, update=True):
        batch = np.asarray(batch, np.float64)
        if update:
            self.pending.append(batch.copy())
        y = batch                                   # the device applies float32 statistics
        if self.demean:
            y = y - self.applied_mean.astype(np.float32).astype(np.float64)
        if self.destd:
            y = y * (1.0 / (self.applied_std + 1e-8)).astype(np.float32).astype(np.float64)
        return np.clip(y, -self.clip, self.clip)

    def sync(self):
        for b in self.pending:
            for row in b:
                self.rs.push(row)
        self.pending = []
        if self.rs.n:
            self.applied_mean, self.applied_std = self.rs.M.copy(), self.rs.std.copy()
