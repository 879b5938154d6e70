"""TimerStat with the reference's semantics (utils/misc.py:39-90): sliding window of 10, `.mean`; `.total` sums
every sample, not only the window.

CudaTimerStat keeps the interface but measures DEVICE time: the learners only enqueue kernels inside the `with` block,
so a host clock would report launch overhead.  Events are recorded on the current stream around the section and read
back lazily by `.mean` -- the learners call it after the single device->host copy of an update, when the events have
completed, so no extra synchronisation is added (reference stats: mpg_learner.py:412,421,435-437; nadp.py:218-230)."""
import time

import numpy as np


class TimerStat:
    def __init__(self, window_size=10):
        self._window_size = window_size
        self._samples = []
        self._start_time = None
        self.count = 0
        self._total = 0.0

    def __enter__(self):
        assert self._start_time is None, 'concurrent updates not supported'
        self._start_time = time.time()

    def __exit__(self, type, value, tb):
        self.push(time.time() - self._start_time)
        self._start_time = None

    def push(self, dt):
        self._samples.append(dt)
        if len(self._samples) > self._window_size:
            self._samples.pop(0)
        self.count += 1
        self._total += dt

    @property
    def mean(self):
        return float(np.mean(self._samples)) if self._samples else 0.0

    @property
    def total(self):
        return self._total


class CudaTimerStat(TimerStat):
    """`with timer:` brackets a section of the current CUDA stream with events; `.mean` is in seconds like TimerStat."""

    def __init__(self, window_size=10):
        super().__init__(window_size)
        self._pending = []

    def __enter__(self):
        import torch
        assert self._start_time is None, 'concurrent updates not supported'
        self._start_time = torch.cuda.Event(enable_timing=True)
        self._start_time.record()

    def __exit__(self, type, value, tb):
        import torch
        end = torch.cuda.Event(enable_timing=True)
        end.record()
        self._pending.append((self._start_time, end))
        self._start_time = None

    def _resolve(self):
        for start, end in self._pending:
            end.synchronize()                       # already complete when read after the update's D2H copy
            self.push(start.elapsed_time(end) * 1e-3)
        self._pending = []

    @property
    def mean(self):
        self._resolve()
        return float(np.mean(self._samples)) if self._samples else 0.0

    @property
    def total(self):
        self._resolve()
        return self._total
