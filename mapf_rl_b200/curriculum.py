"""Curriculum — the reference's adaptive training set of (num_agents, map_length) settings (GlobalBuffer.stat_dict and its
growth rule in GlobalBuffer.stats, worker.py:73-82, 205-226; SURVEY.md §5).

Training starts on `config.init_set` (one agent on a 10 x 10 map, config.py:49).  Every finished episode of a counted
actor appends its `done` flag to a window of the last `window` results of its setting.  `advance()` (called by the
training loop, the way train.py:41-45 calls buffer.stats()) looks at every setting whose window is full: with at least
`pass_rate * window` successes it adds (n + 1, l) while n + 1 <= max_num_agents and (n, l + map_step) while
l < max_map_length.  A setting already present is not added again and nothing is ever removed.  `levels` keeps the
settings in insertion order: `BatchedEnvironment.reset(levels=...)` maps each slot's Philox draw onto that order.

The 200-episode window and the rule that only actors with id >= 10 count are recorded in SURVEY.md §5.  The other
defaults -- pass_rate 0.9, one agent more, five cells more -- are a reading of worker.py:205-226 / config.py that is not
confirmed against the reference here: they are constructor arguments.
"""
from __future__ import annotations

from collections import deque
from typing import Dict, Iterable, List, Tuple

from . import config

Level = Tuple[int, int]


class Curriculum:
    def __init__(self, init_set: Level = config.init_set, max_num_agents: int = config.max_num_agents,
                 max_map_length: int = config.max_map_length, window: int = 200, pass_rate: float = 0.9,
                 agent_step: int = 1, map_step: int = 5):
        self.max_num_agents, self.max_map_length = int(max_num_agents), int(max_map_length)
        self.window, self.pass_rate = int(window), float(pass_rate)
        self.agent_step, self.map_step = int(agent_step), int(map_step)
        self.stat_dict: Dict[Level, deque] = {}
        self._add(tuple(int(x) for x in init_set))

    def _add(self, level: Level):
        if level not in self.stat_dict:
            self.stat_dict[level] = deque(maxlen=self.window)

    @property
    def levels(self) -> List[Level]:
        """The current settings, in the order they were added."""
        return list(self.stat_dict)

    def record(self, num_agents: Iterable[int], map_length: Iterable[int], done: Iterable[bool]):
        """Append finished episodes' results: one (n, l, done) per episode.  A setting outside the current set (an episode
        that started before its level was dropped from a caller's list) is ignored."""
        for n, l, d in zip(num_agents, map_length, done):
            w = self.stat_dict.get((int(n), int(l)))
            if w is not None:
                w.append(bool(d))

    def advance(self) -> List[Level]:
        """The growth rule of GlobalBuffer.stats; returns the settings it added."""
        added = []
        need = self.pass_rate * self.window
        for (n, l), w in list(self.stat_dict.items()):
            if len(w) < self.window or sum(w) < need:
                continue
            nxt = []
            if n + self.agent_step <= self.max_num_agents:
                nxt.append((n + self.agent_step, l))
            if l < self.max_map_length:
                nxt.append((n, l + self.map_step))
            for level in nxt:
                if level not in self.stat_dict:
                    self._add(level)
                    added.append(level)
        return added
