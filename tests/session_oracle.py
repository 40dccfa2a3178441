"""Reference of a persistent search session (TEST INFRASTRUCTURE; DESIGN.md section 17) over tests/batch_oracle.py.

`SessionPlayer(evaluator, L)` is one BatchedPlayer kept across searches with noise off.  `search(history, nodes,
minibatches)` is calc_moves_probabilities with its tree reuse (the new root among the old root, its children and its
grandchildren, else a fresh root) and a develop_tree that runs minibatches while done < nodes and minibatches < cap,
each of k = min(L, nodes - done) descents; None is no limit.  It returns what the device posts: children, visits, W,
best move, PV, minibatches, collisions, the new simulations and the root's visits before the search.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

from oracle import mcts as om
from tests import batch_oracle as bo

f32 = om.f32


class SessionPlayer(bo.BatchedPlayer):
    def __init__(self, evaluator: om.Evaluator, search_batch: int, explore_factor: float = 1.41421):
        assert search_batch >= 2
        params = om.MctsParams(sim_num=2, explore_factor=explore_factor, temperature=om.TemperaturePolicy.from_config([[9999, 0.0]]))
        super().__init__(params, evaluator, om.SplitMix64(0), search_batch)
        self._nodes = math.inf
        self._cap = math.inf

    def new_game(self) -> None:
        self.root = None

    def _develop_tree(self, pos_history: Sequence) -> None:
        self.reused = sum(e.n for e in self.root.children)
        self.minibatches = self.collisions = 0
        self.new_sims = 0
        while self.new_sims < self._nodes and self.minibatches < self._cap:
            k = int(min(self.search_batch, self._nodes - self.new_sims))
            virtual: dict = {}
            claimed: set = set()
            descents = []
            for _ in range(k):
                path = self._select_virtual(virtual)
                leaf = path[-1][1].target if path else self.root
                if self._detect_repetition(pos_history, path):
                    descents.append((path, leaf, "score", f32(0.0)))
                elif leaf.position.is_finished():
                    descents.append((path, leaf, "score", f32(om.to_signed_one(leaf.position.status()[1]))))
                elif id(leaf) in claimed:
                    descents.append((path, leaf, "collision", None))
                else:
                    claimed.add(id(leaf))
                    descents.append((path, leaf, "leaf", None))
                for _, e in path:
                    virtual[id(e)] = virtual.get(id(e), 0) + 1
            evals = {id(leaf): self.evaluator.evaluate(leaf.position) for _, leaf, kind, _ in descents if kind == "leaf"}
            for path, leaf, kind, ev in descents:
                if kind == "collision":
                    self.collisions += 1
                    continue
                if kind == "leaf":
                    per_move, ev = evals[id(leaf)]
                    for m, p in per_move:
                        leaf.children.append(om._Edge(m, p, om._Node(leaf.position.moved_position(m))))
                for src, e in path:
                    e.n += 1
                    e.w = f32(e.w + (ev if src.position.turn == om.P1 else f32(-ev)))
                self.new_sims += 1
            self.minibatches += 1

    def search(self, history: Sequence, nodes: Optional[int] = None, minibatches: Optional[int] = None):
        """-> dict(moves, visits, w, best, pv, minibatches, collisions, simulations, reused) in the device's terms."""
        self._nodes = math.inf if nodes is None else nodes
        self._cap = math.inf if minibatches is None else minibatches
        probs = self.calc_moves_probabilities(history)
        best = self.choose_move_from_probabilities(history, probs)
        edges = list(reversed(self.root.children))
        pv, node = [], self.root
        while node.children and len(pv) < 16:
            top = max(c.n for c in node.children)
            e = next(c for c in node.children if c.n == top)
            pv.append(e.m)
            node = e.target
        return dict(moves=[e.m for e in edges], visits=[e.n for e in edges], w=[e.w for e in edges], best=best, pv=pv, minibatches=self.minibatches,
                    collisions=self.collisions, simulations=self.new_sims, reused=self.reused)
