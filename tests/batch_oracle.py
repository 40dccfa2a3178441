"""Reference of the minibatched search (TEST INFRASTRUCTURE; DESIGN.md section 15) over oracle/mcts.py's MctsPlayer.

`BatchedPlayer(params, evaluator, rng, search_batch)` is an MctsPlayer whose develop_tree, for search_batch > 1, runs
minibatches of descents under virtual loss, written as plainly and sequentially as the definition:

1. k = min(L, sim_num - sims_done) descents in order on a frozen tree; each edge is seen with n' = n + v and
   w' = f32(w - f32(v)), v the descents of this minibatch that took it.  A descent ends where _select ends and is a
   repetition (value 0), a terminal (the winner's +-1), a new leaf (the first descent to end on that unexpanded node)
   or a collision (a later one), then adds 1 to v on every edge of its path.
2. Every new leaf is evaluated once.
3. In descent order: a new leaf gets its children, then it and every repetition / terminal descent is backed up as
   _develop_tree backs up; a collision does nothing.  sims_done grows by the non-collisions.

With search_batch 1 it is MctsPlayer, untouched.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np

from oracle import mcts as om

f32 = om.f32


class BatchedPlayer(om.MctsPlayer):
    def __init__(self, params: om.MctsParams, evaluator: om.Evaluator, rng: om.SplitMix64, search_batch: int = 1):
        super().__init__(params, evaluator, rng)
        assert search_batch >= 1
        self.search_batch = search_batch
        self.minibatches = 0
        self.collisions = 0
        self.choices: List[List[int]] = []  # per minibatch: the root child (insertion index) each descent took, -1 = none
        self.kinds: List[List[Tuple[str, int]]] = []  # per minibatch: (kind, id of the node it ended on) of each descent

    def _heuristic_virtual(self, e, v: int, parent_simcount: int) -> np.float32:
        n = e.n + v
        w = f32(e.w - f32(v))
        exploit = f32(0.0) if n == 0 else f32(w / f32(n))
        explore = f32(f32(self.explore_factor * e.init_score) * f32(np.sqrt(f32(parent_simcount)) / f32(1 + n)))
        return f32(exploit + explore)

    def _select_virtual(self, virtual: dict) -> List[Tuple[object, object]]:
        path = []
        node = self.root
        while True:
            if node.position.is_finished() or not node.children:
                return path
            simcount = 1 + sum(e.n + virtual.get(id(e), 0) for e in node.children)
            best, best_val = None, None
            for e in om._edges(node):
                v = self._heuristic_virtual(e, virtual.get(id(e), 0), simcount)
                if best is None or not (v < best_val):  # max_by keeps the LAST maximum; NaN compares Equal
                    best, best_val = e, v
            path.append((node, best))
            node = best.target

    def _develop_tree(self, pos_history: Sequence) -> None:
        if self.search_batch == 1:
            super()._develop_tree(pos_history)
            self.minibatches += self.p.sim_num
            return
        assert self.p.sim_num > 1
        done = 0
        while done < self.p.sim_num:
            k = min(self.search_batch, self.p.sim_num - done)
            virtual: dict = {}
            claimed: set = set()
            descents = []  # (path, leaf, kind, value); kind: "leaf" | "score" | "collision"
            for _ in range(k):
                path = self._select_virtual(virtual)
                leaf = path[-1][1].target if path else self.root
                if self._detect_repetition(pos_history, path):
                    descents.append((path, leaf, "score", f32(0.0)))
                    self.repetition_hits += 1
                elif leaf.position.is_finished():
                    descents.append((path, leaf, "score", f32(om.to_signed_one(leaf.position.status()[1]))))
                elif id(leaf) in claimed:
                    descents.append((path, leaf, "collision", None))
                else:
                    claimed.add(id(leaf))
                    descents.append((path, leaf, "leaf", None))
                for _, e in path:
                    virtual[id(e)] = virtual.get(id(e), 0) + 1
            self.choices.append([self.root.children.index(p[0][1]) if p else -1 for p, _, _, _ in descents])
            self.kinds.append([(kind, id(leaf)) for _, leaf, kind, _ in descents])
            evals = {id(leaf): self.evaluator.evaluate(leaf.position) for _, leaf, kind, _ in descents if kind == "leaf"}
            for path, leaf, kind, ev in descents:
                if kind == "collision":
                    self.collisions += 1
                    continue
                if kind == "leaf":
                    per_move, ev = evals[id(leaf)]
                    for m, p in per_move:  # create_children, mod.rs:246-262
                        leaf.children.append(om._Edge(m, p, om._Node(leaf.position.moved_position(m))))
                    if leaf is self.root:
                        self._add_dirichlet_noise(leaf)
                else:
                    self.terminal_leaves += 1
                for src, e in path:  # backpropagate, mod.rs:270-281
                    e.n += 1
                    e.w = f32(e.w + (ev if src.position.turn == om.P1 else f32(-ev)))
                self.sims_done += 1
                done += 1
            self.minibatches += 1


def search(history, evaluator, sim_num: int, search_batch: int, explore_factor: float = 1.41421):
    """A fresh player's search of history[-1] with noise off: (player, children moves in edges() order, visits, W, best
    move, PV) -- the PV as the device posts it (most visits, equal counts to the smallest insertion index, <= 16 plies)."""
    params = om.MctsParams(sim_num=sim_num, explore_factor=explore_factor, temperature=om.TemperaturePolicy.from_config([[9999, 0.0]]))
    player = BatchedPlayer(params, evaluator, om.SplitMix64(0), search_batch)
    probs = player.calc_moves_probabilities(history)
    best = player.choose_move_from_probabilities(history, probs)
    edges = list(reversed(player.root.children))
    pv, node = [], player.root
    while node.children and len(pv) < 16:
        top = max(c.n for c in node.children)
        e = next(c for c in node.children if c.n == top)
        pv.append(e.m)
        node = e.target
    return player, [e.m for e in edges], [e.n for e in edges], [e.w for e in edges], best, pv
