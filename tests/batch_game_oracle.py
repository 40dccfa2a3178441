"""Reference of self-play and match games with minibatched searches (TEST INFRASTRUCTURE; DESIGN.md section 16).

`play_from` is oracle/mcts.py's game loop with a tests/batch_oracle.py `BatchedPlayer(L)` for each side.  With L = 1 on
both sides it is the oracle's play_game started after the given history.
"""
from __future__ import annotations

from oracle import mcts as om
from tests.batch_oracle import BatchedPlayer


def play_from(game_idx: int, history, params1: om.MctsParams, params2: om.MctsParams, eval1: om.Evaluator, eval2: om.Evaluator,
              base_seed: int, max_moves: int = 0, search_batch=(1, 1)):
    """oracle/mcts.py's play_game (self_play.rs:179-246) with a BatchedPlayer per side (search_batch[0] for player 1 of
    game 0, i.e. model 1 / A; search_batch[1] for model 2 / B), started after `history` (an opening, oldest first; the
    initial position alone is self-play).  Repetition counts the opening's positions, the temperature policy gets the
    history from the opening position on, and max_moves counts the moves played after it.  Returns (GameRecord,
    player1, player2): the players carry each side's minibatches and collisions."""
    rng = om.SplitMix64(om.game_seed(base_seed, game_idx))
    player1 = BatchedPlayer(params1, eval1, rng, search_batch[0])
    player2 = BatchedPlayer(params2, eval2, rng, search_batch[1])
    history = list(history)
    base = len(history) - 1
    entries, moves = [], []
    limit = getattr(type(history[0]), "REPETITION_LIMIT", None)
    seen = None
    if limit:
        seen = {}
        for p in history:
            seen[p] = seen.get(p, 0) + 1
    while True:
        st, winner = history[-1].status()
        if seen is not None and seen[history[-1]] >= limit:
            st, winner = "finished", None
        if st != "finished" and max_moves and len(moves) >= max_moves:
            st, winner = "finished", None
        if st == "finished":
            break
        who = history[-1].turn
        if game_idx % 2 == 1:
            who = om.opposite(who)
        player = player1 if who == om.P1 else player2
        probs = player.calc_moves_probabilities(history)
        mv = player.choose_move_from_probabilities(history[base:], probs)
        entries.append((history[-1], probs))
        moves.append(mv)
        history.append(history[-1].moved_position(mv))
        if seen is not None:
            seen[history[-1]] = seen.get(history[-1], 0) + 1
    rec = om.GameRecord(game_idx, winner, moves, entries, player1.sims_done + player2.sims_done,
                        player1.terminal_leaves + player2.terminal_leaves, player1.repetition_hits + player2.repetition_hits)
    return rec, player1, player2
