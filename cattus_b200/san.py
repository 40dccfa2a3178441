"""Standard algebraic notation and EPD records for chess positions given as FEN + moves.

Legal moves, check and mate come from the engine's own rules (`cattus_b200_chess_position`, include/cattus_b200_chess.h);
the board is read from the FEN's placement field and the moves played on it.  Moves are the library's encoding
from | to << 6 | promotion << 12 in real board coordinates (promotion 1 q, 2 n, 3 r, 4 b).
"""
from __future__ import annotations

import ctypes as C
import re
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

from . import _lib

START_FEN = "rnbqkbnr/pppppppp/8/8/8/8/PPPPPPPP/RNBQKBNR w KQkq -"
_PROMO_CH = {1: "Q", 2: "N", 3: "R", 4: "B"}
_SAN_RE = re.compile(r"^([NBRQK])?([a-h])?([1-8])?x?([a-h][1-8])(?:=?([NBRQnbrq]))?$")


def _sq(s: int) -> str:
    return "abcdefgh"[s & 7] + "12345678"[s >> 3]


def position_info(fen: Optional[str], moves: Sequence[int] = ()) -> _lib.ChessInfo:
    lib = _lib.load()
    info = _lib.ChessInfo()
    info.struct_size = C.sizeof(_lib.ChessInfo)
    arr = (C.c_uint16 * max(1, len(moves)))(*moves)
    rc = lib.cattus_b200_chess_position((fen or START_FEN).encode(), arr, len(moves), C.byref(info))
    if rc != 0:
        raise ValueError((lib.cattus_b200_chess_last_error() or b"").decode(errors="replace"))
    return info


def legal_moves(fen: Optional[str], moves: Sequence[int] = ()) -> List[int]:
    info = position_info(fen, moves)
    return list(info.moves[: info.n_legal])


def board(fen: Optional[str], moves: Sequence[int] = ()) -> Dict[int, str]:
    """square -> piece letter (upper case white) after the moves."""
    placement = (fen or START_FEN).split()[0]
    b: Dict[int, str] = {}
    for r, row in enumerate(placement.split("/")):
        f = 0
        for ch in row:
            if ch.isdigit():
                f += int(ch)
            else:
                b[(7 - r) * 8 + f] = ch
                f += 1
    for m in moves:
        fr, to, promo = m & 63, (m >> 6) & 63, m >> 12
        pc = b.pop(fr)
        if pc in "Pp" and (fr & 7) != (to & 7) and to not in b:  # en passant: the captured pawn sits beside the origin
            b.pop((fr & 56) | (to & 7), None)
        if pc in "Kk" and abs((fr & 7) - (to & 7)) == 2:  # castling: the rook jumps over the king
            rook_from, rook_to = ((fr & 56) | 7, (fr & 56) | 5) if (to & 7) == 6 else ((fr & 56), (fr & 56) | 3)
            b[rook_to] = b.pop(rook_from)
        if promo:
            pc = _PROMO_CH[promo] if pc == "P" else _PROMO_CH[promo].lower()
        b[to] = pc
    return b


def _san_body(b: Dict[int, str], legal: Sequence[int], m: int) -> str:
    fr, to, promo = m & 63, (m >> 6) & 63, m >> 12
    pc = b[fr].upper()
    if pc == "K" and abs((fr & 7) - (to & 7)) == 2:
        return "O-O" if (to & 7) == 6 else "O-O-O"
    capture = to in b or (pc == "P" and (fr & 7) != (to & 7))
    if pc == "P":
        s = ("abcdefgh"[fr & 7] + "x" if capture else "") + _sq(to)
        return s + ("=" + _PROMO_CH[promo] if promo else "")
    rivals = [o & 63 for o in legal if o != m and (o >> 6) & 63 == to and b[o & 63].upper() == pc]
    dis = ""
    if rivals:
        if all((r & 7) != (fr & 7) for r in rivals):
            dis = "abcdefgh"[fr & 7]
        elif all((r >> 3) != (fr >> 3) for r in rivals):
            dis = "12345678"[fr >> 3]
        else:
            dis = _sq(fr)
    return pc + dis + ("x" if capture else "") + _sq(to)


def move_to_san(fen: Optional[str], moves: Sequence[int], m: int) -> str:
    """SAN of move m in the position fen + moves, with + for check and # for mate."""
    legal = legal_moves(fen, moves)
    if m not in legal:
        raise ValueError(f"move {m} is not legal here")
    after = position_info(fen, list(moves) + [m])
    suffix = ("#" if after.n_legal == 0 else "+") if after.in_check else ""
    return _san_body(board(fen, moves), legal, m) + suffix


def san_line(fen: Optional[str], moves: Sequence[int], line: Sequence[int]) -> List[str]:
    """SAN of each move of `line` played in turn from fen + moves."""
    out, played = [], list(moves)
    for m in line:
        out.append(move_to_san(fen, played, m))
        played.append(m)
    return out


def move_from_san(fen: Optional[str], moves: Sequence[int], san: str) -> int:
    """The legal move a SAN names: piece letter, disambiguation, x, =Q, O-O / O-O-O (or 0-0); + # ! ? are ignored."""
    s = san.strip().rstrip("+#!?").replace("0", "O")
    legal = legal_moves(fen, moves)
    b = board(fen, moves)
    if s in ("O-O", "O-O-O"):
        want = 6 if s == "O-O" else 2
        hits = [m for m in legal if b[m & 63].upper() == "K" and abs((m & 7) - ((m >> 6) & 7)) == 2 and ((m >> 6) & 7) == want]
    else:
        g = _SAN_RE.match(s)
        if not g:
            raise ValueError(f"not a SAN move: {san!r}")
        piece, ff, fr, dest, promo = g.groups()
        piece = piece or "P"
        to = "abcdefgh".index(dest[0]) + 8 * (int(dest[1]) - 1)
        pnum = {"Q": 1, "N": 2, "R": 3, "B": 4}[promo.upper()] if promo else 0
        hits = [m for m in legal if (m >> 6) & 63 == to and b[m & 63].upper() == piece and (m >> 12) == pnum
                and (ff is None or "abcdefgh"[m & 7] == ff) and (fr is None or "12345678"[(m & 63) >> 3] == fr)]
    if len(hits) != 1:
        raise ValueError(f"SAN {san!r} names {'no' if not hits else 'more than one'} legal move here")
    return hits[0]


@dataclass
class EpdRecord:
    fen: str                                  # the four FEN fields
    ops: Dict[str, List[str]] = field(default_factory=dict)

    @property
    def id(self) -> Optional[str]:
        v = self.ops.get("id")
        return " ".join(v) if v else None


def parse_epd(line: str) -> EpdRecord:
    """`<placement> <side> <castling> <en passant> op operands; op operands; ...` -- operands split on blanks, a quoted
    string is one operand."""
    fields = line.strip().split(None, 4)
    if len(fields) < 4:
        raise ValueError(f"an EPD record needs four FEN fields: {line!r}")
    rec = EpdRecord(" ".join(fields[:4]))
    rest = fields[4] if len(fields) > 4 else ""
    for op in _split_ops(rest):
        toks = re.findall(r'"[^"]*"|\S+', op)
        if toks:
            rec.ops[toks[0]] = [t[1:-1] if t.startswith('"') else t for t in toks[1:]]
    return rec


def _split_ops(s: str) -> List[str]:
    out, cur, quoted = [], [], False
    for ch in s:
        if ch == '"':
            quoted = not quoted
        if ch == ";" and not quoted:
            out.append("".join(cur).strip())
            cur = []
        else:
            cur.append(ch)
    if "".join(cur).strip():
        out.append("".join(cur).strip())
    return out


_RESULTS = {None: "1/2-1/2", 0: "1/2-1/2", 1: "1-0", 2: "0-1"}
# PGN's Termination tag has a fixed vocabulary: a game the rules or a repetition ended is "normal", one cut off at
# max_moves is "adjudication"; a comment after the last move says which
_TERMINATION_TAG = {"rules": "normal", "repetition": "normal", "max_moves": "adjudication"}
_TERMINATION_TEXT = {"rules": None, "repetition": "threefold repetition", "max_moves": "draw adjudicated at max_moves"}


def pgn_game(fen: Optional[str], opening: Sequence[int], moves: Sequence[int], winner: Optional[int], termination: str, *, white: str = "?",
             black: str = "?", event: str = "?", round_: str = "?") -> str:
    """One game in PGN: the Seven Tag Roster, SetUp / FEN for a FEN opening and Termination; the movetext holds the
    opening's moves, then the game's, numbered from the FEN's fullmove field (1 without one), and ends with the result.
    winner: None / 0 draw, 1 white, 2 black."""
    result = _RESULTS[winner]
    tags = [("Event", event), ("Site", "?"), ("Date", "????.??.??"), ("Round", round_), ("White", white), ("Black", black), ("Result", result)]
    if fen is not None:
        tags += [("SetUp", "1"), ("FEN", fen)]
    tags.append(("Termination", _TERMINATION_TAG[termination]))
    fields = (fen or START_FEN).split()
    number = int(fields[5]) if len(fields) > 5 else 1
    black_to_move = fields[1] == "b"
    toks, played = [], []
    for k, m in enumerate(list(opening) + list(moves)):
        if not black_to_move:
            toks.append(f"{number}.")
        elif k == 0:
            toks.append(f"{number}...")
        toks.append(move_to_san(fen, played, m))
        played.append(m)
        if black_to_move:
            number += 1
        black_to_move = not black_to_move
    note = _TERMINATION_TEXT[termination]
    if note:
        toks.append("{" + note + "}")
    toks.append(result)
    lines, cur = [], ""
    for t in toks:  # PGN export format: lines of at most 80 characters
        if cur and len(cur) + 1 + len(t) > 79:
            lines.append(cur)
            cur = t
        else:
            cur = f"{cur} {t}" if cur else t
    lines.append(cur)
    return "".join(f'[{k} "{v}"]\n' for k, v in tags) + "\n" + "\n".join(lines) + "\n"


def parse_fen_line(line: str) -> Tuple[Optional[str], List[str]]:
    """`<FEN> [moves m1 m2 ...]` or `startpos [moves ...]` -> (fen or None, LAN moves)."""
    head, _, tail = line.strip().partition(" moves")
    head = head.strip()
    fen = None if head in ("", "startpos") else head
    return fen, tail.split()
