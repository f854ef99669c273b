"""The built-in script of FULLGAME's scripted players, restated in Python from its specification in include/soccer2d.h
("FULLGAME scripted players") alone - not from the kernel or from the C restatement in tests/script_oracle.  Double
precision, libm.  Used with tests/fullgame_twin.py: the script's commands go into the action row, and the twin's
cycle steps the match; tests/test_scripted_twin.py compares that with the C oracle's f64 build one cycle ahead.

A command reaches the cycle as a proto-style float row {cmd, a, b, c}, as a command of the action buffer does: its
arguments are rounded to float32 here, as the f64 oracle's are."""
from __future__ import annotations

import math

import numpy as np

FORMATION = [(-50, 0), (-36, -20), (-36, -7), (-36, 7), (-36, 20), (-20, -24), (-20, -8), (-20, 8), (-20, 24), (-9, -10),
             (-9, 10)]  # F_k, left-team coordinates
PLAY_ON, AFTER_GOAL, BEFORE_KICK_OFF, TIME_OVER = 2, 8, 0, 1
LEFT, RIGHT = 1, 2
NONE, GOTO, INTERCEPT, CATCH, SMART_KICK = 0, 4, 10, 12, 13


def _in_own_penalty_area(x, y, left, half_length):
    """|x| >= L - 16.5 on the team's own side, |y| <= 20.16"""
    return (x <= -(half_length - 16.5) if left else x >= half_length - 16.5) and abs(y) <= 20.16


def _clamp(v, a):
    return max(-a, min(v, a))


def chasers(match, half_length):
    """{LEFT: index, RIGHT: index} (None where a side has nobody eligible): smallest squared distance to the ball, ties
    to the lower index; the keeper only with the ball in its own penalty area or as its side's only player"""
    n = match.n
    pps = n // 2
    bx, by = match.ball.x, match.ball.y
    best = {}
    for side, players in ((LEFT, range(0, pps)), (RIGHT, range(pps, n))):
        keeper = players[0]
        ranked = []
        for j in players:
            if j == keeper and pps > 1 and not _in_own_penalty_area(bx, by, side == LEFT, half_length):
                continue
            p = match.players[j]
            ranked.append(((bx - p.x) ** 2 + (by - p.y) ** 2, j))
        best[side] = min(ranked)[1] if ranked else None  # (tuples: equal distances fall back to the index)
    return best


def command(match, j, is_chaser, sp, psp, catch_ban):
    """rules 1-4 for scripted player j; `sp`: the ServerParam, `psp`: j's (its player type's kickable_margin);
    `catch_ban`: j's catch ban (keepers).  Returns [cmd, a, b, c] as float32."""
    n = match.n
    pps = n // 2
    left = j < pps
    side = LEFT if left else RIGHT
    sg = 1.0 if left else -1.0
    L, W = sp.pitch_half_length, sp.pitch_half_width
    post = sp.goal_width / 2 - 1
    p, ball = match.players[j], match.ball
    bxo, byo = sg * ball.x, sg * ball.y  # b' (own frame)
    keeper = j in (0, pps)
    mode = match.mode
    out = [NONE, 0.0, 0.0, 0.0]
    if mode in (AFTER_GOAL, BEFORE_KICK_OFF, TIME_OVER):
        pass                                                                                      # rule 1
    elif is_chaser and (mode == PLAY_ON or match.side == side):                                   # rule 2
        dx, dy = ball.x - p.x, ball.y - p.y
        d2 = dx * dx + dy * dy
        if mode == PLAY_ON and keeper and catch_ban == 0 and _in_own_penalty_area(ball.x, ball.y, left, L) and d2 <= 1.2 * 1.2:
            ang = math.degrees(math.atan2(dy, dx)) - p.body if (dx or dy) else -p.body
            while ang > 180.0:
                ang -= 360.0
            while ang < -180.0:
                ang += 360.0
            out = [CATCH, ang, 0.0, 0.0]                                                          # 2a
        elif math.sqrt(d2) <= psp.player_size + psp.ball_size + psp.kickable_margin:
            gx, gy = L - bxo, 0.0 - byo
            if gx * gx + gy * gy <= 25.0 ** 2:  # shoot: the far post seen from the kicker
                target, speed = (L, -post if sg * p.y >= 0 else post), sp.ball_speed_max
            else:                                # dribble: 8 m along the way to the goal centre
                g = math.hypot(gx, gy)
                target, speed = (bxo + 8.0 * gx / g, byo + 8.0 * gy / g), 1.0
            out = [SMART_KICK, sg * target[0], sg * target[1], speed]                             # 2b
        elif mode == PLAY_ON:
            out = [INTERCEPT, 0.0, 0.0, 0.0]                                                      # 2c
        else:
            out = [GOTO, ball.x, ball.y, 100.0]                                                   # 2d
    elif keeper:                                                                                  # rule 3
        out = [GOTO, sg * (-L + 2.5), sg * _clamp(0.3 * byo, post), 100.0]
    else:                                                                                         # rule 4
        fx, fy = FORMATION[j if left else j - pps]
        out = [GOTO, sg * _clamp(fx + 0.6 * bxo, L - 2.5), sg * _clamp(fy + 0.3 * byo, W - 2.0), 60.0]
    return np.array(out, np.float32)


def script_rows(match, actions, mask, sp, sps):
    """the action rows [np][4] of one cycle with the players of `mask` replaced by the script's commands (from the
    match as it stands, before the cycle)"""
    rows = np.array(actions, np.float32).reshape(match.n, 4).copy()
    who = chasers(match, sp.pitch_half_length)
    pps = match.n // 2
    for j in range(match.n):
        if (mask >> j) & 1:
            side = LEFT if j < pps else RIGHT
            ban = match.catch_ban[0 if j == 0 else 1] if j in (0, pps) else 0
            rows[j] = command(match, j, who[side] == j, sp, sps[j], ban)
    return rows
