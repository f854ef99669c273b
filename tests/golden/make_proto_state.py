#!/usr/bin/env python
"""Write tests/golden/proto_state.json: the proto-shaped export (soccer2d_b200.proto_state) of one fixed snapshot
and of the player types drawn with seed 5, as JSON - the wire form json_format.ParseDict reads.

This export was checked against the reference's own generated service_pb2 and its ReachBall hooks
(sample_environments/reach_ball_env.py); tests/test_proto_state.py pins it, so that the check holds without the
reference.  With `--reference DIR` (a checkout of the reference) the check is run again before anything is written:
the reference parses both payloads and its state_to_observation / check_trainer_observation run on them.

Usage:  python tests/golden/make_proto_state.py [--reference DIR]
"""
import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for _p in (ROOT, os.path.join(ROOT, "gym-soccer-2d-env_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

SNAPSHOT_PLAYERS = ((-20.0, 4.0, 135.0, 1, 1), (10.0, -3.0, -45.0, 1, 2), (30.0, 0.0, 180.0, 2, 1))  # x, y, body, side, unum
TYPE_OF_PLAYER = [0, 7, 3]
PLAYER_TYPE_SEED = 5


def snapshot():
    from soccer2d_b200 import _abi
    s = _abi.EnvSnapshot()
    s.cycle, s.game_mode_type, s.game_mode_side, s.step_number, s.left_score, s.right_score = 57, 4, 2, 12, 1, 0
    s.ball_x, s.ball_y, s.ball_vx, s.ball_vy = 10.5, -3.25, 0.5, 0.125
    s.num_players = len(SNAPSHOT_PLAYERS)
    for j, (x, y, body, side, unum) in enumerate(SNAPSHOT_PLAYERS):
        p = s.players[j]
        p.x, p.y, p.vx, p.vy, p.body_direction = x, y, 0.25, -0.5, body
        p.stamina, p.effort, p.recovery, p.stamina_capacity, p.side, p.uniform_number = 7500.0, 0.9, 1.0, 120000.0, side, unum
    return s


def state_payload():
    """{"player": State seen by left player 1, "trainer": the trainer's State}, JSON-normalised"""
    from soccer2d_b200.proto_state import state_dict, trainer_state_dict
    snap = snapshot()
    payload = {"player": state_dict(snap, unum=1, side=1, type_of_player=TYPE_OF_PLAYER), "trainer": trainer_state_dict(snap)}
    return json.loads(json.dumps(payload))


def player_types_payload():
    """the 18 PlayerType messages of s2d_generate_player_types(seed 5), JSON-normalised"""
    import ctypes as C

    from soccer2d_b200 import _abi
    from soccer2d_b200.proto_state import player_type_dict
    lib = _abi.load()
    sp = _abi.ServerParam()
    assert lib.s2d_default_server_param(C.byref(sp)) == 0
    types = (_abi.PlayerType * 18)()
    assert lib.s2d_generate_player_types(PLAYER_TYPE_SEED, C.byref(sp), types, 18) == 0
    return json.loads(json.dumps([player_type_dict(k, types[k].as_dict(), sp) for k in range(18)]))


_REF_STATE = r"""
import json, logging, sys
shims, ref, payload = sys.argv[1], sys.argv[2], json.load(sys.stdin)
sys.path[:0] = [ref, shims]              # the reference's modules + stand-ins for gym / pyrusgeom only
from google.protobuf import json_format
import service_pb2 as pb2
import soccer_2d_env
soccer_2d_env.Soccer2DEnv.__init__ = lambda self, *a, **k: None      # no rcssserver / proxy processes offline
from sample_environments.reach_ball_env import ReachBallEnv
log = logging.getLogger("x"); log.disabled = True
state = json_format.ParseDict(payload["player"], pb2.State())
trainer = json_format.ParseDict(payload["trainer"], pb2.State())
wm = state.world_model
env = ReachBallEnv(render_mode=None, logger=log, log_dir="/tmp")
obs = env.state_to_observation(state)
env.step_number = 5
done, reward, info = env.check_trainer_observation(trainer)
print(json.dumps({
    "cycle": wm.cycle, "mode_is_kick_in": wm.game_mode_type == pb2.GameModeType.KickIn_,
    "mode_side_is_right": wm.game_mode_side == pb2.Side.RIGHT, "self_unum": wm.self.uniform_number,
    "self_side_is_left": wm.self.side == pb2.Side.LEFT, "stamina": wm.self.stamina, "n_mates": len(wm.teammates),
    "n_opps": len(wm.opponents), "left_score": wm.left_team_score, "ball_x": wm.ball.position.x, "ball_vy": wm.ball.velocity.y,
    "kickable_mate": wm.kickable_teammate_existance, "mate_unum": wm.teammates[0].uniform_number,
    "type_ids": [wm.self.type_id, wm.teammates[0].type_id, wm.opponents[0].type_id],
    "our_dict": sorted(wm.our_players_dict), "their_dict": sorted(wm.their_players_dict),
    "obs": [float(v) for v in obs], "done": bool(done), "reward": float(reward), "result": info["result"]}))
"""

_REF_TYPES = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
from google.protobuf import json_format
import service_pb2 as pb2
out = []
for d in json.load(sys.stdin):
    m = json_format.ParseDict(d, pb2.PlayerType())
    out.append([m.id, m.player_decay, m.kickable_area, m.real_speed_max, m.cycles_to_reach_max_speed])
print(json.dumps(out))
"""


def _run_reference(code, args, payload):
    """run `code` in a clean interpreter (the reference's module names - soccer_2d_env, sample_environments - are the
    same as this repository's host package, on purpose) and return its last line of JSON"""
    r = subprocess.run([sys.executable, "-c", code] + args, input=json.dumps(payload), capture_output=True, text=True,
                       env={**os.environ, "PYTHONPATH": ""})
    if r.returncode != 0:
        raise SystemExit(r.stderr[-2000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def check_against_reference(ref, state, types):
    from oracle import soccer2d_oracle as O
    got = _run_reference(_REF_STATE, [os.path.join(HERE, "_shims"), ref], state)
    assert got["cycle"] == 57 and got["mode_is_kick_in"] and got["mode_side_is_right"]
    assert got["self_unum"] == 1 and got["self_side_is_left"] and got["stamina"] == 7500.0
    assert (got["n_mates"], got["n_opps"], got["left_score"]) == (1, 1, 1)
    assert got["ball_x"] == 10.5 and got["ball_vy"] == 0.125
    assert got["kickable_mate"] and got["mate_unum"] == 2
    assert got["our_dict"] == [1, 2] and got["their_dict"] == [1] and got["type_ids"] == TYPE_OF_PLAYER
    want = O.build_obs(10.5, -3.25, 0.5, 0.125, -20.0, 4.0, 135.0)
    assert max(abs(a - b) for a, b in zip(got["obs"], want)) <= 1e-12
    d, rw, res, _, _ = O.check_trainer(O.ReachBallConfig(), 0.0, 0.0, 5, 10.5, -3.25, -20.0, 4.0, 135.0)
    assert (got["done"], got["result"]) == (d, O.RESULT_NAMES[res]) and abs(got["reward"] - rw) <= 1e-12 * abs(rw)
    got = _run_reference(_REF_TYPES, [ref], types)
    assert [g[0] for g in got] == list(range(18))
    for g, d in zip(got, types):  # the proto's float fields hold float32
        for v, key in zip(g[1:4], ("player_decay", "kickable_area", "real_speed_max")):
            assert abs(v - d[key]) <= 1e-6 * abs(d[key]), (g[0], key)
        assert g[4] == d["cycles_to_reach_max_speed"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", help="checkout of the reference project: check the export against it first")
    args = ap.parse_args()
    state, types = state_payload(), player_types_payload()
    if args.reference:
        check_against_reference(args.reference, state, types)
    data = {"_generated_by": "tests/golden/make_proto_state.py", "state": state, "player_types": types}
    path = os.path.join(HERE, "proto_state.json")
    with open(path, "w") as f:
        json.dump(data, f, indent=0, separators=(",", ":"))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
