"""CPU-only: the proto-shaped export (soccer2d_b200.proto_state) is the one the reference's own generated
service_pb2 parsed and its ReachBall hooks computed from (stored in tests/golden/proto_state.json; with a checkout of
the reference, tests/golden/make_proto_state.py --reference DIR runs that check again), and the fields those hooks read
carry what the kernels compute from."""
import json
import os

import pytest

import helpers as H
from golden import make_proto_state as G
from oracle import soccer2d_oracle as O
from soccer2d_b200.proto_state import state_dict


@pytest.fixture(scope="module")
def stored():
    with open(os.path.join(H.ROOT, "tests", "golden", "proto_state.json")) as f:
        return json.load(f)


def test_state_dict_parses_into_the_reference_proto_and_feeds_its_hooks(stored):
    payload = G.state_payload()
    assert payload == stored["state"]
    wm, me = payload["player"]["world_model"], payload["player"]["world_model"]["self"]
    assert wm["cycle"] == 57 and wm["game_mode_type"] == "KickIn_" and wm["game_mode_side"] == "RIGHT"
    assert me["uniform_number"] == 1 and me["side"] == "LEFT" and me["stamina"] == 7500.0
    assert (len(wm["teammates"]), len(wm["opponents"]), wm["left_team_score"]) == (1, 1, 1)
    assert wm["ball"]["position"]["x"] == 10.5 and wm["ball"]["velocity"]["y"] == 0.125
    assert wm["kickable_teammate_existance"] and wm["teammates"][0]["uniform_number"] == 2  # player 2 stands next to the ball
    assert sorted(map(int, wm["our_players_dict"])) == [1, 2] and sorted(map(int, wm["their_players_dict"])) == [1]
    assert [me["type_id"], wm["teammates"][0]["type_id"], wm["opponents"][0]["type_id"]] == G.TYPE_OF_PLAYER
    # the fields reach_ball_env.py's state_to_observation / check_trainer_observation read, through the formulas the
    # reference's hooks are pinned to (tests/golden/reach_ball_contract.json), give what the simulator computes from
    ball, pos = wm["ball"], me["position"]
    assert O.build_obs(ball["position"]["x"], ball["position"]["y"], ball["velocity"]["x"], ball["velocity"]["y"],
                       pos["x"], pos["y"], me["body_direction"]) == O.build_obs(10.5, -3.25, 0.5, 0.125, -20.0, 4.0, 135.0)
    tw = payload["trainer"]["world_model"]
    mate = tw["teammates"][0]
    assert O.check_trainer(O.ReachBallConfig(), 0.0, 0.0, 5, tw["ball"]["position"]["x"], tw["ball"]["position"]["y"],
                           mate["position"]["x"], mate["position"]["y"], mate["body_direction"]) == \
        O.check_trainer(O.ReachBallConfig(), 0.0, 0.0, 5, 10.5, -3.25, -20.0, 4.0, 135.0)
    with pytest.raises(ValueError):
        state_dict(G.snapshot(), unum=7, side=1)


def test_player_types_parse_into_the_reference_proto(stored):
    """the drawn player types, exported with the proto's field names, are the PlayerType messages the reference parsed"""
    types = G.player_types_payload()
    assert [t["id"] for t in types] == [t["id"] for t in stored["player_types"]] == list(range(18))
    for got, want in zip(types, stored["player_types"]):
        assert got.keys() == want.keys()
        for key, v in want.items():
            assert got[key] == (v if isinstance(v, int) else pytest.approx(v, rel=1e-12)), (got["id"], key)
    assert types[0]["player_decay"] == pytest.approx(0.4) and types[0]["kickable_area"] == pytest.approx(1.085)
    assert types[0]["real_speed_max"] == pytest.approx(1.0)
    assert all(0.95 < t["real_speed_max"] <= 1.05 and 1 <= t["cycles_to_reach_max_speed"] < 50 for t in types)
