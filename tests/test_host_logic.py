"""Host-side logic of the drop-in (no GPU): action decoding, info dicts, shard layout."""
import numpy as np
import pytest


def test_discrete_to_action():  # tests/test_rl_env_wrapper.py:25 of the reference
    from inversus_b200 import discrete_to_action
    a = discrete_to_action(0)
    assert a.type == "none" and a.direction is None
    a = discrete_to_action(1)
    assert a.type == "move" and a.direction == "up"
    a = discrete_to_action(5)
    assert a.type == "shoot" and a.direction == "up"
    a = discrete_to_action(9)
    assert a.type == "charge_shoot" and a.direction == "up"
    assert [discrete_to_action(i).direction for i in (1, 2, 3, 4)] == ["up", "right", "down", "left"]
    assert [discrete_to_action(i).direction for i in (9, 10, 11, 12)] == ["up", "right", "down", "left"]
    for bad in (-1, 13, 99):
        with pytest.raises(ValueError, match="Invalid action_id"):
            discrete_to_action(bad)


def test_action_table_agrees_with_the_live_reference():
    from ref_harness import SKIP_REASON, import_reference, reference_available
    if not reference_available():
        pytest.skip(SKIP_REASON)
    ew = import_reference()
    from inversus_b200 import discrete_to_action
    for i in range(13):
        r, m = ew.discrete_to_action(i), discrete_to_action(i)
        assert r.type.value == m.type
        assert (r.direction.value if r.direction else None) == m.direction


def test_info_list_behaves_like_a_list_of_dicts():
    from inversus_b200 import InfoList
    il = InfoList(np.array([0, 1 | 4, 2 | 8], np.uint8), np.array([3, 17, 500], np.int32), np.array([0.5, 11.0, -2.1]))
    assert len(il) == 3
    assert il[1] == {"landed_hit": True, "got_hit": False, "win": True, "lose": False,
                     "episode_steps": 17, "episode_return": 11.0}
    assert il[2]["lose"] and il[2]["got_hit"] and not il[2]["win"]
    assert il[0].get("episode_return", 0.0) == 0.5           # training.py:142 access pattern
    assert [d["episode_steps"] for d in il] == [3, 17, 500]
    assert isinstance(il[1]["win"], bool) and isinstance(il[1]["episode_steps"], int)


def test_shard_ranges_partition_the_env_ids():
    from inversus_b200.sharding import shard_range
    for total in (1, 7, 8, 1000, 8_388_608):
        for world in (1, 2, 3, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0
            assert sum(c for _, c in spans) == total
            for (f0, c0), (f1, _) in zip(spans, spans[1:]):
                assert f0 + c0 == f1
            assert max(c for _, c in spans) - min(c for _, c in spans) <= 1
    with pytest.raises(ValueError):
        shard_range(10, 4, 4)
