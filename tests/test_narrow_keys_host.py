"""CPU-only checks of narrow (uint8 / int8) keys: the `key_dtypes` validation, which refuses before any row is stored (no CUDA call is
made), and the exactness rule of stored values (no silent wrap)."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def rm():
    import __graft_entry__ as g
    g.build()  # the mirror loads libfdql.so even before its first row
    from fastdeepqlearning_b200.Replay import replay_memory
    return replay_memory


WIDTHS = {"obs": 12, "action": 3, "achieved_goal": 4, "desired_goal": 4, "reward": 1, "episode_done": 1, "note": 1}


@pytest.mark.parametrize("key_dtypes,match", [
    ({"nope": "uint8"}, "not a key"),
    ({"reward": "uint8"}, "scalar or role"),
    ({"note": "uint8"}, "scalar or role"),          # role-less but width 1
    ({"achieved_goal": "int8"}, "scalar or role"),
    ({"virtual_rewards": "uint8"}, "virtual key"),
    ({"obs": "float16"}, "only uint8 and int8"),
    ({"obs": "int16"}, "only uint8 and int8"),
    ({"obs": "no-such-type"}, "only uint8 and int8"),
])
def test_key_dtypes_refused_before_any_row(rm, key_dtypes, match):
    widths = dict(WIDTHS, virtual_rewards=3)
    r = rm.ReplayMemory(64, 4, 2, device="cuda:0", key_dtypes=key_dtypes)
    with pytest.raises(ValueError, match=match):
        r._jit_initialize(widths)
    assert r._h is None and r._narrow == {}


@pytest.mark.parametrize("dt", ["uint8", "int8", np.uint8, np.int8, np.dtype("int8")])
def test_dtype_spellings(rm, dt):
    import torch
    want = torch.uint8 if np.dtype(dt) == np.uint8 else torch.int8
    assert rm._narrow_dtype("k", dt) is want
    assert rm._narrow_dtype("k", want) is want


def test_exact_values_only(rm):
    import torch
    u8, i8 = torch.uint8, torch.int8
    ok = rm._exact_narrow("k", np.array([0.0, 255.0, 17.0]), u8)
    assert ok.dtype == np.uint8 and ok.tolist() == [0, 255, 17]
    assert rm._exact_narrow("k", np.array([-128, 127]), i8).tolist() == [-128, 127]
    assert rm._exact_narrow("k", np.array([True, False]), u8).tolist() == [1, 0]
    frame = np.arange(256, dtype=np.uint8)
    assert rm._exact_narrow("k", frame, u8) is frame  # already the storage type: no copy
    for bad, dt in ((256.0, u8), (-1, u8), (0.5, u8), (float("nan"), u8), (float("inf"), u8), (128, i8), (-129, i8), (-0.25, i8)):
        with pytest.raises(ValueError):
            rm._exact_narrow("k", np.array([0, bad]), dt)
        with pytest.raises(ValueError):
            rm._exact_narrow("k", torch.tensor([0.0, float(bad)]), dt)
    with pytest.raises(ValueError):
        rm._exact_narrow("k", np.array(["a", "b"]), u8)
    t = rm._exact_narrow("k", torch.tensor([[3.0, 250.0]]), u8)
    assert t.dtype == u8 and t.tolist() == [[3, 250]]
    assert rm._exact_narrow("k", torch.tensor([-128, 127]), i8).dtype == i8
    with pytest.raises(ValueError):
        rm._exact_narrow("k", torch.tensor([-128, 128]), i8)
