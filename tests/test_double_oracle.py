"""The Double DQN oracle (tests/double_oracle.py) pinned on hand-built cases -- CPU only.

Each case states the expected selection or target from the rules of include/ofb_train.h (ofb_trainer_td_targets_double): the
online predictions select (act ties to 0; the pointer's first maximum, NaNs skipped, index 0 for an all-NaN map), the target's
evaluate, the overwritten pointer entry is the [x][y] one, and the roundings are the single-network targets'."""
import numpy as np
import pytest
import torch

from oracle import policy_train_torch as ptt
from tests import double_oracle as do

G = 0.9
N = 400 * 400


def _f32(x):
    return np.float32(x)


def _bits(t):
    return np.asarray(t, dtype=np.float32).view(np.uint32)


def _case(B=1, seed=0):
    g = torch.Generator().manual_seed(seed)
    return dict(act_obs=torch.randn((B, 2), generator=g), ptr_obs=torch.randn((B, 400, 400), generator=g),
                act_on=torch.randn((B, 2), generator=g), ptr_on=torch.randn((B, 400, 400), generator=g),
                act_tg=torch.randn((B, 2), generator=g), ptr_tg=torch.randn((B, 400, 400), generator=g),
                iaction=torch.randint(0, 2, (B,), generator=g, dtype=torch.int32),
                pointer=torch.randint(0, 400, (B, 2), generator=g, dtype=torch.int32),
                reward=torch.randn((B,), generator=g), done=torch.zeros((B,), dtype=torch.uint8))


def _run(c, discount=None, gamma=G):
    return do.td_targets_double(c["act_obs"], c["ptr_obs"], c["act_on"], c["ptr_on"], c["act_tg"], c["ptr_tg"], c["iaction"],
                                c["pointer"], c["reward"], c["done"], gamma=gamma, discount=discount)


def test_act_ties_select_zero():
    a = torch.tensor([[1.0, 1.0], [0.0, -0.0], [2.0, 3.0], [3.0, 2.0], [float("nan"), 1.0], [1.0, float("nan")]])
    assert do.select_act(a).tolist() == [0, 0, 1, 0, 0, 0]


@pytest.mark.parametrize("where", [0, 1, 400 * 200 + 7, N - 1])
def test_pointer_plateau_selects_the_first_index(where):
    m = torch.zeros((1, 400, 400))
    flat = m.view(-1)
    flat[where] = 5.0
    flat[N - 1] = 5.0                                     # a later entry at the same maximum
    flat[where + 1 if where + 1 < N else where] = 5.0
    assert do.select_ptr(m).tolist() == [where]


def test_pointer_skips_nan_and_all_nan_gives_zero():
    m = torch.full((3, 400, 400), -1.0)
    m[0].view(-1)[0] = float("nan")
    m[0].view(-1)[10] = 2.0
    m[0].view(-1)[11] = float("nan")
    m[1].view(-1)[:] = float("nan")
    m[1].view(-1)[N - 1] = -7.0
    m[2].view(-1)[:] = float("nan")
    assert do.select_ptr(m).tolist() == [10, N - 1, 0]


def test_minus_infinity_maps():
    m = torch.full((2, 400, 400), -float("inf"))
    m[1].view(-1)[123] = -1e30
    assert do.select_ptr(m).tolist() == [0, 123]
    c = _case()
    c["ptr_on"] = m[:1].clone()
    c["ptr_tg"] = torch.full((1, 400, 400), -float("inf"))
    t_act, t_ptr, _, td_ptr = _run(c)
    x, y = c["pointer"][0].tolist()
    assert t_ptr[0, x, y].item() == -float("inf") and td_ptr[0].item() == -float("inf")


def test_values_come_from_the_target_maps():
    c = _case(B=4, seed=3)
    t_act, t_ptr, td_act, td_ptr = _run(c)
    a_star, p_star = do.select_act(c["act_on"]), do.select_ptr(c["ptr_on"])
    for b in range(4):
        keep = _f32(1.0)
        va = _f32(c["act_tg"][b, int(a_star[b])].item())
        vp = _f32(c["ptr_tg"].reshape(4, -1)[b, int(p_star[b])].item())
        r = _f32(c["reward"][b].item())
        ta = _f32(r + _f32(_f32(_f32(G) * va) * keep))
        tp = _f32(r + _f32(_f32(_f32(G) * vp) * keep))
        ia, (x, y) = int(c["iaction"][b]), c["pointer"][b].tolist()
        assert _bits(t_act[b, ia].item()) == _bits(ta) and _bits(t_ptr[b, x, y].item()) == _bits(tp)
        assert t_act[b, 1 - ia] == c["act_obs"][b, 1 - ia]
        assert _bits(td_act[b].item()) == _bits(_f32(ta - _f32(c["act_obs"][b, ia].item())))
        assert _bits(td_ptr[b].item()) == _bits(_f32(tp - _f32(c["ptr_obs"][b, x, y].item())))


def test_done_gives_the_reward():
    c = _case(B=3, seed=4)
    c["done"] = torch.tensor([1, 0, 1], dtype=torch.uint8)
    t_act, t_ptr, _, _ = _run(c)
    for b in (0, 2):
        ia, (x, y) = int(c["iaction"][b]), c["pointer"][b].tolist()
        assert t_act[b, ia] == c["reward"][b] and t_ptr[b, x, y] == c["reward"][b]


def test_discount_replaces_gamma():
    c = _case(B=3, seed=5)
    same = _run(c, discount=torch.full((3,), G, dtype=torch.float32))
    scalar = _run(c)
    for x, y in zip(same, scalar):
        assert torch.equal(x, y)
    d = torch.tensor([0.5, 0.125, 0.729], dtype=torch.float32)
    t_act, t_ptr, _, _ = _run(c, discount=d)
    p_star = do.select_ptr(c["ptr_on"])
    for b in range(3):
        x, y = c["pointer"][b].tolist()
        vp = _f32(c["ptr_tg"].reshape(3, -1)[b, int(p_star[b])].item())
        want = _f32(_f32(c["reward"][b].item()) + _f32(_f32(d[b].item()) * vp))
        assert _bits(t_ptr[b, x, y].item()) == _bits(want)


def test_the_pointer_entry_is_the_transposed_one():
    c = _case(seed=6)
    c["pointer"] = torch.tensor([[3, 250]], dtype=torch.int32)
    t_act, t_ptr, _, _ = _run(c)
    diff = (t_ptr != c["ptr_obs"]).nonzero().tolist()
    assert diff == [[0, 3, 250]]                          # ptr_target[x][y] of the [row, col] map


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_synced_maps_give_the_single_network_targets(seed):
    c = _case(B=5, seed=seed)
    c["act_tg"], c["ptr_tg"] = c["act_on"], c["ptr_on"]
    c["done"] = torch.tensor([0, 1, 0, 0, 1], dtype=torch.uint8)
    t_act, t_ptr, td_act, td_ptr = _run(c)
    s_act, s_ptr = ptt.td_targets(c["act_obs"], c["ptr_obs"], c["act_on"], c["ptr_on"], c["iaction"], c["pointer"], c["reward"],
                                  c["done"], gamma=G)
    assert torch.equal(t_act, s_act) and torch.equal(t_ptr, s_ptr)
    rows = torch.arange(5)
    ia, px, py = c["iaction"].long(), c["pointer"][:, 0].long(), c["pointer"][:, 1].long()
    assert torch.equal(td_act, s_act[rows, ia] - c["act_obs"][rows, ia])
    assert torch.equal(td_ptr, s_ptr[rows, px, py] - c["ptr_obs"][rows, px, py])


def test_blend_and_tau_one_copy():
    from ofighters_b200.trainer import blend_weights
    g = torch.Generator().manual_seed(9)
    w = {"a": torch.randn((3, 5), generator=g), "b": torch.randn((7,), generator=g) * 1e-3}
    wt = {"a": torch.randn((3, 5), generator=g), "b": torch.randn((7,), generator=g) * 1e3}
    for tau in (0.25, 0.1, 0.999, 1.0):
        got = blend_weights(w, wt, tau)
        want = do.blend({k: v.numpy() for k, v in w.items()}, {k: v.numpy() for k, v in wt.items()}, tau)
        for k in w:
            assert np.array_equal(got[k].numpy().view(np.uint32), want[k].view(np.uint32)), (tau, k)
    one = blend_weights(w, wt, 1.0)
    for k in w:
        assert np.array_equal(one[k].numpy().view(np.uint32), w[k].numpy().view(np.uint32))


@pytest.mark.parametrize("kw", [dict(double_dqn=True), dict(target_update=0), dict(target_update=1.5), dict(target_update=True),
                                dict(target_update=3, target_tau=0.0), dict(target_update=3, target_tau=1.5),
                                dict(target_update=3, target_tau=float("nan"))])
def test_trainer_refuses_bad_target_arguments_before_touching_a_device(kw):
    from ofighters_b200.trainer import TrainerB200
    with pytest.raises(Exception, match="Invalid"):
        TrainerB200(**kw)
