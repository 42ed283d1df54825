"""PPO update path (SURVEY rows a22 / a23) against the UNMODIFIED reference.

Fixture tests/golden/update_t30_n8.npz = outputs of rl.networks.model.Policy.evaluate_actions,
rl.networks.storage.RolloutStorage (insert, compute_returns, recurrent_generator) and one rl.ppo.PPO.update on a
recorded rollout [T=30, N=8] with episodes ending mid-rollout (tools/make_golden_update.py).  The mirror
(crowdnav_prediction_attngraph_b200.{policy,storage,ppo}) runs the same inputs on CPU — the update path is
PyTorch on whatever device holds the tensors; only act/get_value need the CUDA engine, so the teacher-forced
rollout quantities (value_preds, log-probs, hidden) are taken from the fixture.

Tolerances (fp32, different but algebraically equal association: folded projections, compacted rows):
evaluate_actions value / log-prob / entropy <= 1e-5 relative to the tensor's scale; losses 1e-5 relative;
post-update parameters: per-tensor sums to 1e-6 relative of the abs-sum, leading entries 2e-6 absolute
(the Adam step is lr = 4e-5 per entry, so a wrong-signed or missing gradient moves an entry by >= 4e-5);
single entries of a seeded sample of every tensor 1e-6 absolute (tests/golden/update_t30_n8_entries.npz)."""
import os
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from policy_fixture import synth_state_dict  # noqa: E402

T, N, H, W = 30, 8, 20, 12
HYPER = dict(clip_param=0.2, ppo_epoch=2, num_mini_batch=2, value_loss_coef=0.5, entropy_coef=0.01,
             lr=4e-5, eps=1e-5, max_grad_norm=0.5)
SEED_GEN = 777


def _fixture():
    return np.load(os.path.join(REPO, "tests", "golden", "update_t30_n8.npz"))


class _Args(object):
    num_processes, seq_length, num_mini_batch = N, T, 2


def _mirror_policy():
    from crowdnav_prediction_attngraph_b200.policy import Policy
    from crowdnav_prediction_attngraph_b200.vec_env import Box
    spaces = {'robot_node': Box((1, 7)), 'temporal_edges': Box((1, 2)), 'spatial_edges': Box((H, W)),
              'detected_human_num': Box((1,))}
    pol = Policy(spaces, Box((2,)), base='selfAttn_merge_srnn', base_kwargs=_Args())
    pol.load_state_dict(synth_state_dict(pol.state_dict()))
    return pol, spaces


def _mirror_storage(g, spaces):
    """Fill the mirror RolloutStorage through its own insert() from the recorded rollout."""
    from crowdnav_prediction_attngraph_b200.storage import RolloutStorage
    from crowdnav_prediction_attngraph_b200.vec_env import Box
    ro = RolloutStorage(T, N, spaces, Box((2,)), 128, 256)
    for k in ro.obs:
        ro.obs[k][0].copy_(torch.from_numpy(g["ob_" + k][0]))
    for t in range(T):
        masks = torch.from_numpy(1.0 - g["done"][t].astype(np.float32)).unsqueeze(1)
        ro.insert({k: torch.from_numpy(g["ob_" + k][t + 1]) for k in ro.obs},
                  {'human_node_rnn': torch.from_numpy(g["hidden"][t + 1])}, torch.from_numpy(g["actions"][t]),
                  torch.from_numpy(g["action_log_probs"][t]), torch.from_numpy(g["value_preds"][t]),
                  torch.from_numpy(g["rewards"][t]).unsqueeze(1), masks, torch.ones(N, 1))
    return ro


def _close(a, b, rel):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    scale = max(1.0, float(np.abs(b).max()))
    return float(np.abs(a - b).max()) <= rel * scale, float(np.abs(a - b).max()), scale


def test_storage_returns_and_generator_match_reference():
    g = _fixture()
    pol, spaces = _mirror_policy()
    ro = _mirror_storage(g, spaces)
    assert np.array_equal(ro.masks.numpy(), g["masks"])
    ro.compute_returns(torch.from_numpy(g["value_preds"][-1]), True, 0.99, 0.95, False)
    ok, err, sc = _close(ro.returns.numpy(), g["returns"], 1e-6)
    assert ok, (err, sc)
    adv = ro.returns[:-1] - ro.value_preds[:-1]
    from crowdnav_prediction_attngraph_b200.ppo import global_advantage_normalize
    adv = global_advantage_normalize(adv)
    torch.manual_seed(SEED_GEN)
    obs_b, hxs_b, act_b, vpred_b, ret_b, masks_b, old_lp_b, adv_b = next(iter(ro.recurrent_generator(adv, 2)))
    assert np.array_equal(obs_b["spatial_edges"].numpy(), g["mb_spatial_edges"])     # same permutation, same order
    assert np.array_equal(act_b.numpy(), g["mb_actions"]) and np.array_equal(masks_b.numpy(), g["mb_masks"])
    assert np.array_equal(hxs_b["human_node_rnn"].numpy(), g["mb_h0"])
    ok, err, sc = _close(adv_b.numpy(), g["mb_adv"], 1e-5)
    assert ok, (err, sc)


def test_evaluate_actions_matches_reference():
    g = _fixture()
    pol, spaces = _mirror_policy()
    ro = _mirror_storage(g, spaces)
    ro.returns.copy_(torch.from_numpy(g["returns"]))
    adv = ro.returns[:-1] - ro.value_preds[:-1]
    adv = (adv - adv.mean()) / (adv.std() + 1e-5)
    torch.manual_seed(SEED_GEN)
    obs_b, hxs_b, act_b, vpred_b, ret_b, masks_b, old_lp_b, adv_b = next(iter(ro.recurrent_generator(adv, 2)))
    assert float(masks_b.min()) == 0.0                     # the minibatch holds episode ends (GRU resets at T > 1)
    for packed in (True, False):
        pol.pack_valid_rows = packed
        values, lp, ent, hx = pol.evaluate_actions(obs_b, hxs_b, masks_b, act_b)
        for name, a, b in (("values", values, g["mb_values"]), ("logp", lp, g["mb_logp"]),
                           ("h_final", hx["human_node_rnn"], g["mb_h_final"])):
            ok, err, sc = _close(a.detach().numpy(), b, 1e-5)
            assert ok, (packed, name, err, sc)
        assert abs(float(ent.detach()) - float(g["mb_entropy"])) <= 1e-6, (float(ent.detach()), float(g["mb_entropy"]))
        # gradient norms of a fixed scalar through evaluate_actions, per parameter tensor
        pol.zero_grad()
        (values.mean() + lp.mean() + ent).backward()
        gn = {k: float(p.grad.norm()) if p.grad is not None else -1.0 for k, p in pol.named_parameters()}
        for k, ref in zip(g["grad_keys"], g["grad_norms"]):
            k = str(k)
            assert (gn[k] < 0) == (ref < 0), k
            assert abs(gn[k] - ref) <= 2e-4 * max(1.0, abs(ref)), (packed, k, gn[k], ref)


def _mirror_update(g):
    from crowdnav_prediction_attngraph_b200.ppo import PPO
    pol, spaces = _mirror_policy()
    ro = _mirror_storage(g, spaces)
    ro.compute_returns(torch.from_numpy(g["value_preds"][-1]), True, 0.99, 0.95, False)
    agent = PPO(pol, **HYPER)
    torch.manual_seed(SEED_GEN + 1)
    losses = agent.update(ro)
    return pol, losses


def test_ppo_update_matches_reference_fixture():
    g = _fixture()
    pol, losses = _mirror_update(g)
    for a, b, name in zip(losses, g["losses"], ("value_loss", "action_loss", "dist_entropy")):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(b)), (name, a, b)
    sd = pol.state_dict()
    pre = synth_state_dict(sd)
    moved = 0
    for i, k in enumerate(g["param_keys"]):
        k = str(k)
        s, ab = float(sd[k].double().sum()), float(sd[k].double().abs().sum())
        assert abs(s - g["param_sum"][i]) <= 1e-6 * max(1.0, g["param_abs"][i]), (k, s, g["param_sum"][i])
        assert abs(ab - g["param_abs"][i]) <= 1e-6 * max(1.0, g["param_abs"][i]), k
        head = np.resize(sd[k].reshape(-1)[:4].double().numpy(), 4)
        assert np.abs(head - g["param_head"][i]).max() <= 2e-6, (k, head, g["param_head"][i])
        moved += int((sd[k] != pre[k]).any())
    # everything was trained but human_node_final_linear.* (unused by the forward) and k_linear.bias (a key bias shifts
    # all scores of a query equally: the soft-max is invariant, the gradient is zero up to rounding noise)
    assert moved >= len(g["param_keys"]) - 3


def test_ppo_update_matches_reference_sampled_entries():
    """Single entries after the update: every entry of the small tensors and a seeded sample of 256 entries of each
    larger one (tests/golden/update_t30_n8_entries.npz, the reference's post-update minus initial value)."""
    g = _fixture()
    e = np.load(os.path.join(REPO, "tests", "golden", "update_t30_n8_entries.npz"))
    pol, losses = _mirror_update(g)
    sd = pol.state_dict()
    pre = synth_state_dict(sd)
    assert sorted(sd.keys()) == [str(k) for k in e["param_keys"]]
    worst = 0.0
    for i, k in enumerate(e["param_keys"]):
        k, sel = str(k), e["tensor"] == i
        d_ref = e["delta"][sel].astype(np.float64)
        d_own = (sd[k] - pre[k]).reshape(-1).numpy()[e["index"][sel]].astype(np.float64)
        err = float(np.abs(d_ref - d_own).max())
        worst = max(worst, err)
        # 4 Adam steps of lr 4e-5: |delta| <= 1.6e-4 per entry; agreement to 2 % of ONE step
        assert err <= 1e-6, (k, err, float(np.abs(d_ref).max()))
    print("max |delta_ref - delta_own| over %d sampled entries:" % len(e["delta"]), worst)
