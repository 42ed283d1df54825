#!/usr/bin/env python
"""Golden vectors for the PPO UPDATE path (SURVEY row a22/a23), generated from the UNMODIFIED reference
(rl.networks.model.Policy.evaluate_actions, rl.networks.storage.RolloutStorage, rl.ppo.PPO) in the build
container behind oracle/shims.

A recorded rollout [T=30, N=8] is cut from tests/golden/env_pred_h20.npz (two 30-step windows of its 4
environments, chosen so that episodes end mid-rollout), teacher-forced through the reference policy
(synthetic weights = tests/policy_fixture.synth_state_dict) to get value / log-prob / hidden state, inserted
into the reference RolloutStorage, then: compute_returns (GAE), recurrent_generator under a fixed torch seed,
evaluate_actions on the first minibatch and ONE PPO.update (2 epochs x 2 minibatches, entropy_coef != 0 so the
entropy term is pinned).  Stored: the rollout inputs, returns, the minibatch outputs, the three losses and, per
parameter tensor, its sum / abs-sum / first 4 entries after the update.  A second file, update_t30_n8_entries.npz,
holds how the update moved a seeded sample of single entries (every entry of small tensors, ENTRIES_PER_TENSOR of
each larger one): the full 10 MB of weights are too large to store.

    CROWDNAV_REFERENCE_ROOT=<reference checkout> python tools/make_golden_update.py
"""
import os
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "oracle", "shims"))
sys.path.insert(0, os.environ["CROWDNAV_REFERENCE_ROOT"])
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

T, N, H, W = 30, 8, 20, 12
WINDOWS = None      # filled by pick_windows
HYPER = dict(clip_param=0.2, ppo_epoch=2, num_mini_batch=2, value_loss_coef=0.5, entropy_coef=0.01,
             lr=4e-5, eps=1e-5, max_grad_norm=0.5)
SEED_GEN = 777


def pick_windows(done):
    """two window starts per source env such that every window holds at least one episode end in steps 3..26"""
    starts = []
    for e in range(done.shape[1]):
        idx = np.nonzero(done[:, e])[0]
        got = []
        for d in idx:
            s = int(d) - 11
            if s >= 0 and s + T < done.shape[0] and all(abs(s - g) >= 8 for g in got):
                got.append(s)
            if len(got) == 2:
                break
        assert len(got) == 2, (e, idx)
        starts.append(got)
    return starts


def cut_rollout(g):
    starts = pick_windows(g["done"])
    cols = [(e, s) for e in range(4) for s in starts[e]]          # 8 (source env, start) pairs
    ob = {}
    for k in ["robot_node", "temporal_edges", "spatial_edges", "detected_human_num"]:
        ob[k] = np.stack([g["ob_" + k][s:s + T + 1, e] for e, s in cols], 1).astype(np.float32)
    act = np.stack([g["actions"][s:s + T, e] for e, s in cols], 1).astype(np.float32)
    rew = np.stack([g["reward"][s:s + T, e] for e, s in cols], 1).astype(np.float32)
    done = np.stack([g["done"][s:s + T, e] for e, s in cols], 1)
    return ob, act, rew, done


def reference_objects():
    from make_golden_policy import build_reference_policy
    pol = build_reference_policy("CrowdSimPred-v0", H, W, N)
    pol.base.nminibatch = HYPER["num_mini_batch"]
    pol.base.seq_length = T
    from policy_fixture import synth_state_dict
    pol.load_state_dict(synth_state_dict(pol.state_dict()))
    return pol


def fill_storage(pol, storage_cls, ob, act, rew, done, spaces, act_space):
    """train.py:152-191 with the recorded actions instead of sampled ones."""
    ro = storage_cls(T, N, spaces, act_space, 128, 256)
    for k in ro.obs:
        ro.obs[k][0].copy_(torch.from_numpy(ob[k][0]))
    for t in range(T):
        with torch.no_grad():
            o = {k: ro.obs[k][t] for k in ro.obs}
            hx = {k: ro.recurrent_hidden_states[k][t] for k in ro.recurrent_hidden_states}
            value, feat, hx2 = pol.base(o, hx, ro.masks[t], infer=True)
            dist = pol.dist(feat)
            a = torch.from_numpy(act[t])
            logp = dist.log_probs(a)
        masks = torch.from_numpy(1.0 - done[t].astype(np.float32)).unsqueeze(1)
        ro.insert({k: torch.from_numpy(ob[k][t + 1]) for k in ro.obs}, hx2, a, logp, value,
                  torch.from_numpy(rew[t]).unsqueeze(1), masks, torch.ones(N, 1))
    with torch.no_grad():
        o = {k: ro.obs[k][-1] for k in ro.obs}
        hx = {k: ro.recurrent_hidden_states[k][-1] for k in ro.recurrent_hidden_states}
        nv = pol.get_value(o, hx, ro.masks[-1]).detach()
    ro.compute_returns(nv, True, 0.99, 0.95, False)
    return ro


def spaces_for_reference():
    import gym
    sp = {"robot_node": gym.spaces.Box(-np.inf, np.inf, (1, 7)), "temporal_edges": gym.spaces.Box(-np.inf, np.inf, (1, 2)),
          "spatial_edges": gym.spaces.Box(-np.inf, np.inf, (H, W)), "detected_human_num": gym.spaces.Box(-np.inf, np.inf, (1,))}
    return sp, gym.spaces.Box(-np.inf * np.ones(2), np.inf * np.ones(2), dtype=np.float32)


def run_reference():
    """Everything the fixture stores, computed by the unmodified reference.  Returns (dict of arrays, policy)."""
    from rl.networks.storage import RolloutStorage
    from rl.ppo import PPO
    g = np.load(os.path.join(REPO, "tests", "golden", "env_pred_h20.npz"))
    ob, act, rew, done = cut_rollout(g)
    pol = reference_objects()
    spaces, act_space = spaces_for_reference()
    ro = fill_storage(pol, RolloutStorage, ob, act, rew, done, spaces, act_space)
    out = {"ob_" + k: v for k, v in ob.items()}
    out.update(actions=act, rewards=rew, done=done, value_preds=ro.value_preds.numpy().copy(),
               action_log_probs=ro.action_log_probs.numpy().copy(), returns=ro.returns.numpy().copy(),
               hidden=ro.recurrent_hidden_states['human_node_rnn'].numpy().copy(), masks=ro.masks.numpy().copy())
    adv = ro.returns[:-1] - ro.value_preds[:-1]
    adv = (adv - adv.mean()) / (adv.std() + 1e-5)
    torch.manual_seed(SEED_GEN)
    sample = next(iter(ro.recurrent_generator(adv, HYPER["num_mini_batch"])))
    obs_b, hxs_b, act_b, vpred_b, ret_b, masks_b, old_lp_b, adv_b = sample
    out.update(mb_adv=adv_b.numpy().copy(), mb_actions=act_b.numpy().copy(), mb_masks=masks_b.numpy().copy(),
               mb_spatial_edges=obs_b["spatial_edges"].numpy().copy(), mb_h0=hxs_b["human_node_rnn"].numpy().copy())
    values, lp, ent, hx = pol.evaluate_actions(obs_b, hxs_b, masks_b, act_b)
    out.update(mb_values=values.detach().numpy().copy(), mb_logp=lp.detach().numpy().copy(), mb_entropy=np.float64(ent.item()),
               mb_h_final=hx["human_node_rnn"].detach().numpy().copy())
    # gradient of a fixed scalar through evaluate_actions (no optimiser involved)
    pol.zero_grad()
    (values.mean() + lp.mean() + ent).backward()
    gn = {k: float(p.grad.norm()) if p.grad is not None else -1.0 for k, p in pol.named_parameters()}
    out["grad_keys"] = np.array(sorted(gn.keys()))
    out["grad_norms"] = np.array([gn[k] for k in sorted(gn.keys())])
    pol.zero_grad()
    agent = PPO(pol, **HYPER)
    torch.manual_seed(SEED_GEN + 1)
    vl, al, de = agent.update(ro)
    out.update(losses=np.array([vl, al, de], dtype=np.float64))
    sd = pol.state_dict()
    keys = sorted(sd.keys())
    out["param_keys"] = np.array(keys)
    out["param_sum"] = np.array([float(sd[k].double().sum()) for k in keys])
    out["param_abs"] = np.array([float(sd[k].double().abs().sum()) for k in keys])
    out["param_head"] = np.stack([np.resize(sd[k].reshape(-1)[:4].double().numpy(), 4) for k in keys])
    return out, pol


ENTRIES_PER_TENSOR = 256


def sampled_entries(pol):
    """Per parameter tensor (sorted keys): flat indices of a seeded sample of its entries and how the update moved
    each of them (post-update minus synthetic initial value, in fp32)."""
    from policy_fixture import synth_state_dict
    sd = pol.state_dict()
    pre = synth_state_dict(sd)
    rng = np.random.default_rng(2024)
    keys, tensor, index, delta = sorted(sd.keys()), [], [], []
    for i, k in enumerate(keys):
        n = sd[k].numel()
        idx = np.arange(n) if n <= ENTRIES_PER_TENSOR else np.sort(rng.choice(n, ENTRIES_PER_TENSOR, replace=False))
        d = (sd[k] - pre[k]).reshape(-1).numpy()[idx]
        tensor.append(np.full(len(idx), i, np.int16))
        index.append(idx.astype(np.int32))
        delta.append(d.astype(np.float32))
    return dict(param_keys=np.array(keys), tensor=np.concatenate(tensor), index=np.concatenate(index),
                delta=np.concatenate(delta))


if __name__ == "__main__":
    out, pol = run_reference()
    p = os.path.join(REPO, "tests", "golden", "update_t30_n8.npz")
    np.savez_compressed(p, **out)
    print("wrote", p, os.path.getsize(p), "bytes; losses", out["losses"], "entropy", out["mb_entropy"],
          "dones per env", out["done"].sum(0))
    p = os.path.join(REPO, "tests", "golden", "update_t30_n8_entries.npz")
    np.savez_compressed(p, **sampled_entries(pol))
    print("wrote", p, os.path.getsize(p), "bytes")
