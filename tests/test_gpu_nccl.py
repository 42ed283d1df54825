"""GPU, >= 2 devices: the PPO update collectives on NCCL hardware (SURVEY.md §8e, rl/ppo/ppo.py:37-39,83-86).

Two ranks (one process per GPU, NCCL over NVLink) must reproduce the single-process result on the concatenated
batch -- the same check tests/test_multi_rank_gloo.py makes on CPU with gloo -- and a 2-rank PPO.update on env-sharded
rollouts must leave both replicas with identical parameters equal to the 1-rank update on the whole batch up to
fp32 reduction-order noise."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from crowdnav_prediction_attngraph_b200.ppo import allreduce_gradients, global_advantage_normalize
    torch.manual_seed(0)
    full = torch.randn(6, 8, 1)
    shard = full[:, rank * 4:(rank + 1) * 4].to(dev)
    norm = global_advantage_normalize(shard.clone()).cpu()
    lin = torch.nn.Linear(5, 3).to(dev)
    torch.manual_seed(100 + rank)
    x = torch.randn(7, 5).to(dev)
    lin(x).pow(2).mean().backward()
    local = [p.grad.clone().cpu() for p in lin.parameters()]
    ev = []
    nbytes = allreduce_gradients(list(lin.parameters()), ev)
    torch.cuda.synchronize()
    torch.save(dict(norm=norm, local=local, avg=[p.grad.clone().cpu() for p in lin.parameters()], nbytes=nbytes,
                    ms=ev[0][0].elapsed_time(ev[0][1])), os.path.join(out_dir, "r%d.pt" % rank))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_ppo_collectives_nccl_world2(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r = [torch.load(os.path.join(str(tmp_path), "r%d.pt" % k)) for k in range(2)]
    torch.manual_seed(0)
    full = torch.randn(6, 8, 1)
    ref = (full - full.mean()) / (full.std() + 1e-5)
    got = torch.cat([r[0]["norm"], r[1]["norm"]], dim=1)
    assert torch.allclose(got, ref, atol=1e-6)
    for k in range(2):
        assert r[k]["nbytes"] == (5 * 3 + 3) * 4
        for a, l0, l1 in zip(r[k]["avg"], r[0]["local"], r[1]["local"]):
            assert torch.allclose(a, (l0 + l1) / 2, atol=1e-7)


def _update_worker(rank, world, port, out_dir):
    """Env-sharded rollout [T=30, 32 envs per rank] -> one PPO.update with the NCCL gradient all-reduce."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    if world > 1:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from crowdnav_prediction_attngraph_b200.vec_env import CudaCrowdVecEnv
    from crowdnav_prediction_attngraph_b200.policy import Policy
    from crowdnav_prediction_attngraph_b200.storage import RolloutStorage
    from crowdnav_prediction_attngraph_b200 import ppo
    N, T = 32, 30

    class Args(object):
        num_processes, seq_length, num_mini_batch = N, T, 1
    env = CudaCrowdVecEnv(num_envs=N, nenv_total=N * world, rank_offset=rank * N, seed=5, human_num=20, device=dev)
    torch.manual_seed(1)
    pol = Policy(env.observation_space.spaces, env.action_space, base_kwargs=Args(), base='selfAttn_merge_srnn').to(dev)
    ro = RolloutStorage(T, N, env.observation_space.spaces, env.action_space, 128, 256, device=dev)
    obs = env.reset()
    for k in ro.obs:
        ro.obs[k][0].copy_(obs[k])
    eng = pol._engine(N, dev)
    torch.manual_seed(77)                      # same noise stream on both ranks: the test compares with a re-run below
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    for _ in range(T):
        s = ro.step
        o = {k: ro.obs[k][s] for k in ro.obs}
        noise = torch.randn(N, 2, device=dev, generator=gen)
        v, a, lp, h = eng.act(o, ro.recurrent_hidden_states['human_node_rnn'][s], ro.masks[s], noise=noise)
        nobs, rew, done, info = env.step_device(a)
        ro.insert(nobs, {'human_node_rnn': h}, a, lp, v, rew, (1.0 - done.float()).unsqueeze(1))
    with torch.no_grad():
        nv = pol.get_value({k: ro.obs[k][-1] for k in ro.obs},
                           {'human_node_rnn': ro.recurrent_hidden_states['human_node_rnn'][-1]}, ro.masks[-1]).detach()
    ro.compute_returns(nv, True, 0.99, 0.95, False)
    agent = ppo.PPO(pol, 0.2, 1, 1, 0.5, 0.0, lr=1e-4, eps=1e-5, max_grad_norm=0.5)
    agent.profile = True
    losses = agent.update(ro)
    torch.cuda.synchronize()
    torch.save(dict(sd={k: v.detach().cpu() for k, v in pol.state_dict().items()}, losses=losses, prof=agent.last_profile,
                    storage=dict(obs={k: v.cpu() for k, v in ro.obs.items()}, actions=ro.actions.cpu(), returns=ro.returns.cpu(),
                                 value_preds=ro.value_preds.cpu(), logp=ro.action_log_probs.cpu(), masks=ro.masks.cpu(),
                                 hidden=ro.recurrent_hidden_states['human_node_rnn'].cpu(), rewards=ro.rewards.cpu())),
               os.path.join(out_dir, "u%d.pt" % rank))
    if world > 1:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_update_equals_single_rank_update_on_the_whole_batch(tmp_path):
    port = _free_port()
    mp.spawn(_update_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r = [torch.load(os.path.join(str(tmp_path), "u%d.pt" % k)) for k in range(2)]
    # replicas stay identical
    for k in r[0]["sd"]:
        assert torch.equal(r[0]["sd"][k], r[1]["sd"][k]), k
    assert r[0]["prof"]["allreduce_calls"] == 1 and r[0]["prof"]["allreduce_bytes_per_call"] > 9_000_000
    # single process on the concatenated rollout (64 envs): same update up to reduction order
    from crowdnav_prediction_attngraph_b200.policy import Policy
    from crowdnav_prediction_attngraph_b200.storage import RolloutStorage
    from crowdnav_prediction_attngraph_b200.vec_env import Box
    from crowdnav_prediction_attngraph_b200 import ppo
    import numpy as np
    dev = torch.device("cuda", 0)
    N, T = 64, 30

    class Args(object):
        num_processes, seq_length, num_mini_batch = N, T, 1
    spaces = {'robot_node': Box((1, 7)), 'temporal_edges': Box((1, 2)), 'spatial_edges': Box((20, 12)), 'detected_human_num': Box((1,))}
    torch.manual_seed(1)
    pol = Policy(spaces, Box((2,)), base_kwargs=Args(), base='selfAttn_merge_srnn').to(dev)
    ro = RolloutStorage(T, N, spaces, Box((2,)), 128, 256, device=dev)
    cat = lambda f: torch.cat([f(r[0]["storage"]), f(r[1]["storage"])], dim=1).to(dev)
    for k in ro.obs:
        ro.obs[k].copy_(cat(lambda s: s["obs"][k]))
    ro.actions.copy_(cat(lambda s: s["actions"])); ro.returns.copy_(cat(lambda s: s["returns"]))
    ro.value_preds.copy_(cat(lambda s: s["value_preds"])); ro.action_log_probs.copy_(cat(lambda s: s["logp"]))
    ro.masks.copy_(cat(lambda s: s["masks"])); ro.rewards.copy_(cat(lambda s: s["rewards"]))
    ro.recurrent_hidden_states['human_node_rnn'].copy_(cat(lambda s: s["hidden"]))
    agent = ppo.PPO(pol, 0.2, 1, 1, 0.5, 0.0, lr=1e-4, eps=1e-5, max_grad_norm=0.5)
    agent.update(ro)
    worst = 0.0
    for k, v in pol.state_dict().items():
        worst = max(worst, float((v.cpu() - r[0]["sd"][k]).abs().max()))
    # one Adam step of lr 1e-4: entries move by ~1e-4; agreement to a few percent of a step (fp32 reduction order,
    # and the sign-like Adam normalisation amplifies gradient noise near zero)
    assert worst <= 2e-5, worst


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_unmodified_train_py_under_torchrun_two_ranks(tmp_path):
    """`torchrun --nproc-per-node 2 <reference>/train.py` with the compat aliases: make_vec_envs shards the environments
    over the ranks (32 each), PPO broadcasts the initial weights and all-reduces the gradients over NCCL; train.py itself
    is the reference's file, byte for byte (sha256 manifest).  Both ranks finish 2 updates and rank files agree."""
    import subprocess
    import sys
    import numpy as np
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import test_dropin_reference_scripts as td
    root = td._ref_root()
    td._check_unmodified(root, ["train.py", "arguments.py"])
    w = td._workdir(tmp_path, root, td.C2_EDITS)
    out = os.path.join(w, "out")
    env = dict(os.environ)
    env["PYTHONSAFEPATH"] = "1"
    env["PYTHONPATH"] = os.pathsep.join([w, td.COMPAT, td.REPO, root])
    env["CROWDNAV_B200_TRACE"] = "1"
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(_free_port()), os.path.join(root, "train.py"), "--num-processes", "32",
                        "--env-name", "CrowdSimPred-v0", "--num-env-steps", str(32 * 30 * 2), "--output_dir", out,
                        "--log-interval", "1", "--save-interval", "1"], cwd=w, env=env, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    # both ranks built a 32-environment shard of a 64-environment job
    assert p.stderr.count("N=32 (of 64, offset 0)") == 1 and p.stderr.count("N=32 (of 64, offset 32)") == 1, p.stderr[-2000:]
    sd = torch.load(os.path.join(out, "checkpoints", "00001.pt"), map_location="cpu", weights_only=True)
    assert all(bool(np.isfinite(v.numpy()).all()) for v in sd.values())
