"""GPU tests of the drop-in classes: VectorizedBlockBlastEnv / BlockBlastEnv (reference
tests/test_environment.py KATs), RolloutBuffer (vs the oracle's GAE / normalisation), PPOAgent
(update metrics vs an independent computation) and a short end-to-end training run."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def test_vectorized_env_api_shapes_and_codec(torch):
    from bbgpu.vec_env import VectorizedBlockBlastEnv, BlockBlastEnv
    v = VectorizedBlockBlastEnv(num_envs=4, seed=42)
    assert v.num_envs == 4 and v.action_space.n == 192 and v.single_action_space.n == 192
    obs, infos = v.reset()
    assert obs["board"].shape == (4, 8, 8) and obs["board"].dtype == np.float32
    assert obs["pieces"].shape == (4, 3, 8, 8) and obs["pieces"].dtype == np.float32
    assert obs["action_mask"].shape == (4, 192) and obs["action_mask"].dtype == np.int8
    assert len(infos) == 4 and infos[0]["score"] == 0
    masks = v.get_action_masks()
    assert masks.shape == (4, 192) and masks.dtype == bool and np.array_equal(masks, obs["action_mask"].astype(bool))
    a = v.sample_valid_actions()
    assert a.shape == (4,) and all(masks[i, a[i]] for i in range(4))
    obs2, rew, term, trunc, infos = v.step(a)
    assert rew.shape == (4,) and rew.dtype == np.float32 and term.dtype == bool and not trunc.any()
    assert (obs2["board"].sum(axis=(1, 2)) > 0).all()
    # invalid action: negative reward, flagged, state untouched (tests/test_environment.py:100-114)
    bad = np.array([int(np.where(~v.get_action_masks()[i])[0][0]) for i in range(4)])
    before = v.handle.get_state().tobytes()
    _, rew, term, _, _ = v.step(bad)
    assert (rew == -10.0).all() and not term.any() and v.handle.get_state().tobytes() == before
    v.close()
    e = BlockBlastEnv(seed=3)
    assert (e.BOARD_SIZE, e.NUM_PIECES_PER_TURN, e.ACTION_SPACE_SIZE) == (8, 3, 192)
    assert e._action_to_move(0) == (0, 0, 0) and e._action_to_move(64) == (1, 0, 0) and e._action_to_move(128) == (2, 0, 0)
    assert e._move_to_action(0, 7, 7) == 63
    e.close()


def test_single_env_matches_python_oracle_episode(torch):
    """BlockBlastEnv (no auto-reset) against oracle.Env fed the same Philox trio stream."""
    from bbgpu import philox
    from bbgpu.vec_env import BlockBlastEnv
    from oracle import bb_oracle as O
    seed = 21
    stream = iter(philox.candidate_trios(seed, [0], 512)[0])
    ora = O.Env(draw=lambda: next(stream))
    env = BlockBlastEnv(seed=seed)           # constructor deals draw 0, like the oracle's
    rs = np.random.RandomState(0)
    done = False
    steps = 0
    while not done and steps < 200:
        va = ora.valid_actions()
        assert env.get_valid_actions() == va
        a = int(va[rs.randint(len(va))]) if rs.rand() > 0.1 else int(rs.randint(0, 192))
        oo, orw, od, _, oi = ora.step(a)
        go, grw, gd, gt, gi = env.step(a)
        assert np.float32(orw) == np.float32(grw) and od == gd and gt is False
        assert np.array_equal(oo["board"], go["board"]) and np.array_equal(oo["pieces"], go["pieces"])
        assert np.array_equal(oo["action_mask"], go["action_mask"])
        for k in ("score", "moves", "lines_cleared", "max_combo", "blocks_placed", "holes", "invalid_action"):
            assert oi[k] == gi[k], k
        assert abs(oi["board_fill"] - gi["board_fill"]) < 1e-12
        done = od
        steps += 1
    assert done
    # after game over every action is rejected with -10 (block_blast_env.py:240-245)
    _, r, t, _, info = env.step(0)
    assert r == -10.0 and t is False and info["invalid_action"]
    env.close()


def test_rollout_buffer_gae_and_gathered_samples(torch):
    from bbgpu.rollout import RolloutBuffer
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    from oracle import bb_oracle as O
    T, N = 12, 96
    venv = VectorizedBlockBlastEnv(N, seed=5, output="packed")
    obs, _ = venv.reset()
    buf = RolloutBuffer(T, N)
    rs = np.random.RandomState(1)
    kept = []
    for t in range(T):
        act = venv.sample_valid_actions()
        lp = torch.from_numpy(rs.randn(N).astype(np.float32)).cuda()
        val = torch.from_numpy(rs.randn(N).astype(np.float32)).cuda()
        row = tuple(obs[k].clone() for k in ("board", "pieces", "mask"))     # the env overwrites obs in place
        kept.append(tuple(x.cpu().numpy() for x in row))
        obs, rew, term, trunc, infos = venv.step(act)
        buf.add(*row, act, lp, rew, term.float(), val)
    assert buf.full
    last = torch.from_numpy(rs.randn(N).astype(np.float32)).cuda()
    buf.compute_returns_and_advantages(last, 0.99, 0.95)
    adv, ret = O.gae(buf.rewards.cpu().numpy(), buf.values.cpu().numpy(), buf.dones.cpu().numpy(), last.cpu().numpy(), 0.99, 0.95)
    assert np.array_equal(buf.advantages.cpu().numpy(), adv) and np.array_equal(buf.returns.cpu().numpy(), ret)
    norm = O.normalize_advantages(adv)
    from bbgpu import vec_env as VE
    seen = 0
    for boards, pieces, masks, actions, old_lp, a_n, r in buf.get_samples(500):
        b = boards.shape[0]
        assert boards.shape == (b, 8, 8) and pieces.shape == (b, 3, 8, 8) and masks.shape == (b, 192)
        assert actions.dtype == torch.int64
        seen += b
    assert seen == T * N
    # deterministic check of content: one batch of everything in storage order
    mean, std = buf.advantage_mean_std()
    got = ((buf.advantages.view(-1) - mean) / (std + 1e-8)).cpu().numpy()
    np.testing.assert_allclose(got, norm, rtol=1e-4, atol=1e-5)
    ms = torch.stack([mean, std])
    g = buf.gather(torch.arange(T * N, device="cuda"), ms)
    x, planes = g["obs"].cpu().numpy(), g["mask"].cpu().numpy()
    dense = VE.expand_mask(planes.view(np.uint64)).astype(np.float32)
    for t in (0, T // 2, T - 1):
        b, p, m = kept[t]
        sl = slice(t * N, (t + 1) * N)
        assert np.array_equal(x[sl, 0], VE.expand_board(b.view(np.uint64)))
        assert np.array_equal(x[sl, 1:], VE.expand_pieces(p.view(np.uint32)))
        assert np.array_equal(dense[sl], VE.expand_mask(m.view(np.uint64)).astype(np.float32))
    # the reference-layout add() path stores the same content (the pieces word of a used slot
    # carries another id byte, so it is compared through its expansion)
    buf2 = RolloutBuffer(2, N)
    b, p, m = kept[0]
    z = np.zeros(N, np.float32)
    for _ in range(2):
        buf2.add(VE.expand_board(b.view(np.uint64)), VE.expand_pieces(p.view(np.uint32)), VE.expand_mask(m.view(np.uint64)),
                 np.zeros(N, np.int64), z, z, z, z)
    g2 = buf2.gather(torch.arange(N, device="cuda"), ms)
    assert np.array_equal(g2["obs"].cpu().numpy(), x[:N]) and np.array_equal(g2["mask"].cpu().numpy(), planes[:, :N])
    venv.close()


def test_ppo_update_metrics_on_runner_rollout_match_independent_computation(torch):
    """One epoch, one minibatch = the whole buffer, eval mode (no dropout / batch-stat noise):
    the metrics of PPOAgent.update must equal ppo.py:372-406 evaluated with the oracle's
    masked log-prob / entropy on the same logits."""
    from bbgpu.ppo import PPOAgent, PPOConfig
    from bbgpu.rollout import RolloutBuffer
    from bbgpu.train import RolloutRunner
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    from bbgpu import vec_env as VE
    from oracle import bb_oracle as O
    torch.manual_seed(0)
    T, N = 8, 64
    agent = PPOAgent(PPOConfig(num_epochs=1, batch_size=T * N, learning_rate=1e-3))
    agent.eval()
    venv = VectorizedBlockBlastEnv(N, seed=9, output="packed")
    venv.reset()
    buf = RolloutBuffer(T, N)
    last = RolloutRunner(venv, agent, buf, use_graph=False).run()
    assert (buf.rewards > -5).all()                   # K3 only samples valid actions
    # independent expectation, before the update changes the weights
    g = buf.gather(torch.arange(T * N, device="cuda"), None)
    dense = VE.expand_mask(g["mask"].cpu().numpy().view(np.uint64)).astype(np.float32)
    with torch.no_grad():
        logits, values = agent.network.trunk(g["obs"])
    adv, ret = O.gae(buf.rewards.cpu().numpy(), buf.values.cpu().numpy(), buf.dones.cpu().numpy(), last.cpu().numpy(), 0.99, 0.95)
    a_n = O.normalize_advantages(adv)
    acts = buf.actions.view(-1).cpu().numpy()
    _, new_lp, ent = O.masked_policy_terms(logits.cpu().numpy(), dense, acts)
    old_lp = buf.log_probs.view(-1).cpu().numpy()
    np.testing.assert_allclose(new_lp, old_lp, rtol=1e-4, atol=1e-5)     # K3's log-prob == oracle's on the same weights
    ratio = np.exp(new_lp - old_lp)
    pol = -np.minimum(ratio * a_n, np.clip(ratio, 0.8, 1.2) * a_n).mean()
    vl = ((values.cpu().numpy() - ret.reshape(-1)) ** 2).mean()
    before = [p.detach().clone() for p in agent.network.parameters()]
    m = agent.update(buf, last)
    assert abs(m["policy_loss"] - pol) < 1e-4 and abs(m["value_loss"] - vl) < 1e-3 * max(1.0, vl)
    assert abs(m["entropy"] - ent.mean()) < 1e-4
    assert abs(m["total_loss"] - (pol + 0.5 * vl - 0.01 * ent.mean())) < 1e-3 * max(1.0, vl)
    assert m["clip_fraction"] < 1e-3 and abs(m["approx_kl"]) < 1e-4
    assert any(not torch.equal(a, b) for a, b in zip(before, agent.network.parameters()))
    venv.close()


def test_short_training_run_and_checkpoint_keys(torch, tmp_path):
    from bbgpu.train import train
    from bbgpu.ppo import PPOAgent
    cfg = {"training": {"num_envs": 256, "batch_size": 1024, "rollout_steps": 16, "total_timesteps": 3 * 256 * 16},
           "ppo": {"num_epochs": 2}, "logging": {"log_interval": 1, "save_interval": 1},
           "paths": {"checkpoint_dir": str(tmp_path / "ck"), "log_dir": str(tmp_path / "logs")}}
    hist = train(cfg, seed=42)
    assert len(hist) == 3 and hist[-1]["step"] == 3 * 256 * 16
    assert 5 < hist[-1]["avg_length"] < 40 and hist[-1]["episodes"] > 50
    assert np.isfinite([h["policy_loss"] for h in hist]).all() and hist[0]["entropy"] > 0.5
    ck = torch.load(str(tmp_path / "ck" / "final.pt"), weights_only=False)
    # the reference's three keys (ppo.py:425-431) + our resume position, which its load() ignores
    assert set(ck.keys()) == {"network_state_dict", "optimizer_state_dict", "config", "b200_state"}
    assert "conv_encoder.0.weight" in ck["network_state_dict"] and ck["config"]["num_epochs"] == 2
    a = PPOAgent()
    a.load(str(tmp_path / "ck" / "final.pt"))
    assert os.path.exists(str(tmp_path / "ck" / "latest.pt")) and os.path.exists(str(tmp_path / "ck" / ("checkpoint_%d.pt" % (3 * 256 * 16))))
    # numpy-facing API of the agent on the reference-layout observation
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    v = VectorizedBlockBlastEnv(8, seed=1)
    obs, _ = v.reset()
    acts, lps, vals = a.select_actions(obs)
    assert acts.shape == (8,) and lps.shape == (8,) and vals.shape == (8,)
    assert all(obs["action_mask"][i, acts[i]] for i in range(8))
    act1, info = a.select_action({k: obs[k][0] for k in ("board", "pieces", "action_mask")}, deterministic=True)
    assert obs["action_mask"][0, act1] == 1 and set(info) == {"log_prob", "entropy", "value"}
    assert a.get_values(obs).shape == (8,)
    v.close()


def test_batched_deterministic_evaluation(torch):
    """scripts/evaluate.py semantics, batched: one episode per env, argmax policy, reproducible."""
    from bbgpu.evaluate import evaluate
    from bbgpu.ppo import PPOAgent
    torch.manual_seed(1)
    agent = PPOAgent()
    r1 = evaluate(agent, num_episodes=200, seed=3)
    r2 = evaluate(agent, num_episodes=200, seed=3)
    assert r1["finished"] == 200 and np.array_equal(r1["scores"], r2["scores"]) and np.array_equal(r1["lengths"], r2["lengths"])
    assert 3 < r1["mean_length"] < 60 and r1["min_score"] > 0 and r1["max_score"] >= r1["mean_score"]
    assert agent.training            # mode restored


def test_evaluation_episodes_replay_through_the_oracle(torch):
    """scripts/evaluate.py:23-90 semantics against the oracle: every env plays ONE episode with the argmax
    policy in eval mode; the logged action sequences are replayed through the Python oracle (reference
    single-env semantics, no auto-reset) fed the same Philox trio streams — per-episode final score, length,
    lines cleared, max combo and summed reward must be identical, and every logged action must be the argmax
    of a valid action (never rejected)."""
    from bbgpu import philox
    from bbgpu.evaluate import evaluate
    from bbgpu.ppo import PPOAgent
    from oracle import bb_oracle as O
    torch.manual_seed(5)
    agent = PPOAgent()
    n, seed = 48, 9
    res = evaluate(agent, num_episodes=n, seed=seed, return_actions=True)
    assert res["finished"] == n and res["actions"].shape[1] == n
    streams = philox.candidate_trios(seed, np.arange(n), 1024)
    for i in range(n):
        it = iter(streams[i])
        env = O.Env(draw=lambda: next(it))
        total, t, term, info = 0.0, 0, False, None
        while not term:
            _, r, term, _, info = env.step(int(res["actions"][t, i]))
            assert not info["invalid_action"], (i, t)
            total += float(np.float32(r))
            t += 1
        assert info["score"] == res["scores"][i] and info["moves"] == res["lengths"][i] == t, (i, info, res["scores"][i])
        assert info["lines_cleared"] == res["lines"][i] and info["max_combo"] == res["max_combos"][i]
        assert abs(total - res["rewards_per_episode"][i]) < 1e-4 * max(1.0, abs(total))
    assert res["mean_score"] == float(res["scores"].mean()) and res["max_length"] == int(res["lengths"].max())


class _ReferenceAgentOnCPU:
    """The reference's PPOAgent as far as loading a checkpoint goes (src/agents/ppo.py:246, :252, :433-439):
    a BlockBlastNetwork on the CPU (test_network_is_state_dict_compatible_with_reference pins the module against
    the reference's recorded outputs), a plain Adam(lr, eps=1e-5) over its parameters, and load = torch.load with
    its defaults, network.load_state_dict(ck['network_state_dict']) and optimizer.load_state_dict(ck['optimizer_state_dict'])."""

    def __init__(self, torch):
        from bbgpu.network import BlockBlastNetwork
        from bbgpu.ppo import PPOConfig
        self.torch = torch
        self.network = BlockBlastNetwork()
        self.optimizer = torch.optim.Adam(self.network.parameters(), lr=PPOConfig().learning_rate, eps=1e-5)

    def load(self, path):
        ck = self.torch.load(path, map_location="cpu")
        self.network.load_state_dict(ck["network_state_dict"])
        self.optimizer.load_state_dict(ck["optimizer_state_dict"])


def test_checkpoint_loads_in_the_references_own_agent(torch, tmp_path):
    """PPOAgent.save -> the reference's PPOAgent.load (src/agents/ppo.py:433-439) on the CPU: same
    parameters, the optimizer state accepted, and the loaded network then computes the logits and values
    our network computes on the same observation (fp32) and keeps training from the loaded state."""
    from bbgpu.ppo import PPOAgent
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    torch.manual_seed(2)
    mine = PPOAgent()
    venv = VectorizedBlockBlastEnv(32, seed=4, output="packed")
    from bbgpu.rollout import RolloutBuffer
    from bbgpu.train import RolloutRunner
    buf = RolloutBuffer(8, 32)
    lv = RolloutRunner(venv, mine, buf, use_graph=False).run()
    mine.update(buf, lv)                                   # so that the optimizer has state to save
    path = str(tmp_path / "ck.pt")
    mine.save(path)
    theirs = _ReferenceAgentOnCPU(torch)
    theirs.load(path)
    sd_m, sd_t = mine.network.state_dict(), theirs.network.state_dict()
    assert set(sd_m) == set(sd_t)
    for k in sd_m:
        assert torch.equal(sd_m[k].cpu(), sd_t[k]), k
    assert len(theirs.optimizer.state_dict()["state"]) == len(mine.optimizer.state_dict()["state"])
    nv = VectorizedBlockBlastEnv(16, seed=8)
    obs, _ = nv.reset()
    mine.eval(); theirs.network.eval()
    with torch.no_grad():
        lg_t, v_t = theirs.network(torch.from_numpy(obs["board"]), torch.from_numpy(obs["pieces"]))
        lg_m, v_m = mine.network(torch.from_numpy(obs["board"]).cuda(), torch.from_numpy(obs["pieces"]).cuda())
    assert torch.allclose(lg_t, lg_m.cpu(), atol=2e-3, rtol=2e-3) and torch.allclose(v_t, v_m.cpu(), atol=2e-3, rtol=2e-3)
    theirs.optimizer.zero_grad()                           # and it can keep training from the loaded state
    m = torch.from_numpy(obs["action_mask"]).float()
    a, lp, ent, val = theirs.network.get_action_and_value(torch.from_numpy(obs["board"]), torch.from_numpy(obs["pieces"]),
                                                          m, action=lg_t.masked_fill(m == 0, float("-inf")).argmax(1))
    (-(lp.mean()) + val.pow(2).mean()).backward()
    theirs.optimizer.step()
    nv.close(); venv.close()


def test_vectorized_env_infos_match_oracle_including_terminal_observation(torch):
    """infos[i] of every step (block_blast_env.py:266-288) and, for finished episodes, the
    terminal statistics, final_score and terminal_observation (wrappers.py:97-100), against the
    Python oracle fed the same Philox trio streams."""
    from bbgpu import philox
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    from oracle import bb_oracle as O
    n, seed, T = 16, 77, 260
    streams = philox.candidate_trios(seed, np.arange(n), 600)

    def mk(i):
        it = iter(streams[i])
        return O.Env(draw=lambda: next(it))
    ora = O.VecEnv([mk(i) for i in range(n)])          # each oracle env dealt draw 0 in its constructor
    venv = VectorizedBlockBlastEnv(n, seed=seed)        # ... like bb_env_create; no further reset on either side
    rs = np.random.RandomState(4)
    n_term = 0
    for t in range(T):
        masks = venv.get_action_masks()
        acts = np.array([int(rs.choice(np.where(masks[i])[0])) if rs.rand() > 0.05 else int(rs.randint(0, 192)) for i in range(n)])
        oobs, orew, oterm, _, oinfos = ora.step(acts)
        gobs, grew, gterm, gtrunc, ginfos = venv.step(acts)
        assert np.array_equal(orew.view(np.uint32), grew.view(np.uint32)) and np.array_equal(oterm, gterm)
        for i in range(n):
            oi, gi = oinfos[i], ginfos[i]
            for k in ("score", "moves", "lines_cleared", "max_combo", "blocks_placed", "holes", "invalid_action"):
                assert oi[k] == gi[k], (t, i, k, oi[k], gi[k])
            assert abs(oi["board_fill"] - gi["board_fill"]) < 1e-12
            assert ("last_move" in oi) == ("last_move" in gi), (t, i)
            if "last_move" in oi:
                assert oi["last_move"] == gi["last_move"], (t, i, oi["last_move"], gi["last_move"])
            if oterm[i]:
                n_term += 1
                assert gi["final_score"] == oi["final_score"]
                for k in ("board", "pieces", "action_mask"):
                    assert np.array_equal(oi["terminal_observation"][k], gi["terminal_observation"][k]), (t, i, k)
            else:
                assert "final_score" not in gi
    assert n_term > 100
    venv.close()


def test_flat_view_and_game_state_restore(torch):
    """BlockBlastEnvFlat (block_blast_env.py:326-389) and GameState get/set (engine.py:456-476)
    over a slot of the batched state."""
    import json
    from bbgpu import philox
    from bbgpu.vec_env import BlockBlastEnv, BlockBlastEnvFlat, GameState
    from oracle import bb_oracle as O
    seed = 33
    flat = BlockBlastEnvFlat(seed=seed)
    ref = BlockBlastEnv(seed=seed)
    assert flat.observation_space["obs"].shape == (178,)
    rs = np.random.RandomState(1)
    for step in range(25):
        fo, ro = flat._get_observation(), ref._get_observation()
        st = ref.get_state()
        assert fo["obs"].dtype == np.float32 and fo["obs"].shape == (178,)
        assert np.array_equal(fo["obs"][:64], ro["board"].reshape(64))
        assert np.array_equal(fo["action_mask"], ro["action_mask"])
        onehot = fo["obs"][64:175].reshape(3, 37)
        for i in range(3):
            if st.pieces_used[i]:
                assert onehot[i].sum() == 0 and fo["obs"][175 + i] == 1.0 and ro["pieces"][i].sum() == 0
            else:
                assert onehot[i].argmax() == st.current_pieces[i] and onehot[i].sum() == 1 and fo["obs"][175 + i] == 0.0
                plane = np.zeros((8, 8), np.float32)
                for dr, dc in O.PIECE_CELLS[st.current_pieces[i]]:
                    plane[dr, dc] = 1.0
                assert np.array_equal(ro["pieces"][i], plane)
        va = ref.get_valid_actions()
        if not va:
            break
        a = int(va[rs.randint(len(va))])
        r1 = flat.step(a)
        r2 = ref.step(a)
        assert r1[1] == r2[1] and r1[2] == r2[2]
        if r2[2]:
            break
    # serialise mid-game, restore into a fresh env with another seed: same position, same rules
    st = ref.get_state()
    blob = json.dumps(st.to_dict())
    other = BlockBlastEnv(seed=999)
    other.set_state(GameState.from_dict(json.loads(blob)))
    o1, o2 = ref._get_observation(), other._get_observation()
    for k in ("board", "pieces", "action_mask"):
        assert np.array_equal(o1[k], o2[k]), k
    i1, i2 = ref._get_info(), other._get_info()
    assert (i1["score"], i1["moves"], i1["holes"]) == (i2["score"], i2["moves"], i2["holes"])
    st2 = other.get_state()
    assert st2.to_dict() == st.to_dict()
    va = other.get_valid_actions()
    if va and sum(st.pieces_used) < 2:        # a move that does not trigger a deal is RNG-free
        a = va[0]
        (oa, ra, ta, _, ia), (ob, rb, tb, _, ib) = ref.step(a), other.step(a)
        assert ra == rb and ta == tb and np.array_equal(oa["board"], ob["board"]) and ia["score"] == ib["score"]
    # a game-over state restores as game over: every action rejected
    st.status = "game_over"
    other.set_state(st)
    _, r, t, _, info = other.step(0)
    assert r == -10.0 and not t and info["invalid_action"] and other.get_state().status == "game_over"
    for e in (flat, ref, other):
        e.close()


@pytest.mark.parametrize("use_graph", [False, True])
def test_rollout_runner_rows_replay_through_the_oracle(torch, use_graph):
    """train.RolloutRunner writes every rollout result in place (K3 -> buffer.actions / log_probs, K1 ->
    rewards / terminated / next packed observation row) and, with use_graph, replays the whole rollout as
    one CUDA graph.  Three consecutive rollouts (eager first, then capture + replay) are replayed through
    the C oracle fed the same Philox trio streams and the recorded actions: rewards (bit patterns), done
    flags, boards, pieces and masks of every step must be identical, the episode statistics K1
    accumulates must equal the oracle's, and log-probs / values must be those of the actions' rows."""
    from bbgpu import philox
    from bbgpu.ppo import PPOAgent, PPOConfig
    from bbgpu.rollout import RolloutBuffer
    from bbgpu.train import RolloutRunner
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    from oracle import bb_oracle_c as OC
    n, T, seed = 96, 24, 11
    torch.manual_seed(0)
    agent = PPOAgent(PPOConfig(precision="bf16"), seed=seed)
    agent.train()
    venv = VectorizedBlockBlastEnv(n, seed=seed, output="packed")      # dealt once at creation, like the oracle envs
    ora = OC.CVecEnv(philox.candidate_trios(seed, np.arange(n), 2048))
    buf = RolloutBuffer(T, n)
    runner = RolloutRunner(venv, agent, buf, use_graph=use_graph)
    eps = score = length = 0
    for it in range(3):
        lv = runner.run()
        torch.cuda.synchronize()
        assert buf.full and lv.shape == (n,) and torch.isfinite(lv).all()
        acts = buf.actions.cpu().numpy()
        rew, term = buf.rewards.cpu().numpy(), buf.terminated.cpu().numpy()
        boards = buf.boards.cpu().numpy().view(np.uint64)
        pieces = buf.pieces.cpu().numpy().view(np.uint8).reshape(T + 1, n, 4)
        masks = buf.action_masks.cpu().numpy().view(np.uint64)
        assert np.array_equal(buf.dones.cpu().numpy(), term.astype(np.float32))
        b0, p0, m0 = ora.export()
        assert np.array_equal(boards[0], b0) and np.array_equal(pieces[0], p0) and np.array_equal(masks[0].T, m0)
        for t in range(T):
            # the sampled action is valid under the mask of the row it was sampled on
            a = acts[t]
            assert ((masks[t][a // 64, np.arange(n)] >> (a % 64).astype(np.uint64)) & np.uint64(1)).all(), (it, t)
            oo = ora.step(a)
            assert not oo["invalid"].any()
            assert np.array_equal(oo["rewards"].view(np.uint32), rew[t].view(np.uint32)), (it, t)
            assert np.array_equal(oo["terminated"], term[t]), (it, t)
            assert np.array_equal(oo["mask"], masks[t + 1].T), (it, t)
            assert np.array_equal(oo["board"], boards[t + 1]) and np.array_equal(oo["pieces"], pieces[t + 1]), (it, t)
            done = oo["terminated"].astype(bool)
            eps += int(done.sum())
            score += int(oo["ep_score"][done].sum())
            length += int(oo["ep_len"][done].sum())
        assert torch.isfinite(buf.log_probs).all() and (buf.log_probs <= 0).all() and torch.isfinite(buf.values).all()
    st = venv.episode_stats.cpu().tolist()
    assert st[0] == 3 * n * T and st[1] == eps and eps > 20 and st[2] == score and st[3] == length
    # one PPO update from the in-place buffer (graph-replayed minibatch step on the second call)
    for _ in range(2):
        m = agent.update(buf, lv, use_graph=use_graph)
        assert all(np.isfinite(v) for v in m.values()) and m["entropy"] > 0.1
    venv.close()


@pytest.mark.parametrize("obs_dtype", ["float32", "bfloat16"])
def test_gather_minibatch_equals_fancy_indexing(torch, obs_dtype):
    """bb_gather_minibatch (RolloutBuffer.gather) against the reference's own recipe for a minibatch
    (ppo.py:171-213): flatten (T, N), normalise the advantages over the whole buffer, fancy-index every
    array with the sample indices — board / piece planes through K2 on the gathered packed words."""
    from bbgpu import capi
    from bbgpu.rollout import RolloutBuffer
    T, N, B = 6, 37, 101
    g = torch.Generator(device="cuda").manual_seed(3)
    buf = RolloutBuffer(T, N)
    buf.boards[:T] = torch.randint(-2 ** 62, 2 ** 62, (T, N), device="cuda", generator=g)
    buf.pieces[:T] = (torch.randint(0, 37, (T, N), device="cuda", generator=g) | (torch.randint(0, 37, (T, N), device="cuda", generator=g) << 8)
                      | (torch.randint(0, 37, (T, N), device="cuda", generator=g) << 16) | (torch.randint(0, 8, (T, N), device="cuda", generator=g) << 24)).int()
    buf.action_masks[:T] = torch.randint(-2 ** 62, 2 ** 62, (T, 3, N), device="cuda", generator=g)
    buf.actions.copy_(torch.randint(0, 192, (T, N), device="cuda", generator=g))
    for t in (buf.log_probs, buf.advantages, buf.returns):
        t.copy_(torch.randn(T, N, device="cuda", generator=g))
    idx = torch.randint(0, T * N, (B,), device="cuda", generator=g)           # with repeats
    mean, std = buf.advantages.mean(), buf.advantages.std(unbiased=False)
    dt = getattr(torch, obs_dtype)
    out = buf.gather(idx, torch.stack([mean, std]).float(), obs_dtype=dt)
    torch.cuda.synchronize()
    t_i, n_i = idx // N, idx % N
    assert torch.equal(out["actions"], buf.actions[t_i, n_i]) and torch.equal(out["logp"], buf.log_probs[t_i, n_i])
    assert torch.equal(out["ret"], buf.returns[t_i, n_i])
    assert torch.equal(out["mask"], buf.action_masks[t_i, :, n_i].t().contiguous())
    want_adv = (buf.advantages[t_i, n_i] - mean) / (std + 1e-8)
    torch.testing.assert_close(out["adv"], want_adv, rtol=1e-6, atol=1e-6)
    ref = torch.empty((B, 4, 8, 8), dtype=dt, device="cuda")
    capi.unpack_obs(buf.boards[t_i, n_i].contiguous(), buf.pieces[t_i, n_i].contiguous(), out["mask"], B, obs=ref, n=B)
    assert torch.equal(out["obs"], ref) and out["obs"].dtype == dt
    assert float(out["obs"][:, 0].float().sum()) == float(sum(bin(int(x) & (2 ** 64 - 1)).count("1") for x in buf.boards[t_i, n_i].tolist()))


def test_dense_add_stores_the_packed_rows(torch):
    """RolloutBuffer.add with the reference's dense arrays packs them into the rows the env writes:
    gather gives the same minibatch as from a buffer filled with those packed rows, PPOAgent.update
    runs on it (three minibatches, the last one short), and a piece plane that is not a piece at the
    origin is rejected."""
    from bbgpu import vec_env as VE
    from bbgpu.ppo import PPOAgent, PPOConfig
    from bbgpu.rollout import RolloutBuffer
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    T, N = 4, 64
    venv = VectorizedBlockBlastEnv(N, seed=3, output="packed")
    obs, _ = venv.reset()
    dense_buf, packed_buf = RolloutBuffer(T, N), RolloutBuffer(T, N)
    rs = np.random.RandomState(2)
    for t in range(T):
        act = venv.sample_valid_actions()
        lp, val = (torch.from_numpy(rs.randn(N).astype(np.float32)).cuda() for _ in range(2))
        row = tuple(obs[k].clone() for k in ("board", "pieces", "mask"))
        obs, rew, term, _, _ = venv.step(act)
        packed_buf.add(*row, act, lp, rew, term.float(), val)
        b, p, m = (x.cpu().numpy() for x in row)
        dense_buf.add(VE.expand_board(b.view(np.uint64)), VE.expand_pieces(p.view(np.uint32)),
                      VE.expand_mask(m.view(np.uint64)), act.cpu().numpy(), lp.cpu().numpy(), rew.cpu().numpy(),
                      term.float().cpu().numpy(), val.cpu().numpy())
    assert ((packed_buf.pieces[:T] >> 24) & 7).any()           # used slots (all-zero planes) are covered
    last = torch.from_numpy(rs.randn(N).astype(np.float32)).cuda()
    for buf in (dense_buf, packed_buf):
        buf.compute_returns_and_advantages(last, 0.99, 0.95)
    ms = torch.stack(packed_buf.advantage_mean_std())
    idx = torch.randperm(T * N, device="cuda")
    gd, gp = dense_buf.gather(idx, ms), packed_buf.gather(idx, ms)
    for k in gp:
        assert torch.equal(gd[k], gp[k]), k
    agent = PPOAgent(PPOConfig(num_epochs=1, batch_size=100))
    metrics = agent.update(dense_buf, last)
    assert all(np.isfinite(v) for v in metrics.values())
    bad = VE.expand_pieces(p.view(np.uint32)).copy()
    bad[5, 1] = 0
    bad[5, 1, 7, 7] = 1                                         # one cell, but not at the origin
    with pytest.raises(ValueError):
        RolloutBuffer(1, N).add(VE.expand_board(b.view(np.uint64)), bad, VE.expand_mask(m.view(np.uint64)),
                                np.zeros(N, np.int64), *(np.zeros(N, np.float32),) * 4)
    venv.close()


def test_get_samples_equals_the_torch_formula_bitwise(torch):
    """get_samples (gather + one dense-mask expansion per minibatch) yields, bit for bit, what the
    torch statement of ppo.py:171-213 yields on the same permutation: float32 advantages
    (a - mean) / (std + 1e-8), fancy-indexed scalars, K2-expanded planes and dense mask."""
    from bbgpu import capi
    from bbgpu.rollout import RolloutBuffer
    T, N, B = 6, 37, 64                                          # 222 samples: the last minibatch is short
    g = torch.Generator(device="cuda").manual_seed(5)
    buf = RolloutBuffer(T, N)
    buf.boards[:T] = torch.randint(-2 ** 62, 2 ** 62, (T, N), device="cuda", generator=g)
    buf.pieces[:T] = (torch.randint(0, 37, (T, N), device="cuda", generator=g) | (torch.randint(0, 37, (T, N), device="cuda", generator=g) << 8)
                      | (torch.randint(0, 37, (T, N), device="cuda", generator=g) << 16) | (torch.randint(0, 8, (T, N), device="cuda", generator=g) << 24)).int()
    buf.action_masks[:T] = torch.randint(-2 ** 62, 2 ** 62, (T, 3, N), device="cuda", generator=g)
    buf.actions.copy_(torch.randint(0, 192, (T, N), device="cuda", generator=g))
    for t in (buf.log_probs, buf.rewards, buf.values):
        t.copy_(torch.randn(T, N, device="cuda", generator=g))
    buf.dones.copy_((torch.rand(T, N, device="cuda", generator=g) < 0.1).float())
    buf.compute_returns_and_advantages(torch.randn(N, device="cuda", generator=g), 0.99, 0.95)
    torch.manual_seed(8)
    got = list(buf.get_samples(B))
    torch.manual_seed(8)
    perm = torch.randperm(T * N, device="cuda")
    mean, std = buf.advantage_mean_std()
    adv = (buf.advantages.view(-1) - mean) / (std + 1e-8)
    assert len(got) == 4
    for i, start in enumerate(range(0, T * N, B)):
        idx = perm[start:start + B]
        n = idx.numel()
        masks = buf.action_masks[idx // N, :, idx % N].t().contiguous()
        obs = torch.empty((n, 4, 8, 8), dtype=torch.float32, device="cuda")
        dense = torch.empty((n, 192), dtype=torch.float32, device="cuda")
        capi.unpack_obs(buf.boards.view(-1)[idx], buf.pieces.view(-1)[idx], masks, n, obs=obs, mask_dense=dense, n=n)
        want = (obs[:, 0], obs[:, 1:], dense, buf.actions.view(-1)[idx].long(), buf.log_probs.view(-1)[idx], adv[idx],
                buf.returns.view(-1)[idx])
        for k, (w, h) in enumerate(zip(want, got[i])):
            assert h.dtype == w.dtype and h.shape == w.shape, (i, k)
            if w.dtype == torch.float32:
                w, h = w.view(torch.int32), h.view(torch.int32)
            assert torch.equal(h, w), (i, k)
