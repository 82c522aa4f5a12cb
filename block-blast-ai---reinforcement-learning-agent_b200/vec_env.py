"""Drop-in mirrors of the reference's environment classes on top of the CUDA env kernels.

``VectorizedBlockBlastEnv``  <- src/environment/wrappers.py:14-141
``BlockBlastEnv``            <- src/environment/block_blast_env.py:20-323 (single env, no auto-reset)

Same constructor arguments, method names, return arity, shapes and dtypes.  All game logic
runs in ``libbbgpu.so`` (one fused kernel per vec step); this file only moves buffers and
reshapes the packed observation into the reference's layout.

Output modes (``output=``):
  "numpy"   reference-compatible: numpy obs dict / rewards / terminated / truncated / infos.
            ``obs_format="dense"`` (default): the observation arrives in the reference's own layout
            (board (N,8,8) f32, pieces (N,3,8,8) f32, action_mask (N,192) int8), expanded on the
            device and copied in one 1,221 B/env transfer (``bb_env_step_host_dense``) — what a
            caller that reads the arrays every step (PPOAgent.select_actions) wants.
            ``obs_format="lazy"``: one packed D2H copy (41 B/env, ``bb_env_step_host``); the dense
            arrays are expanded on the host only if somebody asks for them (``LazyObs``) — for
            callers that consume the packed protocol or touch few observations.
  "torch"   same keys and shapes, CUDA tensors, nothing crosses PCIe (K2 expands on device).
  "packed"  CUDA tensors in the packed protocol: obs = {'board': int64[N], 'pieces': int32[N],
            'mask': int64[3,N]} — what the on-device rollout path consumes.
"""
import dataclasses
import os

import numpy as np

from . import capi

BOARD_SIZE = 8
NUM_PIECES_PER_TURN = 3
ACTION_SPACE_SIZE = 192


class _Box:
    def __init__(self, low, high, shape, dtype):
        self.low, self.high, self.shape, self.dtype = low, high, shape, dtype


class _Discrete:
    def __init__(self, n):
        self.n = n

    def sample(self):
        return int(np.random.randint(self.n))


class _DictSpace:
    def __init__(self, spaces):
        self.spaces = dict(spaces)

    def __getitem__(self, k):
        return self.spaces[k]


def _spaces():
    obs = _DictSpace({
        "board": _Box(0.0, 1.0, (8, 8), np.float32),
        "pieces": _Box(0.0, 1.0, (3, 8, 8), np.float32),
        "action_mask": _Box(0, 1, (ACTION_SPACE_SIZE,), np.int8),
    })
    return obs, _Discrete(ACTION_SPACE_SIZE)


_PIECE_PLANES = None


def piece_planes():
    """float32 [38, 8, 8]: piece i drawn at the origin (Piece.to_mask, pieces.py:39-45);
    index 37 is the all-zero plane of a used piece.  Built from the library's own table."""
    global _PIECE_PLANES
    if _PIECE_PLANES is None:
        masks, _, _ = capi.piece_table()
        bits = np.unpackbits(masks.view(np.uint8).reshape(37, 8), axis=1, bitorder="little")
        planes = np.zeros((38, 8, 8), np.float32)
        planes[:37] = bits.reshape(37, 8, 8)
        _PIECE_PLANES = planes
    return _PIECE_PLANES


def expand_board(board_u64):
    b = np.ascontiguousarray(board_u64, dtype=np.uint64)
    return np.unpackbits(b.view(np.uint8).reshape(-1, 8), axis=1, bitorder="little").reshape(-1, 8, 8).astype(np.float32)


def expand_pieces(pieces_u32):
    p = np.ascontiguousarray(pieces_u32, dtype=np.uint32)
    ids = np.stack([(p >> (8 * k)) & 0xFF for k in range(3)], axis=1).astype(np.int64)
    used = np.stack([(p >> (24 + k)) & 1 for k in range(3)], axis=1).astype(bool)
    return piece_planes()[np.where(used, 37, ids)]


def expand_mask(mask_planes_u64):
    m = np.ascontiguousarray(np.asarray(mask_planes_u64, dtype=np.uint64).T)      # [N,3]
    return np.unpackbits(m.view(np.uint8).reshape(-1, 24), axis=1, bitorder="little").astype(np.int8)


class LazyObs(dict):
    """Observation dict whose dense arrays are expanded from the packed host copy on first
    access (keys and layouts of wrappers.py:118-126)."""

    def __init__(self, board, pieces, mask):
        super().__init__()
        self.packed = dict(board=board, pieces=pieces, mask=mask)

    def __missing__(self, key):
        if key == "board":
            v = expand_board(self.packed["board"])
        elif key == "pieces":
            v = expand_pieces(self.packed["pieces"])
        elif key == "action_mask":
            v = expand_mask(self.packed["mask"])
        else:
            raise KeyError(key)
        self[key] = v
        return v

    def keys(self):
        return ["board", "pieces", "action_mask"]

    def __iter__(self):
        return iter(self.keys())

    def __len__(self):
        return 3

    def items(self):
        return [(k, self[k]) for k in self.keys()]

    def __contains__(self, k):
        return k in ("board", "pieces", "action_mask")


def _last_move(word):
    """info word -> the reference's info['last_move'] (block_blast_env.py:281-286)."""
    return {"blocks_placed": (word >> 4) & 0xF, "lines_cleared": (word >> 1) & 7,
            "combo_multiplier": (word >> 8) & 7, "score_gained": (word >> 18) & 0x3FFF}


class LazyInfos:
    """Sequence of per-env info dicts (block_blast_env.py:266-288) built on demand.

    The training loop only reads ``final_score``/``score`` and ``moves`` of terminated envs
    (scripts/train.py:196-201); those come from the step's own outputs.  The other fields are
    read from the env state when first asked for (one device->host state copy)."""

    def __init__(self, venv, terminated, invalid, ep_score, ep_len, fetch=None):
        self._venv, self._term, self._inv = venv, terminated, invalid
        self._eps, self._epl = ep_score, ep_len
        self._fetch = fetch            # callable -> (info words, ep_score, ep_len): the step left them on the device
        self._state = None
        self._ends = None
        self._step_id = getattr(venv, "_step_id", 0)

    def _tail(self):
        """info word / ep_score / ep_len arrays of the step, fetched from the device on first use."""
        if self._fetch is not None:
            if self._step_id != getattr(self._venv, "_step_id", 0):
                raise RuntimeError("infos of an older step: the per-step info arrays have been overwritten")
            self._inv, self._eps, self._epl = self._fetch()
            self._fetch = None

    def _end(self, i):
        """Episode-end record of env i (terminal state), fetched from the device on first use."""
        if self._ends is None:
            if self._step_id != getattr(self._venv, "_step_id", 0):
                raise RuntimeError("infos of an older step: the episode-end log has been overwritten")
            self._ends = self._venv._d_ep_end.cpu().numpy().view(capi.EPISODE_END_DTYPE).copy()
        return self._ends[i]

    def __len__(self):
        return len(self._term)

    def _rec(self):
        if self._state is None:
            self._state = self._venv._handle.get_state()
        return self._state

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[k] for k in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        self._tail()
        if bool(self._term[i]):
            # the finished episode (the env itself has already been reset): wrappers.py:97-100
            e = self._end(i)
            return {"score": int(self._eps[i]), "final_score": int(self._eps[i]), "moves": int(self._epl[i]),
                    "lines_cleared": int(e["lines_total"]), "max_combo": int(e["max_streak"]),
                    "blocks_placed": int(e["blocks_total"]), "board_fill": (int(e["holes_fill"]) >> 8) / 64,
                    "holes": int(e["holes_fill"]) & 0xFF, "invalid_action": False,
                    "last_move": _last_move(int(e["last_move"])),
                    "terminal_observation": {"board": expand_board(np.array([e["board"]], np.uint64))[0],
                                             "pieces": expand_pieces(np.array([e["pieces"]], np.uint32))[0],
                                             "action_mask": np.zeros(ACTION_SPACE_SIZE, np.int8)}}
        s = self._rec()[i]
        board = int(s["board"])
        word = int(self._inv[i]) if self._inv is not None else 0          # the step's info word
        d = {"score": int(s["score"]), "moves": int(s["moves"]), "lines_cleared": int(s["lines_total"]),
             "max_combo": int(s["max_streak"]), "blocks_placed": int(s["blocks_total"]),
             "board_fill": bin(board).count("1") / 64, "holes": int(s["aux"] & 0xFF), "invalid_action": bool(word & 1)}
        if self._inv is not None and not (word & 1):
            d["last_move"] = _last_move(word)
        return d

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class VectorizedBlockBlastEnv:
    """Batched Block Blast env on one GPU (reference: wrappers.py:14-141).

    Extra keyword-only arguments (not in the reference): ``output`` (see module docstring),
    ``global_env_offset`` (id of env 0 of this shard — trajectories depend on
    ``(seed, global id, actions)`` only, so shards over several GPUs reproduce the one-GPU
    run), ``reseed_on_reset`` (the reference re-seeds env i with ``seed+i`` on EVERY reset when
    a seed is given, so each episode replays the same trio stream; default False = the stream
    continues, True = that behaviour)."""

    def __init__(self, num_envs, seed=None, reward_config=None, *, output="numpy",
                 global_env_offset=0, reseed_on_reset=False, reuse_buffers=False, obs_format="dense"):
        import torch
        assert output in ("numpy", "torch", "packed")
        assert obs_format in ("dense", "lazy")
        self.num_envs = int(num_envs)
        self.reward_config = reward_config
        self.output = output
        self.obs_format = obs_format
        self.global_env_offset = int(global_env_offset)
        self.reseed_on_reset = bool(reseed_on_reset)
        # numpy mode: False = every step returns fresh arrays (reference behaviour); True = zero-copy
        # views of two alternating pinned buffer sets, valid until the second-next step() call
        self.reuse_buffers = bool(reuse_buffers)
        self.seed = int.from_bytes(os.urandom(8), "little") if seed is None else int(seed)
        self.observation_space, self.action_space = _spaces()
        self.single_action_space = self.action_space
        self._torch = torch
        self._make_handle()
        n, dev = self.num_envs, self._handle.device
        # device-resident step outputs (reused every step)
        self._d_actions = torch.zeros(n, dtype=torch.int32, device=dev)
        self._d_rewards = torch.zeros(n, dtype=torch.float32, device=dev)
        self._d_term = torch.zeros(n, dtype=torch.uint8, device=dev)
        self._d_mask = torch.zeros((3, n), dtype=torch.int64, device=dev)
        self._d_board = torch.zeros(n, dtype=torch.int64, device=dev)
        self._d_pieces = torch.zeros(n, dtype=torch.int32, device=dev)
        self._d_ep_score = torch.zeros(n, dtype=torch.int32, device=dev)
        self._d_ep_len = torch.zeros(n, dtype=torch.int32, device=dev)
        self._d_info = torch.zeros(n, dtype=torch.int32, device=dev)
        self._d_ep_end = torch.zeros(n * 32, dtype=torch.uint8, device=dev)      # episode-end log (32 B records)
        self._handle.set_episode_end_buffer(self._d_ep_end)
        # episode statistics accumulated by the step kernel: env-steps, episodes, sum of final scores,
        # sum of episode lengths, max final score (what scripts/train.py:196-201 reads from infos)
        self.episode_stats = torch.zeros(8, dtype=torch.int64, device=dev)
        self._step_id = 0
        if output == "numpy":
            pin = dict(pin_memory=True)
            self._h_actions = torch.zeros(n, dtype=torch.int32, **pin)
            # two result sets (double buffering), each ONE pinned block in the library's layout so a
            # step's results arrive in a single transfer
            self._h_sets = [capi.pinned_result_block(n) for _ in range(2)]
            self._h_dense = [capi.pinned_dense_block(n) for _ in range(2)] if obs_format == "dense" else None
            self._h_flip = 0
        self._dones = np.zeros(n, dtype=bool)
        self._h_actions_np = self._h_actions.numpy() if output == "numpy" else None

    # ------------------------------------------------------------------ plumbing
    def _make_handle(self):
        flags = capi.ENV_RESEED_ON_RESET if self.reseed_on_reset else 0
        self._handle = capi.EnvHandle(self.num_envs, self.seed, self.global_env_offset, self.reward_config, flags)

    @property
    def handle(self):
        return self._handle

    def _obs_device(self, observe=True):
        """obs of the current states in the selected device format (observe=False: the step kernel
        has just written board / pieces / mask itself)."""
        torch = self._torch
        if observe:
            self._handle.observe(self._d_board, self._d_pieces, self._d_mask)
        if self.output == "packed":
            return {"board": self._d_board, "pieces": self._d_pieces, "mask": self._d_mask}
        n = self.num_envs
        obs = torch.empty((n, 4, 8, 8), dtype=torch.float32, device=self._d_board.device)
        dense = torch.empty((n, ACTION_SPACE_SIZE), dtype=torch.uint8, device=self._d_board.device)
        capi.unpack_obs(self._d_board, self._d_pieces, self._d_mask, n, obs=obs, mask_dense=dense)
        return {"board": obs[:, 0], "pieces": obs[:, 1:], "action_mask": dense.view(torch.int8), "nchw": obs}

    def _dense_views(self, d):
        keep = (lambda x: x) if self.reuse_buffers else (lambda x: x.copy())
        return {"board": keep(d["board"].numpy()), "pieces": keep(d["pieces"].numpy()),
                "action_mask": keep(d["action_mask"].numpy())}

    def _obs_numpy(self):
        t = self._torch
        if self.obs_format == "dense":
            d = self._h_dense[self._h_flip]
            self._handle.observe_host_dense(d["_block"])
            return self._dense_views(d)
        h = self._h_sets[self._h_flip]
        self._handle.observe(self._d_board, self._d_pieces, self._d_mask)
        h["board"].copy_(self._d_board, non_blocking=True)
        h["pieces"].copy_(self._d_pieces, non_blocking=True)
        h["mask"].copy_(self._d_mask, non_blocking=True)
        t.cuda.current_stream().synchronize()
        return LazyObs(h["board"].numpy().view(np.uint64).copy(), h["pieces"].numpy().view(np.uint32).copy(),
                       h["mask"].numpy().view(np.uint64).copy())

    # ------------------------------------------------------------------ reference API
    def reset(self, seed=None):
        """wrappers.py:53-73.  A non-None seed re-creates the Philox streams with it."""
        if seed is not None:
            self._handle.close()
            self.seed = int(seed)
            self._make_handle()     # deals once, like constructing the reference envs
            self._handle.set_episode_end_buffer(self._d_ep_end)
        self._handle.reset()
        self._dones.fill(False)
        obs = self._obs_numpy() if self.output == "numpy" else self._obs_device()
        return obs, LazyInfos(self, np.zeros(self.num_envs, bool), None, None, None)

    def step(self, actions):
        """wrappers.py:75-116: returns (obs, rewards, terminated, truncated, infos)."""
        torch = self._torch
        n = self.num_envs
        self._step_id += 1
        if self.output == "numpy":
            a = np.asarray(actions.cpu() if isinstance(actions, torch.Tensor) else actions).reshape(-1)
            assert a.shape[0] == n, "expected %d actions" % n
            if a is not self._h_actions_np:
                self._h_actions.numpy()[:] = a      # int cast like int(action) in wrappers.py:94
            self._h_flip ^= 1
            h = self._h_sets[self._h_flip]
            keep = (lambda x: x) if self.reuse_buffers else (lambda x: x.copy())

            def fetch(h=h, keep=keep):
                # info word / ep_score / ep_len stay on the device until somebody reads infos
                self._handle.fetch_step_info(h["ep_score"], h["ep_len"], h["info"])
                return keep(h["info"].numpy().view(np.uint32)), keep(h["ep_score"].numpy()), keep(h["ep_len"].numpy())

            if self.obs_format == "dense":
                d = self._h_dense[self._h_flip]
                self._handle.step_host_dense(self._h_actions, d["_block"])
                rewards = keep(d["rewards"].numpy())
                term = d["term"].numpy().view(bool) if self.reuse_buffers else d["term"].numpy().astype(bool)
                return (self._dense_views(d), rewards, term, np.zeros(n, dtype=bool),
                        LazyInfos(self, term, None, None, None, fetch))
            self._handle.step_host(self._h_actions, h["rewards"], h["term"], h["board"], h["pieces"], h["mask"],
                                   None, None, None)
            rewards = keep(h["rewards"].numpy())
            term = h["term"].numpy().view(bool) if self.reuse_buffers else h["term"].numpy().astype(bool)
            obs = LazyObs(keep(h["board"].numpy().view(np.uint64)), keep(h["pieces"].numpy().view(np.uint32)),
                          keep(h["mask"].numpy().view(np.uint64)))
            return obs, rewards, term, np.zeros(n, dtype=bool), LazyInfos(self, term, None, None, None, fetch)
        if isinstance(actions, torch.Tensor):
            self._d_actions.copy_(actions.reshape(-1), non_blocking=True)
        else:
            self._d_actions.copy_(torch.as_tensor(np.asarray(actions).reshape(-1).astype(np.int32)))
        # the step kernel writes the packed next observation itself (no separate observe launch)
        self._handle.step(self._d_actions, self._d_rewards, self._d_term, self._d_mask, self._d_ep_score,
                          self._d_ep_len, self._d_info, self._d_board, self._d_pieces, self.episode_stats)
        obs = self._obs_device(observe=False)
        term = self._d_term.bool()
        infos = {"ep_score": self._d_ep_score, "ep_len": self._d_ep_len, "info": self._d_info}
        return obs, self._d_rewards, term, torch.zeros_like(term), infos

    def step_into(self, actions, rewards, terminated, next_obs):
        """Device-resident step with caller-owned outputs (one kernel launch, nothing else):
        ``actions`` int32[N], ``rewards`` f32[N], ``terminated`` u8[N] and the packed observation after
        the step written straight into ``next_obs`` = {'board', 'pieces', 'mask'} — e.g. rows of a
        RolloutBuffer.  Episode statistics accumulate in ``self.episode_stats``."""
        self._step_id += 1
        self._handle.step(actions, rewards, terminated, next_obs["mask"], None, None, None, next_obs["board"],
                          next_obs["pieces"], self.episode_stats)

    def current_obs_into(self, obs):
        """Packed observation of the current states written into ``obs`` (device tensors)."""
        self._handle.observe(obs["board"], obs["pieces"], obs["mask"])

    def get_action_masks(self):
        """wrappers.py:128-131: bool [N,192]."""
        torch = self._torch
        self._handle.observe(None, None, self._d_mask)
        dense = torch.empty((self.num_envs, ACTION_SPACE_SIZE), dtype=torch.uint8, device=self._d_mask.device)
        capi.unpack_obs(None, None, self._d_mask, self.num_envs, obs=None, mask_dense=dense, n=self.num_envs)
        if self.output == "numpy":
            return dense.cpu().numpy().astype(bool)
        return dense.bool()

    def sample_valid_actions(self):
        """wrappers.py:133-136: a uniformly random valid action per env (0 if none), drawn by a
        Philox-keyed kernel (not numpy's global RNG)."""
        self._sample_ctr = getattr(self, "_sample_ctr", 0) + 1
        if self.output == "numpy":
            self._handle.sample_valid_actions(self._sample_ctr, None, self._h_actions)
            # reuse_buffers: hand back the pinned int32 buffer itself; step() recognises it and skips the copy
            return self._h_actions_np if self.reuse_buffers else self._h_actions_np.astype(np.int64)
        self._handle.sample_valid_actions(self._sample_ctr, self._d_actions, None)
        return self._d_actions.clone()

    def expand(self, samples=1):
        """One-ply look-ahead of every env's current state (bb_env_expand, ``capi.EnvHandle.expand``):
        one item per valid action (np.where(mask) order), ``samples`` items for an action that places
        the last unused piece (its new trio drawn from the LOOKAHEAD stream, not the env's own).
        Keys: offsets [N+1], action, reward, terminated, info, board, pieces [items], mask [3, items].
        No env state changes; every call advances this env's own expansion counter.  CUDA tensors in
        "torch" / "packed" mode, numpy copies in "numpy" mode."""
        self._expand_ctr = getattr(self, "_expand_ctr", 0) + 1
        out = self._handle.expand(self._expand_ctr, samples)
        if self.output == "numpy":
            out = {k: v.cpu().numpy() for k, v in out.items()}
            for k, dt in (("info", np.uint32), ("board", np.uint64), ("pieces", np.uint32), ("mask", np.uint64)):
                out[k] = out[k].view(dt)
        return out

    def close(self):
        self._handle.close()


class BlockBlastEnv:
    """Single environment with the reference's semantics (block_blast_env.py:20-323): no
    auto-reset — after game over every action is rejected with reward -10 until ``reset``.
    A view over a 1-env ``bb_env``; meant for evaluation / play, not throughput."""

    metadata = {"render_modes": ["human", "ansi"]}
    BOARD_SIZE = BOARD_SIZE
    NUM_PIECES_PER_TURN = NUM_PIECES_PER_TURN
    ACTION_SPACE_SIZE = ACTION_SPACE_SIZE

    def __init__(self, render_mode=None, reward_config=None, seed=None):
        import torch
        self._torch = torch
        self.render_mode = render_mode
        self.seed_value = seed
        self.reward_config = dict(capi.REWARD_DEFAULTS)
        if reward_config:
            self.reward_config.update(reward_config)
        self.observation_space, self.action_space = _spaces()
        self._open(seed)

    def _open(self, seed):
        torch = self._torch
        s = int.from_bytes(os.urandom(8), "little") if seed is None else int(seed)
        flags = capi.ENV_NO_AUTO_RESET | (capi.ENV_RESEED_ON_RESET if seed is not None else 0)
        self._h = capi.EnvHandle(1, s, 0, self.reward_config, flags)
        dev = self._h.device
        self._a = torch.zeros(1, dtype=torch.int32, device=dev)
        self._r = torch.zeros(1, dtype=torch.float32, device=dev)
        self._t = torch.zeros(1, dtype=torch.uint8, device=dev)
        self._m = torch.zeros((3, 1), dtype=torch.int64, device=dev)
        self._i = torch.zeros(1, dtype=torch.int32, device=dev)

    def _action_to_move(self, action):
        return action // 64, (action % 64) // 8, action % 8

    def _move_to_action(self, piece_idx, row, col):
        return piece_idx * 64 + row * 8 + col

    def _state(self):
        return self._h.get_state()[0]

    def _get_observation(self, s=None):
        s = self._state() if s is None else s
        self._h.observe(None, None, self._m)
        m = self._m.cpu().numpy().view(np.uint64)
        return {"board": expand_board(np.array([s["board"]]))[0], "pieces": expand_pieces(np.array([s["pieces"]]))[0],
                "action_mask": expand_mask(m)[0]}

    def _get_info(self, info_word=None, s=None):
        s = self._state() if s is None else s
        info = {"score": int(s["score"]), "moves": int(s["moves"]), "lines_cleared": int(s["lines_total"]),
                "max_combo": int(s["max_streak"]), "blocks_placed": int(s["blocks_total"]),
                "board_fill": bin(int(s["board"])).count("1") / 64, "holes": _holes(int(s["board"])),
                "invalid_action": False}
        if info_word is not None:
            info["last_move"] = _last_move(info_word)
        return info

    def reset(self, seed=None, options=None):
        if seed is not None:
            self.seed_value = seed
            self._h.close()
            self._open(seed)
        self._h.reset()
        return self._get_observation(), self._get_info()

    def step(self, action):
        torch = self._torch
        self._a.fill_(int(action))
        self._h.step(self._a, self._r, self._t, None, None, None, self._i)
        # one device->host read for the three step outputs, one state copy for obs and info
        word, rbits, term = torch.stack([self._i[0], self._r.view(torch.int32)[0], self._t[0].to(torch.int32)]).tolist()
        word &= 0xFFFFFFFF
        reward = float(np.array([rbits], np.int32).view(np.float32)[0])
        st = self._state()
        if word & 1:
            info = self._get_info(s=st)
            info["invalid_action"] = True
            return self._get_observation(st), -10.0, False, False, info
        return self._get_observation(st), reward, bool(term), False, self._get_info(word, st)

    def get_action_mask(self):
        return self._get_observation()["action_mask"].astype(bool)

    def get_valid_actions(self):
        return np.where(self.get_action_mask())[0].tolist()

    def sample_valid_action(self):
        va = self.get_valid_actions()
        return int(np.random.choice(va)) if va else 0

    # ---- GameState (de)serialisation over the env's slot of the batched state
    # (GameEngine.get_state/set_state + GameState.to_dict/from_dict, engine.py:44-78, 456-476)
    def get_state(self):
        s = self._state()
        board = expand_board(np.array([s["board"]]))[0].astype(np.int8)
        p = int(s["pieces"])
        return GameState(board=board, current_pieces=[p & 0xFF, (p >> 8) & 0xFF, (p >> 16) & 0xFF],
                         pieces_used=[bool((p >> (24 + i)) & 1) for i in range(3)], score=int(s["score"]),
                         combo_count=int(s["streak"]), moves_made=int(s["moves"]),
                         status="game_over" if (int(s["aux"]) >> 16) & 1 else "playing")

    def set_state(self, state):
        """Restore board, trio, used flags, score, combo and move counters (engine.py:466-476);
        the shaped-reward baselines (holes / centre filled) restart from the restored board, and
        the lifetime counters the reference does not serialise keep their values."""
        rec = self._h.get_state()
        grid = np.asarray(state.board).astype(bool).reshape(64)
        board = int(sum(1 << i for i in np.flatnonzero(grid)))
        ids = [int(i) for i in state.current_pieces]
        if len(ids) != 3 or any(not 0 <= i < 37 for i in ids):
            raise ValueError("current_pieces must be three piece indices in [0, 37)")
        used = sum((1 << i) for i, u in enumerate(state.pieces_used) if u)
        over = 1 if str(getattr(state.status, "value", state.status)) == "game_over" else 0
        rec["board"][0] = board
        rec["pieces"][0] = ids[0] | (ids[1] << 8) | (ids[2] << 16) | (used << 24)
        rec["aux"][0] = _holes(board) | (bin(board & 0x00003C3C3C3C0000).count("1") << 8) | (over << 16)
        rec["score"][0], rec["streak"][0], rec["moves"][0] = state.score, state.combo_count, state.moves_made
        self._h.set_state(rec)

    def render(self):
        return None

    def close(self):
        self._h.close()


@dataclasses.dataclass
class GameState:
    """The reference's serialisable game state (engine.py:44-78): same fields, same dict layout;
    ``status`` is the enum's string value ("playing" / "game_over")."""
    board: np.ndarray
    current_pieces: list
    pieces_used: list
    score: int
    combo_count: int
    moves_made: int
    status: str = "playing"

    def to_dict(self):
        return {"board": np.asarray(self.board).tolist(), "current_pieces": list(self.current_pieces),
                "pieces_used": list(self.pieces_used), "score": self.score, "combo_count": self.combo_count,
                "moves_made": self.moves_made, "status": str(getattr(self.status, "value", self.status))}

    @classmethod
    def from_dict(cls, data):
        return cls(board=np.array(data["board"], dtype=np.int8), current_pieces=list(data["current_pieces"]),
                   pieces_used=list(data["pieces_used"]), score=data["score"], combo_count=data["combo_count"],
                   moves_made=data["moves_made"], status=data["status"])


class BlockBlastEnvFlat(BlockBlastEnv):
    """Flat-observation view (block_blast_env.py:326-389): ``obs`` = board (64) + one-hot of each
    unused piece (3 x 37, all-zero when used) + used flags (3) = 178 floats, plus ``action_mask``."""

    def __init__(self, **kwargs):
        super().__init__(**kwargs)
        self.observation_space = _DictSpace({
            "obs": _Box(0.0, 1.0, (64 + 3 * 37 + 3,), np.float32),
            "action_mask": _Box(0, 1, (ACTION_SPACE_SIZE,), np.int8),
        })

    def _get_observation(self, s=None):
        s = self._state() if s is None else s
        base = super()._get_observation(s)
        p = int(s["pieces"])
        onehot = np.zeros((3, 37), np.float32)
        used = np.zeros(3, np.float32)
        for i in range(3):
            if (p >> (24 + i)) & 1:
                used[i] = 1.0
            else:
                onehot[i, (p >> (8 * i)) & 0xFF] = 1.0
        return {"obs": np.concatenate([base["board"].reshape(64), onehot.reshape(111), used]),
                "action_mask": base["action_mask"]}


def _holes(board):
    """Host-side restatement used only for the single-env info dict of a game-over state
    (aux carries the post-move value for live states)."""
    k = 0
    for r in range(8):
        for c in range(8):
            if (board >> (r * 8 + c)) & 1:
                continue
            ok = True
            for dr, dc in ((-1, 0), (1, 0), (0, -1), (0, 1)):
                rr, cc = r + dr, c + dc
                if 0 <= rr < 8 and 0 <= cc < 8 and not (board >> (rr * 8 + cc)) & 1:
                    ok = False
            k += ok
    return k
