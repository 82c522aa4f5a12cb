#!/usr/bin/env python3
"""bench.py — env-steps/s of the fused Block Blast step kernel (BASELINE.json config 3:
random valid-action policy, 262,144 envs per GPU per launch), with roofline, CPU baseline and
the end-to-end numbers through the drop-in API.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = ONE launch of the fused K1 kernel over ONE batch of `--envs` environments
(policy action pick, placement, line clears, scoring, Philox trio regeneration with the
solvability search, game over, reward, auto-reset, next mask), reading and writing the full
packed protocol (129 algorithmic bytes per env-step).  To keep every launch HBM-cold the
bench rotates over `--batches` independent env batches whose combined footprint exceeds the
126 MB L2 (stated in config.l2).  The batches are independent, so consecutive launches
alternate over `--streams` CUDA streams (default 2): launch k+1 fills the SMs that the few
long warps of launch k (trio searches) leave idle.  The timed region is one block of exactly K
launches bracketed by barrier + synchronize, right after the W warm-up launches.  Weak
scaling: every rank owns its own batches; there is no data-path collective.

--dump-outputs DIR writes what the last timed launch returned to its caller (rank 0) as float
.npy files, so that two builds can be compared output for output: every input is derived from
the fixed seed, so the same arguments give the same arrays.

CPU arm (--impl reference, and the cpu_baseline keys): the REAL reference
(VectorizedBlockBlastEnv(64, seed=42) + sample_valid_actions loop, scripts/benchmark.py:101-144;
PPOAgent collect + update, scripts/train.py:169-209) from oracle/_ref (oracle/make_ref.py) when
it travelled with the snapshot — kind "reference"; the oracle port otherwise — kind "port".
All CPU legs run on rank 0 BEFORE torch.distributed is initialised, so no GPU spins in an NCCL
barrier while they run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NCU_DRAM_BYTES_PER_LAUNCH = 18.9e6 + 0.1e6   # measured by ncu for one 262,144-env launch (see TRAFFIC_SOURCE)
TRAFFIC_SOURCE = ("ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch "
                  "(profiles/r2_kernels_ncu_summary.json, bb_step_kernel<1, 0>); reads are the 12.6 MB of state + the 6.3 MB "
                  "mask of the previous step, the 21 MB of outputs + state write-back were still in the 126 MB L2 when the "
                  "capture ended")
BOUND_NOTE = ("integer-issue bound, not HBM bound: ALU pipe 62% busy while an SM is active, 27.9 M warp instructions, "
              "21.6 of 32 lanes active per instruction (ncu); a lone launch leaves SMs idle while its longest warps drain "
              "(SMs active 76% of the launch; 95% inside a 64-step launch), which the second stream fills")
ALGO_BYTES_PER_ENV_STEP = 129          # SURVEY.md §8d / DESIGN.md: 48 R + 48 W + 4 + 4 + 1 + 24
STATE_BYTES, OUT_BYTES = 48, 33
METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"


_REAL_STDOUT = None


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled every 100 ms from before the preroll until 0.25 s
    after the timed block (the timed block alone can be shorter than one period: ~40 ms at --steps 1000)."""
    WINDOW = ("every 100 ms from before the preroll to 0.25 s after the timed block: preroll, warm-up, "
              "timed block, then idle")
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "window": self.WINDOW}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for k, nme in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": self.WINDOW}


# ----------------------------------------------------------------------------- CPU arms
def _py_port_worker(args):
    """One process: the Python oracle port of VectorizedBlockBlastEnv(64) + sample_valid_actions
    (method of the reference's scripts/benchmark.py:101-144)."""
    seed, n_envs, seconds, min_steps = args
    import numpy as np
    from oracle import bb_oracle as O
    rng = np.random.RandomState(seed)
    envs = [O.Env(seed=seed * 1000 + i, rng_factory=O.numpy_rng_factory) for i in range(n_envs)]
    vec = O.VecEnv(envs)
    vec.reset()
    for _ in range(2):
        vec.step(vec.sample_valid_actions(rng))
    t0 = time.perf_counter()
    steps = 0
    while steps < min_steps or time.perf_counter() - t0 < seconds:
        vec.step(vec.sample_valid_actions(rng))
        steps += 1
    return steps * n_envs, time.perf_counter() - t0


def cpu_python_port(n_procs, seconds, n_envs=64, min_steps=1):
    import multiprocessing as mp
    if n_procs == 1:
        res = [_py_port_worker((0, n_envs, seconds, min_steps))]
    else:
        with mp.get_context("fork").Pool(n_procs) as pool:
            res = pool.map(_py_port_worker, [(k, n_envs, seconds, min_steps) for k in range(n_procs)])
    return sum(r[0] for r in res) / max(r[1] for r in res), sum(r[0] for r in res)


def cpu_c_port(n_threads, seconds, n_envs=4096):
    """The plain-C oracle port, random-valid rollout, OpenMP over envs."""
    import numpy as np
    from bbgpu import philox
    from oracle import bb_oracle_c as OC
    chunk = 64
    streams = philox.candidate_trios(42, np.arange(n_envs), 4096)
    env = OC.CVecEnv(streams, n_threads=n_threads)
    rs = np.random.RandomState(0)
    words = rs.randint(0, 2 ** 32, size=(chunk, n_envs), dtype=np.uint64).astype(np.uint32)
    env.random_rollout(8, words)
    t0 = time.perf_counter()
    done = 0
    while time.perf_counter() - t0 < seconds:
        d, _, _ = env.random_rollout(chunk, words)
        done += d
        if env.stats()[:, 7].max() > 3500:      # candidate streams nearly used up: restart them
            env = OC.CVecEnv(streams, n_threads=n_threads)
    return done / (time.perf_counter() - t0), done


def cpu_ppo_port(seconds_hint=20.0, threads=None):
    """Fallback when oracle/_ref is absent: PPO samples/s of the reference's schedule on the host CPU
    (config 1: 64 envs x 128 steps, 10 epochs x 4 minibatches of 2048), from TIMED COMPONENTS: the Python
    oracle env step, one 64-sample CNN forward and one 2048-sample forward+backward+Adam step of the same
    5.29 M-parameter network in torch on the CPU."""
    import numpy as np
    import torch
    from bbgpu.network import BlockBlastNetwork
    from oracle import bb_oracle as O
    if threads:
        torch.set_num_threads(int(threads))
    torch.manual_seed(0)
    net = BlockBlastNetwork()
    net.train()
    opt = torch.optim.Adam(net.parameters(), lr=3e-4, eps=1e-5)
    envs = [O.Env(seed=100 + i, rng_factory=O.numpy_rng_factory) for i in range(64)]
    vec = O.VecEnv(envs)
    obs, _ = vec.reset()
    rng = np.random.RandomState(0)
    t0 = time.perf_counter()
    n_env = 0
    while time.perf_counter() - t0 < seconds_hint * 0.25:
        obs, *_ = vec.step(vec.sample_valid_actions(rng))
        n_env += 1
    t_env = (time.perf_counter() - t0) / n_env
    b, p = torch.from_numpy(obs["board"]), torch.from_numpy(obs["pieces"])
    with torch.no_grad():
        net.forward(b, p)
        t0 = time.perf_counter()
        for _ in range(3):
            net.forward(b, p)
        t_fwd = (time.perf_counter() - t0) / 3
    x = torch.rand(2048, 4, 8, 8).round()
    m = torch.ones(2048, 192)
    a = torch.zeros(2048, dtype=torch.long)
    t_upd = []
    for _ in range(2):
        t0 = time.perf_counter()
        _, lp, ent, v = net.evaluate_actions(x, m, a)
        loss = -(lp.mean()) + 0.5 * (v ** 2).mean() - 0.01 * ent.mean()
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(net.parameters(), 0.5)
        opt.step()
        t_upd.append(time.perf_counter() - t0)
    t_mb = min(t_upd)
    iteration = 128 * (t_env + t_fwd) + 40 * t_mb
    return 8192 / iteration, dict(env_vec_step_s=t_env, fwd64_s=t_fwd, minibatch2048_step_s=t_mb,
                                  iteration_s=iteration, torch_threads=torch.get_num_threads())


def cpu_legs(args):
    """Every CPU measurement of the default run (rank 0, before any GPU / NCCL work)."""
    from oracle import ref_runner
    cores = os.cpu_count() or 1
    out = {}
    secs = args.cpu_seconds
    if ref_runner.available():
        v1, tot1 = ref_runner.env_loop_all_cores(1, secs)
        out["cpu_baseline"] = {"value": v1, "unit": UNIT, "cores": 1, "kind": "reference",
                               "sample": "%d env-steps in %.0f s: the unmodified reference (oracle/_ref) VectorizedBlockBlastEnv(64, seed=42) + "
                                         "sample_valid_actions loop, serial Python as shipped (wrappers.py:93-108)" % (tot1, secs)}
        va, tota = ref_runner.env_loop_all_cores(cores, min(secs, 6.0))
        out["cpu_baseline_all_cores"] = {"value": va, "unit": UNIT, "cores": cores, "kind": "reference",
                                         "sample": "%d env-steps: the same loop in %d independent processes (one per host core)" % (tota, cores)}
    else:
        v1, tot1 = cpu_python_port(1, secs)
        out["cpu_baseline"] = {"value": v1, "unit": UNIT, "cores": 1, "kind": "port",
                               "sample": "%d env-steps: oracle/bb_oracle.py VecEnv(64) + sample_valid_actions (oracle/_ref absent: run "
                                         "oracle/make_ref.py where /root/reference is mounted)" % tot1}
    v_c, tot_c = cpu_c_port(cores, min(secs, 6.0))
    out["cpu_baseline_c_port"] = {"value": v_c, "unit": UNIT, "cores": cores, "kind": "port",
                                  "sample": "%d env-steps: oracle/bb_oracle.c random-valid rollout, 4096 envs, OpenMP over all host cores" % tot_c}
    if not args.no_ppo:
        if ref_runner.available():
            v, parts = ref_runner.ppo_iteration(1, cores)
            out["ppo_cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": parts["torch_threads"], "kind": "reference",
                                       "sample": "the unmodified reference PPOAgent (oracle/_ref) on the CPU, schedule of scripts/train.py:169-209: "
                                                 "full 128-step x 64-env collect timed, 1 of the 10 update epochs (4 x 2048) timed and scaled to 10",
                                       **parts}
        else:
            v, parts = cpu_ppo_port(secs, cores)
            out["ppo_cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": parts["torch_threads"], "kind": "port",
                                       "sample": "reference schedule (64 envs x 128 steps, 10 epochs x 4 x 2048) computed from timed components", **parts}
    return out


def kernel_rooflines(dev, peak):
    """CUDA-event timings of the companion kernels at config-3/4 sizes, inputs larger than L2;
    achieved = algorithmic bytes / time (DESIGN.md section 4)."""
    import torch
    from bbgpu import capi
    out = {}

    def timeit(fn, iters=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3 / iters

    # context for the write-dominated K2: what a pure-write stream (torch fill_) reaches on this GPU
    big = torch.empty(256 * 1024 * 1024, dtype=torch.float32, device=dev)
    t = timeit(lambda: big.fill_(1.0), iters=10)
    out["write_only_fill_GBs"] = big.numel() * 4 / t / 1e9
    del big
    # K4 GAE: T=128 x N=262,144, 20 B/sample (+4N last values) = 671 MB per launch
    T, N = 128, 262144
    r, v = torch.randn(T, N, device=dev), torch.randn(T, N, device=dev)
    d = (torch.rand(T, N, device=dev) < 0.07).float()
    lv = torch.randn(N, device=dev)
    adv, ret = torch.empty_like(r), torch.empty_like(r)
    mom = torch.zeros(2, dtype=torch.float64, device=dev)
    t = timeit(lambda: capi.gae(r, v, d, lv, 0.99, 0.95, adv, ret, mom))
    b = 20 * T * N + 4 * N
    out["K4_gae"] = {"samples": T * N, "us": t * 1e6, "algorithmic_bytes": b, "achieved_GBs": b / t / 1e9,
                     "frac_of_hbm_peak": b / t / 1e9 / peak, "samples_per_sec": T * N / t}
    del r, v, d, adv, ret
    # K3 masked sample: n=524,288 rows of f32 logits: 804 B/row = 421 MB per launch
    n = 524288
    logits = torch.randn(n, 192, device=dev)
    mask = torch.randint(-2 ** 62, 2 ** 62, (3, n), dtype=torch.int64, device=dev) | 1
    act = torch.empty(n, dtype=torch.int32, device=dev)
    lp, en = torch.empty(n, device=dev), torch.empty(n, device=dev)
    t = timeit(lambda: capi.masked_sample(logits, mask, n, 1, 1, 0, act, lp, en))
    b = 804 * n
    out["K3_masked_sample_f32"] = {"rows": n, "us": t * 1e6, "algorithmic_bytes": b, "achieved_GBs": b / t / 1e9,
                                   "frac_of_hbm_peak": b / t / 1e9 / peak}
    lb = logits.bfloat16()
    t = timeit(lambda: capi.masked_sample(lb, mask, n, 1, 1, 0, act, lp, en))
    b = 420 * n
    out["K3_masked_sample_bf16"] = {"rows": n, "us": t * 1e6, "algorithmic_bytes": b, "achieved_GBs": b / t / 1e9,
                                    "frac_of_hbm_peak": b / t / 1e9 / peak}
    # K3 backward (PPO update path): 768 B logits read + 768 B grad written + 36 B mask/action/grads per row
    gl = torch.empty_like(logits)
    g1, g2 = torch.randn(n, device=dev), torch.randn(n, device=dev)
    t = timeit(lambda: capi.masked_head_backward(logits, mask, n, act, g1, g2, gl))
    b = (768 * 2 + 36) * n
    out["K3_backward_f32"] = {"rows": n, "us": t * 1e6, "algorithmic_bytes": b, "achieved_GBs": b / t / 1e9,
                              "frac_of_hbm_peak": b / t / 1e9 / peak}
    # fused PPO loss tail (bb_ppo_loss): logits read + gradient written + 24 B mask + 7 scalars per row
    vals, gv = torch.randn(n, device=dev), torch.empty(n, device=dev)
    sums = torch.zeros(5, dtype=torch.float64, device=dev)
    t = timeit(lambda: capi.ppo_loss(logits, mask, n, act, lp, g1, g2, vals, 0.2, 0.5, 0.01, gl, gv, sums))
    b = (768 * 2 + 24 + 28) * n
    out["ppo_loss_f32"] = {"rows": n, "us": t * 1e6, "algorithmic_bytes": b, "achieved_GBs": b / t / 1e9,
                           "frac_of_hbm_peak": b / t / 1e9 / peak}
    glb = torch.empty_like(lb)
    t = timeit(lambda: capi.ppo_loss(lb, mask, n, act, lp, g1, g2, vals, 0.2, 0.5, 0.01, glb, gv, sums))
    b = (384 * 2 + 24 + 28) * n
    out["ppo_loss_bf16"] = {"rows": n, "us": t * 1e6, "algorithmic_bytes": b, "achieved_GBs": b / t / 1e9,
                            "frac_of_hbm_peak": b / t / 1e9 / peak}
    del logits, lb, gl, glb
    # K2 obs unpack: 36 B in, 1,024 B f32 planes out (+ 192 B u8 mask) per env
    board = torch.randint(-2 ** 62, 2 ** 62, (n,), dtype=torch.int64, device=dev)
    pieces = torch.randint(0, 37, (n,), dtype=torch.int32, device=dev) * 0x010101
    obs = torch.empty((n, 4, 8, 8), device=dev)
    t = timeit(lambda: capi.unpack_obs(board, pieces, mask, n, obs=obs, n=n))
    b = (12 + 1024) * n
    out["K2_unpack_obs_f32"] = {"envs": n, "us": t * 1e6, "algorithmic_bytes": b, "achieved_GBs": b / t / 1e9,
                                "frac_of_hbm_peak": b / t / 1e9 / peak}
    obs16 = torch.empty((n, 4, 8, 8), dtype=torch.bfloat16, device=dev)
    t = timeit(lambda: capi.unpack_obs(board, pieces, mask, n, obs=obs16, n=n))
    b = (12 + 512) * n
    out["K2_unpack_obs_bf16"] = {"envs": n, "us": t * 1e6, "algorithmic_bytes": b, "achieved_GBs": b / t / 1e9,
                                 "frac_of_hbm_peak": b / t / 1e9 / peak}
    for k in ("K2_unpack_obs_f32", "K2_unpack_obs_bf16"):
        out[k]["frac_of_write_only_fill"] = out[k]["achieved_GBs"] / out["write_only_fill_GBs"]
    del board, pieces, obs, obs16
    # BatchNorm + ReLU + residual add of the CNN (bf16 NHWC [rows, 128]): forward reads x twice and the
    # skip once, writes y; backward reads (x, y, dy) twice, writes dx and dskip
    rows, ch = 32768 * 64, 128
    mk = lambda: torch.randn(rows, ch, device=dev).to(torch.bfloat16)
    x, skip, y, dy, dx, dsk = mk(), mk(), mk(), mk(), mk(), mk()
    gamma, beta = torch.rand(ch, device=dev) + 0.5, torch.randn(ch, device=dev)
    rm, rv = torch.zeros(ch, device=dev), torch.ones(ch, device=dev)
    sm, sr = torch.empty(ch, device=dev), torch.empty(ch, device=dev)
    dg, db = torch.empty(ch, device=dev), torch.empty(ch, device=dev)
    ws = torch.empty(capi.bn_workspace_size(ch), device=dev)
    t = timeit(lambda: capi.bn_relu_forward(x, skip, gamma, beta, None, rm, rv, 0.1, 1e-5, True, y, sm, sr, ws, rows, ch))
    b = 4 * rows * ch * 2
    out["BN_relu_residual_forward_bf16"] = {"rows": rows, "channels": ch, "us": t * 1e6, "algorithmic_bytes": b,
                                            "achieved_GBs": b / t / 1e9, "frac_of_hbm_peak": b / t / 1e9 / peak}
    t = timeit(lambda: capi.bn_relu_backward(x, y, dy, gamma, sm, sr, dx, dsk, dg, db, ws, rows, ch))
    b = 8 * rows * ch * 2
    out["BN_relu_residual_backward_bf16"] = {"rows": rows, "channels": ch, "us": t * 1e6, "algorithmic_bytes": b,
                                             "achieved_GBs": b / t / 1e9, "frac_of_hbm_peak": b / t / 1e9 / peak}
    # layers without a residual input: the ReLU mask is recomputed from x, y is not read (x, dy twice; dx written)
    t = timeit(lambda: capi.bn_relu_backward_no_skip(x, dy, gamma, beta, sm, sr, dx, dg, db, ws, rows, ch))
    b = 5 * rows * ch * 2
    out["BN_relu_backward_no_skip_bf16"] = {"rows": rows, "channels": ch, "us": t * 1e6, "algorithmic_bytes": b,
                                            "achieved_GBs": b / t / 1e9, "frac_of_hbm_peak": b / t / 1e9 / peak}
    return out


FWD_FLOP_PER_SAMPLE = 113.05e6          # BlockBlastNetwork forward (BASELINE.md section 3)


def _mfu(samples_per_sec_per_gpu, epochs):
    """Model FLOP utilisation of the CNN work per collected sample: 1 forward in the collect + epochs x
    (forward + backward = 3 forwards) in the update, against the measured sustained bf16 matmul rate."""
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"]) * 1e12
        src = "MEASURED_PEAKS.json bf16_tflops_sustained"
    except Exception:
        peak, src = 1377.7e12, "fallback 1377.7 TF/s"
    flop = FWD_FLOP_PER_SAMPLE * (1 + 3 * epochs)
    return {"flop_per_collected_sample": flop, "achieved_tflops_per_gpu": samples_per_sec_per_gpu * flop / 1e12,
            "mfu": samples_per_sec_per_gpu * flop / peak, "peak_source": src}


def gpu_ppo_leg(rank, world, dev, n_envs, T, minibatch, epochs, precision, use_graph, iters, warm):
    """Masked-PPO collect + GAE + update on the device-resident path; returns samples/s and the phase
    times of the median timed iteration.  ``warm`` untimed iterations first (cuDNN autotuning, allocator
    growth, CUDA-graph capture when ``use_graph``)."""
    import torch
    import torch.distributed as dist
    from bbgpu.ppo import PPOAgent, PPOConfig
    from bbgpu.rollout import RolloutBuffer
    from bbgpu.train import RolloutRunner
    from bbgpu.vec_env import VectorizedBlockBlastEnv
    offset = (64 + rank) * n_envs
    agent = PPOAgent(PPOConfig(batch_size=minibatch, num_epochs=epochs, precision=precision), dev, seed=42,
                     global_env_offset=offset)
    agent.train()
    venv = VectorizedBlockBlastEnv(n_envs, seed=42, output="packed", global_env_offset=offset)
    buf = RolloutBuffer(T, n_envs, device=dev)
    runner = RolloutRunner(venv, agent, buf, use_graph=use_graph)
    rows = []
    for it in range(warm + iters):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        last = runner.run()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        metrics = agent.update(buf, last, use_graph=use_graph)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t2 = time.perf_counter()
        if it >= warm:
            rows.append((t2 - t0, t1 - t0, t2 - t1))
    rows.sort()
    tot, col, upd = rows[len(rows) // 2]
    tt = torch.tensor([tot], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    venv.close()
    sps = world * n_envs * T / float(tt.item())
    return dict(samples_per_sec=sps, envs_per_gpu=n_envs, rollout_steps=T, minibatch_per_gpu=minibatch, epochs=epochs,
                precision=precision, cuda_graph=bool(use_graph), iterations_timed=iters, collect_s=col, update_s=upd,
                total_s=tot, total_s_min=rows[0][0], total_s_max=rows[-1][0], entropy=metrics["entropy"],
                approx_kl=metrics["approx_kl"], **_mfu(sps / world, epochs),
                grad_allreduce="1 flat NCCL all-reduce of 21.2 MB per optimiser step" if world > 1 else "n/a (1 GPU)")


def run_reference_arm(args, rank, world):
    """bench.py --impl reference: the reference's own CPU implementation of the path on all host cores."""
    if rank != 0:
        return
    from oracle import ref_runner
    cores = os.cpu_count() or 1
    n_envs = 64
    per_step_s = 0.06                      # ~64 envs x ~1 ms per Python env-step
    budget = min(150.0, max(5.0, (args.steps + args.warmup) * per_step_s))
    t0 = time.perf_counter()
    if ref_runner.available():
        value, total = ref_runner.env_loop_all_cores(cores, budget, n_envs=n_envs, min_steps=max(1, min(args.steps, 50)))
        kind, what = "reference", "the unmodified reference (oracle/_ref): VectorizedBlockBlastEnv(64, seed=42+1000k) + sample_valid_actions loop"
    else:
        value, total = cpu_python_port(cores, budget, n_envs=n_envs, min_steps=max(1, min(args.steps, 50)))
        kind, what = "port", "oracle/bb_oracle.py (Python restatement of the reference's cell-grid engine; oracle/_ref absent)"
    wall = time.perf_counter() - t0
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n_envs * cores / value,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": {"workload": "random valid-action policy, VectorizedBlockBlastEnv(64) per process, "
                                   "%d processes (one per host core)" % cores,
                       "step": "one 64-env vec step per process (bounded sample of config 3)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": "%d env-steps in %.1f s: %s x %d processes" % (total, wall, what, cores)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def _median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def _spread(xs, per):
    xs = sorted(xs)
    q = lambda f: xs[min(len(xs) - 1, int(f * len(xs)))]
    return {"blocks": len(xs), "median": _median(xs) / per, "min": xs[0] / per, "p10": q(0.1) / per, "p90": q(0.9) / per,
            "max": xs[-1] / per}


DUMP_MAX_ROWS = 65536          # 788 B per dumped env: at most 52 MB in all


def dump_step_outputs(out_dir, o, env_offset, seed):
    """Write one bb_env_step_random launch's results as its caller receives them, for at most
    DUMP_MAX_ROWS envs of the batch (a fixed seeded sample of a larger one): env_id (global env id),
    actions, rewards, terminated, and action_mask [rows, 192] (action = piece slot * 64 + cell)."""
    import numpy as np
    n = o["actions"].numel()
    rows = np.arange(n) if n <= DUMP_MAX_ROWS else np.sort(np.random.default_rng(seed).choice(n, DUMP_MAX_ROWS, replace=False))
    mask = np.ascontiguousarray(o["mask"].cpu().numpy()[:, rows])
    dense = np.unpackbits(mask.view(np.uint8).reshape(3, len(rows), 8), axis=2, bitorder="little")
    arrays = {"env_id": (env_offset + rows).astype(np.float64),
              "actions": o["actions"].cpu().numpy()[rows].astype(np.float32),
              "rewards": o["rewards"].cpu().numpy()[rows],
              "terminated": o["term"].cpu().numpy()[rows].astype(np.float32),
              "action_mask": dense.transpose(1, 0, 2).reshape(len(rows), 192).astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=262144, help="envs per batch (= per launch) per GPU")
    ap.add_argument("--batches", type=int, default=8, help="independent env batches rotated per GPU (L2-cold launches)")
    ap.add_argument("--streams", type=int, default=2, help="CUDA streams the independent batches alternate over")
    ap.add_argument("--preroll", type=int, default=64, help="untimed random steps to reach the steady-state mix")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed launch's outputs (rank 0) to DIR/<name>.npy (bench_outputs/ is git-ignored)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps per e2e block; 0 = min(steps, 100)")
    ap.add_argument("--e2e-min-seconds", type=float, default=2.0)
    ap.add_argument("--cpu-seconds", type=float, default=8.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ppo", action="store_true")
    ap.add_argument("--no-kernels", action="store_true")
    ap.add_argument("--ppo-envs", type=int, default=131072, help="envs per GPU for the config-4 PPO leg (1,048,576 / 8)")
    ap.add_argument("--ppo-steps", type=int, default=8)
    ap.add_argument("--ppo-minibatch", type=int, default=32768)
    ap.add_argument("--ppo-epochs", type=int, default=10, help="the reference's PPOConfig.num_epochs (ppo.py:34)")
    ap.add_argument("--ppo-precision", default="bf16", choices=["bf16", "fp32"])
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    # stdout must carry exactly ONE JSON line: libraries (NCCL prints its version banner there)
    # get stderr; the line is written to the saved descriptor at the end
    sys.stdout.flush()
    global _REAL_STDOUT
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    # CPU legs first, on rank 0, before CUDA / NCCL exist in this process: the other ranks wait in the
    # TCP-store rendezvous of init_process_group (a host-side wait, no GPU busy-spin)
    cpu = cpu_legs(args) if (rank == 0 and not args.no_cpu) else {}

    import numpy as np
    import torch
    import torch.distributed as dist
    from bbgpu import capi
    from bbgpu.vec_env import VectorizedBlockBlastEnv

    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    binding = None
    if world > 1:
        # host side of the e2e path: keep each rank's Python thread, copy completions and pinned buffers on the
        # cores / memory of its GPU's NUMA node
        from bbgpu.dist import pin_to_gpu_numa
        binding = pin_to_gpu_numa(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(minutes=20))
    L = capi.lib()

    n, M, K, W, S = args.envs, args.batches, args.steps, max(3, args.warmup), max(1, args.streams)
    assert M % S == 0, "--batches must be a multiple of --streams (a batch always runs on the same stream)"
    seed = 42
    # independent batches; global env ids are disjoint across batches and ranks
    envs, outs = [], []
    for b in range(M):
        envs.append(capi.EnvHandle(n, seed, global_env_offset=(rank * M + b) * n))
        outs.append(dict(actions=torch.zeros(n, dtype=torch.int32, device=dev),
                         rewards=torch.zeros(n, dtype=torch.float32, device=dev),
                         term=torch.zeros(n, dtype=torch.uint8, device=dev),
                         mask=torch.zeros((3, n), dtype=torch.int64, device=dev)))
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    # the sampler's start-up wait comes before the preroll, so the GPU does not idle between the
    # preroll, the warm-up and the timed block
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    for e, o in zip(envs, outs):
        e.step_random(args.preroll, None, None, None, o["mask"])          # desynchronise episodes (all envs start in lockstep)
    torch.cuda.synchronize()

    main_stream = torch.cuda.current_stream()
    streams = [torch.cuda.Stream() for _ in range(S)]
    sptr = [s.cuda_stream for s in streams]
    largs = [(e.h, 1, o["actions"].data_ptr(), o["rewards"].data_ptr(), o["term"].data_ptr(), o["mask"].data_ptr(),
              stats.data_ptr(), o["mask"].data_ptr()) for e, o in zip(envs, outs)]
    step_random = L.bb_env_step_random

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ends = [torch.cuda.Event() for _ in range(S)]

    def block(k0, count, ptrs):
        """`count` launches alternating over the streams in `ptrs`; device time of the whole block in ms."""
        ns = len(ptrs)
        barrier()
        ev0.record(main_stream)
        for s in streams[:ns]:
            s.wait_event(ev0)
        for k in range(k0, k0 + count):
            rc = step_random(*largs[k % M], ptrs[k % ns])       # the policy reads the mask the previous step wrote (mask_in)
            if rc:
                raise capi.BBGpuError(capi.last_error())
        for s, e in zip(streams[:ns], ends):
            e.record(s)
            main_stream.wait_event(e)
        ev1.record(main_stream)
        barrier()
        return ev0.elapsed_time(ev1)

    block(0, W, sptr)                                         # warm-up, directly before the timed block
    stats.zero_()

    def agree(count):
        """the same block count on every rank (each block contains barriers): max over ranks"""
        t = torch.tensor([int(count)], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return int(t.item())

    t_wall0 = time.perf_counter()
    ms = block(W, K, sptr)                                    # the timed steps: exactly K launches
    wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    s = stats.cpu().tolist()
    assert s[0] == n * K, "kernel did not process the expected number of env-steps"
    if args.dump_outputs and rank == 0:
        last = (W + K - 1) % M
        dump_step_outputs(args.dump_outputs, outs[last], (rank * M + last) * n, seed)
    tms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_max = float(tms.item())
    value = world * n * K / (ms_max * 1e-3)

    # K-launch blocks serialised on ONE stream (launch k+1 waits for the last warp of launch k), beside
    # the value: median of 5..100 blocks, about 0.5 s of device time (ms_max is the same on every rank)
    ms_single = _median([block(W + K * (i + 1), K, sptr[:1]) for i in range(max(5, min(100, int(500.0 / ms_max) + 1)))])

    # L2-warm variant (single batch, state+outputs 21 MB stay in L2): reported beside, not as value
    o0 = outs[0]
    for k in range(20):
        envs[0].step_random(1, o0["actions"], o0["rewards"], o0["term"], o0["mask"], stats)
    barrier()
    ev0.record()
    kw = 1000
    for k in range(kw):
        envs[0].step_random(1, o0["actions"], o0["rewards"], o0["term"], o0["mask"], stats)
    ev1.record()
    barrier()
    ms_warm = ev0.elapsed_time(ev1)

    # fused rollout: ONE launch runs 256 steps with the env state in registers
    ev0.record()
    envs[0].step_random(256, None, None, None, None, stats)
    ev1.record()
    barrier()
    ms_fused = ev0.elapsed_time(ev1)

    # rollout kernel: one launch = 16 steps, EVERY step's actions/rewards/terminated/masks written ([16, N] arrays)
    R = 16
    RA = torch.zeros((R, n), dtype=torch.int32, device=dev); RR = torch.zeros((R, n), dtype=torch.float32, device=dev)
    RT = torch.zeros((R, n), dtype=torch.uint8, device=dev); RM = torch.zeros((R, 3, n), dtype=torch.int64, device=dev)
    for b in range(2):
        envs[b].rollout_random(R, RA, RR, RT, RM, stats)
    barrier()
    ev0.record()
    for k in range(32):
        envs[k % M].rollout_random(R, RA, RR, RT, RM, stats)
    ev1.record()
    barrier()
    ms_roll = ev0.elapsed_time(ev1)
    del RA, RR, RT, RM
    for e in envs:
        e.close()
    del outs, largs
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ e2e through the drop-in API
    Ke = args.e2e_steps or min(K, 100)

    def e2e_leg(obs_format, min_seconds, touch):
        venv = VectorizedBlockBlastEnv(n, seed=seed, output="numpy", global_env_offset=(world * M + rank) * n,
                                       reuse_buffers=True, obs_format=obs_format)
        venv.reset()
        for _ in range(3):
            venv.step(venv.sample_valid_actions())
        blocks, n_term, n_blocks = [], 0, 3
        while len(blocks) < n_blocks:
            if len(blocks) == 3:
                n_blocks = agree(min(500, max(3, int(min_seconds / _median(blocks)) + 1)))
                if n_blocks == 3:
                    break
            barrier()
            t0 = time.perf_counter()
            for _ in range(Ke):
                a = venv.sample_valid_actions()                    # kernel + D2H 4 B/env (numpy actions, as the reference)
                obs, rew, term, trunc, infos = venv.step(a)        # H2D 4 B/env, K1 (+ K2 for dense), one D2H of the result block
                n_term += int(np.count_nonzero(term))              # the caller reads the result
                if touch:
                    touch(obs)
            barrier()
            blocks.append(time.perf_counter() - t0)
        venv.close()
        med = torch.tensor([_median(blocks)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(med, op=dist.ReduceOp.MAX)
        return world * n * Ke / float(med.item()), _spread(blocks, Ke * 1e-3)

    e2e_value, e2e_spread = e2e_leg("lazy", args.e2e_min_seconds, None)
    # reference-layout observation delivered every step: board (N,8,8) f32, pieces (N,3,8,8) f32, action_mask
    # (N,192) int8 expanded on the DEVICE (K2) and copied in one 1,221 B/env transfer; the caller looks at them
    e2e_dense, dense_spread = e2e_leg("dense", min(args.e2e_min_seconds, 1.5),
                                      lambda obs: (obs["board"][::4096, 0, 0].sum(), obs["pieces"][::4096, 0, 0, 0].sum(),
                                                   obs["action_mask"][::4096, 0].sum()))
    h2d = 4 * n
    d2h = 4 * n + 41 * n
    torch.cuda.empty_cache()

    kernels = kernel_rooflines(dev, load_peaks()[0]) if (rank == 0 and not args.no_kernels) else None
    torch.cuda.empty_cache()
    ppo = ppo_ref = None
    if not args.no_ppo:
        # (a) BASELINE config 4 shape: 131,072 envs per GPU (1,048,576 over 8), the reference's 10 epochs
        ppo = gpu_ppo_leg(rank, world, dev, args.ppo_envs, args.ppo_steps, args.ppo_minibatch, args.ppo_epochs,
                          args.ppo_precision, False, 1, 2)
        torch.cuda.empty_cache()
        # (b) the reference's OWN schedule per GPU (config/default.yaml as scripts/train.py reads it: 64 envs x
        #     128 steps, minibatch 2048, 10 epochs), CUDA-graph replayed — like-for-like with ppo_cpu_baseline
        ppo_ref = gpu_ppo_leg(rank, world, dev, 64, 128, 2048, 10, args.ppo_precision, True, 9, 3)
        torch.cuda.empty_cache()

    if rank == 0:
        peak, peak_src = load_peaks()
        per_launch_s = ms_max * 1e-3 / K
        achieved = ALGO_BYTES_PER_ENV_STEP * n / per_launch_s / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": {"workload": "random valid-action policy, %d envs per GPU per launch (BASELINE config 3)" % n,
                       "envs_per_gpu_per_launch": n, "batches_rotated": M, "streams": S, "seed": seed,
                       "l2": "rotating %d independent env batches per GPU: %.0f MB of state+outputs > 126 MB L2, "
                             "every launch reads its state from HBM" % (M, M * n * (STATE_BYTES + OUT_BYTES) / 1e6),
                       "protocol": "packed: state 48 B R+W, action 4 B, reward 4 B, terminated 1 B, mask 24 B R+W",
                       "parallelism": "env shards per GPU, no data-path collective; launches of independent batches "
                                      "alternate over %d streams" % S},
            "timing": {"block_steps": K, "what": "device ms per step of the one timed block of K launches "
                       "(barrier + synchronize on both sides)", **_spread([ms], K),
                       "timed_device_s": ms * 1e-3, "launches_timed": K},
            "gpu_launches": K,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": NCU_DRAM_BYTES_PER_LAUNCH,
                         "traffic_source": TRAFFIC_SOURCE,
                         "bound_note": BOUND_NOTE,
                         "kernel": "bb_step_kernel<true,false>",
                         "algorithmic_bytes_per_launch": ALGO_BYTES_PER_ENV_STEP * n, "peak_source": peak_src,
                         "launch_us": per_launch_s * 1e6,
                         "launch_us_is": "block time / K with launches of independent batches overlapping on %d streams" % S,
                         "launch_us_single_stream": ms_single / K * 1e3,
                         "frac_single_stream": ALGO_BYTES_PER_ENV_STEP * n / (ms_single * 1e-3 / K) / 1e9 / peak},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps_per_block": Ke, "timing_ms_per_step": e2e_spread,
                    "observation": "PACKED / LAZY: the step returns board u64, pieces u32 and 3 x u64 mask words per env (41 B/env with "
                                   "reward and done flag); the reference-layout float arrays are only built if the caller indexes obs[...]",
                    "api": "VectorizedBlockBlastEnv(output='numpy', obs_format='lazy', reuse_buffers=True): sample_valid_actions() + "
                           "step(actions); numpy results are zero-copy views of double-buffered pinned memory",
                    "dense": {"value": e2e_dense, "unit": UNIT, "h2d_bytes_per_step": 4 * n, "d2h_bytes_per_step": 4 * n + 1221 * n,
                              "timing_ms_per_step": dense_spread,
                              "observation": "DENSE reference layout delivered every step (wrappers.py:118-126): board (N,8,8) f32, pieces "
                                             "(N,3,8,8) f32, action_mask (N,192) int8, expanded on the device by K2 and copied in one block",
                              "api": "VectorizedBlockBlastEnv(output='numpy', obs_format='dense', reuse_buffers=True)"}},
            "clocks": clocks,
            "host_binding_rank0": binding,
            "extra": {"single_stream_env_steps_per_sec": n * K / (ms_single * 1e-3),
                      "l2_warm_single_batch_env_steps_per_sec": n * kw / (ms_warm * 1e-3),
                      "fused_256_step_launch_env_steps_per_sec": n * 256 / (ms_fused * 1e-3),
                      "rollout16_all_outputs_env_steps_per_sec": n * 16 * 32 / (ms_roll * 1e-3),
                      "episodes": s[1], "mean_episode_len": (s[3] / s[1]) if s[1] else None,
                      "mean_final_score": (s[2] / s[1]) if s[1] else None, "wall_s_timed_region": wall},
        }
        line["kernels"] = kernels
        if ppo is not None:
            line["ppo"] = ppo
            line["ppo_reference_schedule"] = ppo_ref
        for k in ("cpu_baseline", "cpu_baseline_all_cores", "cpu_baseline_c_port"):
            if k in cpu:
                line[k] = cpu[k]
        if ppo is not None and "ppo_cpu_baseline" in cpu:
            cb = cpu["ppo_cpu_baseline"]
            line["ppo_reference_schedule"]["cpu_baseline"] = cb
            line["ppo_reference_schedule"]["ratio_per_gpu_vs_cpu_box"] = ppo_ref["samples_per_sec"] / world / cb["value"]
            line["ppo"]["cpu_baseline"] = cb
            line["ppo"]["ratio_per_gpu_vs_cpu_box"] = ppo["samples_per_sec"] / world / cb["value"]
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
