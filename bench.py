#!/usr/bin/env python
"""bench.py -- env-steps/sec of the widowGo1 hot path (BASELINE.json metric).

One "step" = one PPO iteration over one batch of synthetic sim-state tensors:
  T=40 x [ policy act -> (synthetic physics stand-in) -> fused post-physics step -> reward store ]
  -> critic bootstrap + GAE -> update() (5 epochs x 4 mini-batches of M = N*T/4 rows).
`value` = world * N * T / iteration time, inputs already resident in HBM.
`e2e`   = the same through the public API with HOST sim-state buffers: every env step copies that
          step's six Isaac-Gym-layout tensors from pinned host memory and reads rewards/dones back.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our arm (configs[1]: flat terrain, 4096 envs/GPU)
    python bench.py --config rough | roa                             # configs[2] (height scan + terrain curriculum) / configs[3] (ROA, 8192 envs)
    python bench.py --impl reference [--gpus N] --steps K --warmup W   # the reference path on host cores, same config
    python bench.py --steps K --warmup W --dump-outputs DIR          # + what the last timed step computed, as DIR/*.npy

The headline runs the error-compensated tensor-core path (`--precision tf32x3`: fp32-grade, passes the fp32 parity assertions of
tests/test_gpu_ppo.py); the line also carries the plain-TF32 numbers (`tf32`) and, report-only, the reference's own rsl_rl as eager
PyTorch on the same GPU (`reference_eager_b200`).

Multi-GPU: launched by torch.distributed.run, one rank per GPU, 4096 envs per rank (weak scaling);
one NCCL all-reduce of the flat gradient per PPO mini-batch + one of the advantage statistics.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

N_ENVS, T_STEPS = 4096, 40
K1_BYTES_PER_ENV = 10653            # SURVEY.md section 8d, reference buffer semantics
K1_BYTES_HEIGHT_SCAN = 1870         # config 3: + 187 x (3 x int16 gather + fp32 write) per env-step (SURVEY 8d)
CONFIGS = {
    "flat": dict(envs=4096, params="flat", label="widowGo1 flat terrain, 4096 envs/GPU (BASELINE.json configs[1])"),
    "rough": dict(envs=4096, params="rough", label="widowGo1 rough terrain: 187-point height scan on the 10000x600 int16 field + terrain "
                                                   "curriculum, 4096 envs/GPU (BASELINE.json configs[2])"),
    "roa": dict(envs=8192, params="flat", label="widowGo1 Regularized Online Adaptation: teacher update() + student update_dagger(), "
                                               "8192 envs/GPU (BASELINE.json configs[3])"),
}
DTYPE = {"fp32": "f32", "tf32": "tf32", "tf32x3": "tf32x3 (three TF32 tensor-core products per GEMM, fp32 accumulate: fp32-grade)"}
MLP_PATH = {"fp32": "fp32 CUDA-core tile GEMM", "tf32": "TF32 tcgen05 fused layer chains (fp32 accumulate in TMEM)",
            "tf32x3": "3xTF32 tcgen05 fused layer chains (hi/lo operand split, low parts in TMEM, fp32 accumulate)"}
HP = dict(value_loss_coef=1.0, use_clipped_value_loss=True, clip_param=0.2, entropy_coef=0.0, num_learning_epochs=5,
          num_mini_batches=4, learning_rate=2e-4, gamma=0.99, lam=0.95, max_grad_norm=1.0,
          min_policy_std=[[0.15, 0.25, 0.25] * 4 + [0.2] * 3 + [0.05] * 3], mixing_schedule=[1.0, 0, 1],
          priv_reg_coef_schedual=[0, 1, 1000, 1000])
INIT_STD = [[0.8, 1.0, 1.0] * 4 + [1.0] * 6]


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return dict(hbm_gbs=6650.0, bf16_tflops=1590.0), "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (profiling recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.02)

    def finish(self):
        self._halt.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(self.rows))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Workload:
    def __init__(self, device, rank, config="flat", T=T_STEPS, world=1, group=None, host_inputs=False, precision="tf32x3"):
        import envstate as E
        from dwbc_b200 import synth
        from dwbc_b200.actor_critic import FlatActorCritic
        from dwbc_b200.env import FusedWidowGo1Core
        from dwbc_b200.ppo import FusedPPO
        cfg = CONFIGS[config]
        n_envs = cfg["envs"]
        self.device, self.N, self.T, self.world, self.config = device, n_envs, T, world, config
        p = E.make_params(cfg["params"], n_envs)
        st = synth.initial_env_state(p, 100 + rank)
        st.update(synth.sim_state(p, 100 + rank, 0, rp_sigma=0.05, z_lo=0.327))
        if p.measure_heights:
            st["height_samples"] = synth.height_field(p, 100 + rank)
            # sub-terrain platforms laid out INSIDE the 1000 m x 60 m field (WG:253) so that the scans of different envs touch
            # different parts of the 12 MB table: levels along x (90 m apart), types along y (2.9 m apart)
            tl, tc = p.max_terrain_level, p.terrain_num_cols
            org = np.zeros((tl, tc, 3), np.float32)
            org[:, :, 0] = (np.arange(tl, dtype=np.float32)[:, None] + 0.5) * np.float32(p.tot_rows * p.horizontal_scale / tl) - np.float32(p.border_size)
            org[:, :, 1] = (np.arange(tc, dtype=np.float32)[None, :] + 0.5) * np.float32(p.tot_cols * p.horizontal_scale / tc) - np.float32(p.border_size)
            st["terrain_origins"] = org
            st["env_origins"] = org[st["terrain_levels"], st["terrain_types"]]
        self.p = p
        self.env = FusedWidowGo1Core(p, device, state=st, seed=1000 + rank, sync_stats=False)
        self.env.update_command_curriculum()
        ac = FlatActorCritic(device=device, seed=0, init_std=INIT_STD, num_priv=24, num_hist=10, num_prop=76)  # same params on all ranks
        self.alg = FusedPPO(ac, device=device, world_size=world, process_group=group, precision=precision, **HP)
        self.alg.init_storage(n_envs, T, [p.num_obs], [None], [p.num_actions])
        self.alg.counter = 1500           # priv-reg coef 0.5, mixing ratio 1.0: every loss branch active
        self.alg.generator = torch.Generator(device=device)
        self.alg.generator.manual_seed(7 + rank)
        # ---- synthetic physics stand-in: T distinct sim states (366 MB > L2), regenerated on device ----
        g = torch.Generator(device=device)
        g.manual_seed(31 + rank)
        base = {k: torch.from_numpy(v).to(device) for k, v in synth.sim_state(p, 100 + rank, 1, rp_sigma=0.05, z_lo=0.327).items()}
        if p.terrain_curriculum:          # robots stand near their (current) platform, +-5 m (the kernel moves platforms on resets; the pool is static)
            base["root_states"][:, 0, 0:2] += self.env.env_origins[:, 0:2]
        self.pool = []
        for t in range(T):
            s = {}
            for k in ("root_states", "dof_state", "rigid_body_state", "contact_forces", "force_sensor", "torques"):
                noise = torch.randn(base[k].shape, device=device, generator=g) * 0.02
                s[k] = (base[k] + noise * base[k].abs().clamp(min=0.05)).contiguous()
            q = s["root_states"][:, 0, 3:7]
            s["root_states"][:, 0, 3:7] = q / q.norm(dim=-1, keepdim=True)
            self.pool.append(s)
        self.sim_bytes = sum(v.numel() * 4 for v in self.pool[0].values())
        self.host_inputs = host_inputs
        if host_inputs:
            self.host_pool = [{k: v.cpu().pin_memory() for k, v in s.items()} for s in self.pool]
            # two device-side input sets: the copy engine fills one (copy stream) while the kernels of the previous env step read the other
            self.dev_in = [{k: torch.empty_like(v) for k, v in self.pool[0].items()} for _ in range(2)]
            self.copy_stream = torch.cuda.Stream(device=device)
            self.env.bind_sim(**self.dev_in[0])
            self.host_out = torch.empty(n_envs, 3, dtype=torch.float32).pin_memory()
            self.dev_out = torch.empty(n_envs, 3, device=device)
        self.k1_events = []
        self.env.set_obs_target(self.alg.storage.obs_row(0))
        self.obs = self.alg.storage.obs_row(0)
        self.last = None

    def rollout(self, time_k1=False, hist_encoding=False):
        env, alg, T = self.env, self.alg, self.T
        obs = self.obs
        if obs.data_ptr() != alg.storage.obs_row(0).data_ptr():
            alg.storage.obs_row(0).copy_(obs)            # carry obs_T of the previous iteration into row 0
            obs = alg.storage.obs_row(0)
        if self.host_inputs:
            main = torch.cuda.current_stream()
            copied = [torch.cuda.Event() for _ in range(T)]
            consumed = [torch.cuda.Event() for _ in range(T)]

            def h2d(t):                                   # this step's simulator state: pinned host -> device set t & 1, on the copy stream
                with torch.cuda.stream(self.copy_stream):
                    if t >= 2:
                        self.copy_stream.wait_event(consumed[t - 2])      # the kernels of step t-2 have finished reading this set
                    else:
                        self.copy_stream.wait_stream(main)                # (first two steps: everything issued before this iteration)
                    for k, dst in self.dev_in[t & 1].items():
                        dst.copy_(self.host_pool[t][k], non_blocking=True)
                    copied[t].record(self.copy_stream)
            h2d(0)
        for t in range(T):
            if self.host_inputs and t + 1 < T:
                h2d(t + 1)                                # overlaps the policy inference and the post-physics kernel of step t
            actions = alg.act(obs, obs, hist_encoding)
            # --- physics stand-in: Isaac Gym would simulate and refresh these tensors in place ---
            if self.host_inputs:
                main.wait_event(copied[t])
                env.bind_sim(**self.dev_in[t & 1])
            else:
                env.bind_sim(**self.pool[t])
            env.set_obs_target(alg.storage.obs_row(t + 1))
            st_ = alg.storage          # rewards / dones of this transition go straight into the storage rows (SURVEY f2)
            env.set_transition_target(st_.values[t], st_.rewards[t], st_.dones[t], alg.gamma)
            env.pre_physics_step(actions)
            if time_k1:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                env.post_physics_step()
                e1.record()
                self.k1_events.append((e0, e1))
            else:
                env.post_physics_step()
            obs = env.obs_buf
            if self.host_inputs:
                consumed[t].record(main)
            alg.process_env_step(env.rew_buf, env.arm_rew_buf, env.reset_buf, env.extras)
            if self.host_inputs:                      # the step's result goes back to the host
                self.dev_out[:, 0], self.dev_out[:, 1], self.dev_out[:, 2] = env.rew_buf, env.arm_rew_buf, env.reset_buf.float()
                self.host_out.copy_(self.dev_out, non_blocking=True)
        return obs

    def iteration(self, time_k1=False):
        obs = self.rollout(time_k1)
        self.alg.compute_returns(obs)
        self.last = self.alg.update()
        self.obs = obs

    def dagger_iteration(self):
        """Every `dagger_update_freq`-th iteration of ROA (OPR:125-169): student rollout (history-encoder latent) + update_dagger()."""
        obs = self.rollout(hist_encoding=True)
        self.alg.compute_returns(obs)
        self.last = self.alg.update_dagger()
        self.obs = obs


DUMP_LIMIT_BYTES = 64 * 2**20
DUMP_ENVS = 4096            # per-env arrays of a larger run (roa: 8192 envs) are a fixed, seeded sample of this many envs
DUMP_OBS_ROWS = 2048        # rollout observations [T, N, 860] (563 MB at 4096 envs): a fixed, seeded sample of (t, env) rows


def dump_outputs(w, out_dir):
    """Writes what the last timed iteration handed its caller as out_dir/<name>.npy: update()'s losses, the parameters after the
    update, the rollout storage it trained on and the last observation.  The samples are drawn from a fixed seed, so two runs
    with the same arguments write the same rows.  The weight gradients are summed with float atomics in no fixed order, so the
    parameters, and everything computed from them in later iterations, agree between two runs to rounding, not bit for bit."""
    s, N, T = w.alg.storage, w.N, w.T
    g = torch.Generator().manual_seed(0)
    envs = torch.arange(N) if N <= DUMP_ENVS else torch.randperm(N, generator=g)[:DUMP_ENVS].sort().values
    rows = torch.randperm(T * N, generator=g)[:DUMP_OBS_ROWS].sort().values
    envs, rows = envs.to(w.device), rows.to(w.device)
    out = {"update_losses": torch.tensor(w.last, dtype=torch.float64),
           "params": torch.cat([v.reshape(-1) for v in w.alg.actor_critic.state_dict().values()]),
           "last_obs": w.obs[envs],
           "observations_sample": s.observations.reshape(T * N, -1)[rows]}
    for k in ("actions", "actions_log_prob", "values", "rewards", "dones", "returns", "advantages"):
        out[k] = getattr(s, k)[:, envs]
    out = {k: (v.cpu().numpy() if v.dtype == torch.float64 else v.float().cpu().numpy()) for k, v in out.items()}
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_LIMIT_BYTES, f"--dump-outputs would write {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def cuda_ms(fn, reps, barrier, device, world):
    """fn() `reps` times between CUDA events, max over ranks."""
    import torch.distributed as dist
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1) / reps], device=device)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms)


def run_ours(args):
    import torch.distributed as dist
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback on the product path)"
    torch.cuda.set_device(local)
    device = f"cuda:{local}"
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(device))
    from dwbc_b200 import _lib as L
    from dwbc_b200 import shard
    lib = L.lib()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- multi-GPU numerics where the driver sees them: the sharded update against the union batch (SURVEY 8e) ----
    dist_parity = None
    if world > 1:
        from dwbc_b200.actor_critic import FlatActorCritic
        from dwbc_b200.ppo import FusedPPO

        def make_alg(n, w, g):
            ac = FlatActorCritic(device=device, seed=0, init_std=INIT_STD, num_priv=24, num_hist=10, num_prop=76)
            alg = FusedPPO(ac, device=device, world_size=w, process_group=g, precision=args.precision, **dict(HP, num_learning_epochs=2, num_mini_batches=2))
            alg.init_storage(n, 8, [860], [None], [18])
            alg.counter = 1500
            return alg
        dist_parity = shard.union_batch_parity(make_alg, rank, world, device, 64, 8, 2)
        barrier()

    def timed(w, steps, time_k1=False):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.dwbc_launch_count()
        e0.record()
        for _ in range(steps):
            w.iteration(time_k1)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), lib.dwbc_launch_count() - l0

    w = Workload(device, rank, config=args.config, world=world, group=group, precision=args.precision)
    for _ in range(max(args.warmup, 3)):
        w.iteration()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches = timed(w, args.steps, time_k1=True)
    clocks = sampler.finish() if sampler else None
    if args.dump_outputs and rank == 0:       # before the measurements below move the workload on
        dump_outputs(w, args.dump_outputs)
    k1_ms = float(np.mean([a.elapsed_time(b) for a, b in w.k1_events])) if w.k1_events else None
    value = world * w.N * w.T * args.steps / (ms / 1e3)

    # ---- K1 alone, back to back: the per-step host work exceeds the kernel time, so events around a single launch measure
    # the host.  Queue T launches behind a spin kernel and time the batch; inputs rotate through the sim-state pool and the
    # rollout storage (both larger than L2).
    def k1_queued(reps=5):
        out = []
        for _ in range(reps):
            torch.cuda.synchronize()
            torch.cuda._sleep(40_000_000)
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for t in range(w.T):
                w.env.bind_sim(**w.pool[t])
                w.env.set_obs_target(w.alg.storage.obs_row(t + 1))
                w.env.post_physics_step()
            a1.record()
            torch.cuda.synchronize()
            out.append(a0.elapsed_time(a1) / w.T)
        return float(np.median(out))
    k1_ms_inline = k1_ms
    k1_ms = k1_queued()

    # ---- the halves of an iteration on their own (max over ranks): rollout, bootstrap + GAE, update() ----
    def roll():
        w.obs = w.rollout()
        w.alg.storage.clear()
    roll_ms = cuda_ms(roll, 3, barrier, device, world)
    gae_ms = cuda_ms(lambda: w.alg.compute_returns(w.obs), 3, barrier, device, world)
    upd_ms = cuda_ms(lambda: w.alg.update(), 3, barrier, device, world)
    # ---- the one exchange step of the path: NCCL all-reduce of the flat gradient (675 KB), once per mini-batch (SURVEY 8e) ----
    allreduce_us = None
    if world > 1:
        allreduce_us = 1e3 * cuda_ms(lambda: w.alg._allreduce(0, w.alg.actor_critic.num_params), 20, barrier, device, world)
    dag = None
    if args.config == "roa":
        w.dagger_iteration()
        dag = dict(student_iteration_ms=cuda_ms(w.dagger_iteration, 2, barrier, device, world),
                   update_dagger_ms=cuda_ms(lambda: w.alg.update_dagger(), 2, barrier, device, world),
                   note="every dagger_update_freq = 20th iteration (OPR:125-169): rollout with the history-encoder latent + update_dagger() (PPO:265-291)")

    # ---- the other tensor-core mode on the same workload (reported next to the headline; dtype names which is which) ----
    other = {"tf32x3": "tf32", "tf32": "tf32x3"}.get(args.precision)
    alt = None
    if other:
        w.alg.precision = other
        for _ in range(2):
            w.iteration()
        ams, _ = timed(w, max(3, args.steps // 4))
        alt = {"dtype": DTYPE[other], "value": world * w.N * w.T * max(3, args.steps // 4) / (ams / 1e3), "unit": "env-steps/s",
               "ms_per_step": ams / max(3, args.steps // 4), "ppo_update_ms": cuda_ms(lambda: w.alg.update(), 3, barrier, device, world),
               "parity": "fp32 tolerances (tests/test_gpu_ppo.py::test_ppo_update_matches_reference_golden[tf32x3])" if other == "tf32x3" else
                         "TF32 tolerances (tests/test_gpu_ppo.py: TF32_TOL, 2 x the errors measured against the reference golden)"}
        w.alg.precision = args.precision

    # ---- e2e: host sim-state buffers, H2D every env step, D2H of the step result ----
    we = Workload(device, rank, config=args.config, world=world, group=group, host_inputs=True, precision=args.precision)
    for _ in range(3):
        we.iteration()
    ems, _ = timed(we, args.steps)
    e2e = world * we.N * we.T * args.steps / (ems / 1e3)
    del we

    if rank == 0:
        pk, src = peaks()
        k1_bytes = K1_BYTES_PER_ENV + (K1_BYTES_HEIGHT_SCAN if w.p.measure_heights else 0)
        achieved = w.N * k1_bytes / (k1_ms * 1e-3) / 1e9
        traffic = None
        tfile = os.path.join(ROOT, "profiles", "k1_traffic.json")
        if os.path.exists(tfile) and args.config == "flat":
            traffic = json.load(open(tfile)).get("dram_bytes_per_launch")
        mb_rows = w.N * w.T // 4
        line = {
            "metric": "env-steps/sec (widowGo1, 4096 envs/GPU)", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[args.precision], "data": "synthetic",
            "config": {"workload": CONFIGS[args.config]["label"] + ", T=40 rollout + GAE + PPO update (5 epochs x 4 mini-batches)",
                       "envs_per_gpu": w.N, "rollout_steps": w.T, "mini_batch_rows": mb_rows, "n_obs": 860,
                       "mlp_path": MLP_PATH[args.precision], "rng": "in-kernel Philox",
                       "cache": "inputs_larger_than_L2 (sim-state pool %d MB + rollout obs %d MB per GPU)" %
                                (w.sim_bytes * w.T // 2**20, (w.T + 1) * w.N * 860 * 4 // 2**20),
                       "parallelism": f"env-sharded dp{world}"},
            "ppo_update_ms": upd_ms, "ppo_minibatch_ms": upd_ms / 20, "rollout_ms": roll_ms, "gae_ms": gae_ms, "gpu_launches": int(launches),
            "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": int(w.sim_bytes * w.T), "d2h_bytes_per_step": int(w.N * 12 * w.T),
                    "ms_per_step": ems / args.steps},
            "roofline": {"kernel": "env_step_v2_kernel (fused post-physics, K1)", "bound": "hbm", "achieved": achieved, "peak": pk["hbm_gbs"],
                         "unit": "GB/s", "frac": achieved / pk["hbm_gbs"], "traffic": traffic, "peak_source": src,
                         "us_per_launch": k1_ms * 1e3, "algorithmic_bytes_per_launch": w.N * k1_bytes,
                         "timing": "CUDA events around 40 back-to-back launches queued behind a spin kernel (includes the 1-launch stats memset); "
                                   "events around single launches inside the rollout read %.1f us because the host submits slower than the kernel runs" % (k1_ms_inline * 1e3)},
            # second half of BASELINE's metric: the ActorCritic GEMMs of update() against the tensor-core roof.  Algorithmic work =
            # SURVEY 8d: 518 808 MAC per mini-batch row (forward 195 736 incl. the history encoder, backward 323 072), 20 mini-batches.
            "roofline_mlp": mlp_roofline(upd_ms, mb_rows, pk, args.precision),
            "clocks": clocks,
        }
        if alt:
            line["also"] = alt
        if dag:
            line["roa"] = dag
        if dist_parity:
            line["dist_parity"] = dist_parity
        if allreduce_us is not None:
            line["grad_allreduce"] = {"us_per_call": allreduce_us, "bytes": int(w.alg.actor_critic.num_params * 4), "calls_per_update": 20,
                                      "note": "NCCL all-reduce of the flat gradient buffer, back to back (max over ranks); exposed between the weight-gradient kernel and clip+Adam"}
        torch.cuda.synchronize()
        if world == 1:
            line["reference_eager_b200"] = reference_eager_block(device, w.N, w.T, roll_ms, gae_ms, upd_ms, k1_ms * w.T)
        line["cpu_baseline"] = cpu_baseline(args)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def reference_eager_block(device, n_envs, T, our_rollout_ms, our_gae_ms, our_update_ms, our_k1_total_ms):
    """Report-only: the UNMODIFIED reference rsl_rl (baseline/_ref) as eager PyTorch on this GPU -- act + process_env_step x T,
    compute_returns, update() on synthetic rollout data of the metric's shapes.  The reference has no Blackwell kernels: this IS its
    GPU path (SURVEY 2b / 8d).  The env half (legged_gym + Isaac Gym) cannot run here and is outside this block on both sides:
    `ours_same_scope_ms` = our rollout minus the post-physics kernels + bootstrap/GAE + update()."""
    from baseline import reference_eager as R
    why = R.available()
    if why:
        return {"unavailable": why}
    out = {}
    try:
        for name, tf in (("fp32", False), ("allow_tf32", True)):
            out[name] = R.time_iterations(device, n_envs, T, steps=3, warmup=2, allow_tf32=tf)
        torch.backends.cuda.matmul.allow_tf32 = False
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"reference eager run failed: {type(e).__name__}: {e}"}
    ours = our_rollout_ms - our_k1_total_ms + our_gae_ms + our_update_ms
    out["ours_same_scope_ms"] = ours
    out["ours_update_ms"] = our_update_ms
    out["speedup_update_vs_fp32"] = out["fp32"]["update_ms"] / our_update_ms
    out["speedup_same_scope_vs_fp32"] = out["fp32"]["iteration_ms"] / ours
    out["speedup_same_scope_vs_allow_tf32"] = out["allow_tf32"]["iteration_ms"] / ours
    out["note"] = "torch %s eager, device %s; allow_tf32 = the default of the reference's pinned torch 1.10" % (torch.__version__, torch.cuda.get_device_name(0))
    return out


def mlp_roofline(update_ms, mb_rows, pk, precision):
    flop = 2.0 * 518808 * mb_rows * 20
    achieved = flop / (update_ms * 1e-3) / 1e12
    bf16 = pk.get("bf16_tflops_sustained", pk.get("bf16_tflops", 1426.0))      # a kernel timed inside a long step: sustained figure
    tensor = precision in ("tf32", "tf32x3")
    peak = bf16 / 2 if tensor else 72.0      # TF32 dense = half the measured bf16 rate; fp32 CUDA cores: 148 SMs x 128 FMA x 1.9 GHz
    out = {"kernels": "chain2_kernel (fused forward / backward layer chains, loss in the epilogue) + wgrad_group_kernel" if tensor else "gemm_simt_kernel",
           "bound": "tensor" if tensor else "fp32 pipe", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
           "algorithmic_gflop_per_update": flop / 1e9, "update_ms": update_ms,
           "note": "ALGORITHMIC flops (SURVEY 8d) over the whole update(): Adam, packing, the history-encoder pass and every activation store / reload "
                   "included"}
    if precision == "tf32x3":
        out["executed_tensor_tflops"] = 3 * achieved
        out["note"] += "; the 3xTF32 path EXECUTES three tensor-core products per algorithmic one (executed_tensor_tflops), the fraction is quoted on the algorithmic count"
    return out


# ------------------------------------------------------------------------------------------------
# CPU legs: the reference's algorithm on the box's host cores, at the metric's own config (4096 envs x 40 steps).
# Update half = the UNMODIFIED reference rsl_rl (baseline/_ref: PPO.act / process_env_step / compute_returns / update) when it
# is installed (baseline/install_reference.sh), else the oracle port; env half = the oracle port of WidowGo1.post_physics_step (the
# reference env imports the closed isaacgym package).
# ------------------------------------------------------------------------------------------------
def make_oracle_iteration(n_envs, T, seed=100):
    import envstate as E
    from dwbc_b200 import synth
    from oracle import ppo_oracle as PO
    from oracle.pipeline import OracleIteration
    p = E.make_params("flat", n_envs)
    st = synth.initial_env_state(p, seed)
    st.update(synth.sim_state(p, seed, 0, rp_sigma=0.05, z_lo=0.327))
    manifest = PO.param_manifest()
    vals = synth.policy_params(manifest, 0)
    P = {n: (torch.tensor(INIT_STD) if v is None else torch.from_numpy(v).clone()) for (n, _), v in zip(manifest, vals)}
    sims = [synth.sim_state(p, seed, t, rp_sigma=0.05, z_lo=0.327) for t in range(1, 5)]
    tabs = [torch.from_numpy(synth.rand_table(p, seed, t)) for t in range(1, 5)]
    return OracleIteration(p, E.oracle_state(p, st), E.runtime(p), P, dict(HP), lambda t: sims[t % 4], lambda t: tabs[t % 4], T)


class CpuIteration:
    """One PPO iteration on the host: oracle env step + (reference rsl_rl | oracle port) policy / update."""

    def __init__(self, n_envs, T):
        from baseline import reference_eager as R
        self.it = make_oracle_iteration(n_envs, T)
        self.N, self.T = n_envs, T
        self.kind = "port"
        self.alg = None
        if R.available() is None:
            self.alg = R.make_reference_alg("cpu", n_envs, T)
            self.kind = "reference rsl_rl (unmodified, baseline/_ref) for act / process_env_step / compute_returns / update + oracle port of the post-physics step"
        self.obs = torch.zeros(n_envs, 860)

    def run(self):
        if self.alg is None:
            r = self.it.run()
            return dict(rollout=r["rollout"], gae=r["gae"], update=r["update"])
        it, alg = self.it, self.alg
        t0 = time.perf_counter()
        obs = self.obs
        with torch.inference_mode():                     # OPR:131-147
            for _ in range(self.T):
                it.step_count += 1
                actions = alg.act(obs, obs, False)
                it._load(it.sim_fn(it.step_count), actions)
                obs, rew, arew, rst, ex = it.env.post_physics_step(it.rand_fn(it.step_count), it.rt)
                alg.process_env_step(rew, arew, rst, {"time_outs": it.env.s.time_out_buf})
            t1 = time.perf_counter()
            alg.compute_returns(obs)
        t2 = time.perf_counter()
        alg.update()
        t3 = time.perf_counter()
        self.obs = obs
        return dict(rollout=t1 - t0, gae=t2 - t1, update=t3 - t2)


def pick_threads(n_envs=256):
    """torch CPU intra-op threading is counter-productive past a point for these op sizes (128
    OpenMP threads were 30x SLOWER than 8 on a 128-core host): probe a short slice of the
    workload at several thread counts up to all cores and keep the fastest, i.e. give the CPU arm
    its best configuration.  Returns (threads_used, host_cores)."""
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, cores) if c <= cores})
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        it = make_oracle_iteration(n_envs, 2)
        it.hp = dict(it.hp, num_learning_epochs=1, num_mini_batches=1)
        it.run()
        t0 = time.perf_counter()
        it.run()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
        if dt > 4 * best_t:
            break
    torch.set_num_threads(best)
    return best, cores


def cpu_baseline(args, n_envs=N_ENVS):
    cores, host_cores = pick_threads(512)
    it = CpuIteration(n_envs, T_STEPS)
    t0 = time.perf_counter()
    r = it.run()
    dt = time.perf_counter() - t0
    return {"value": n_envs * T_STEPS / dt, "unit": "env-steps/s", "cores": cores, "host_cores": host_cores, "kind": "reference" if it.alg is not None else "port",
            "implementation": it.kind,
            "sample": f"one full PPO iteration at the metric's config ({n_envs} envs x {T_STEPS} steps, 5 epochs x 4 mini-batches), "
                      f"{dt:.2f} s: rollout {r['rollout']:.2f} s, GAE {r['gae']:.3f} s, update {r['update']:.2f} s"}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    n_envs = N_ENVS
    cores, host_cores = pick_threads(512)
    it = CpuIteration(n_envs, T_STEPS)
    steps, warmup = args.steps, min(args.warmup, 1)      # ~5 s per iteration: one warm-up iteration is enough on the host
    for _ in range(warmup):
        it.run()
    t0 = time.perf_counter()
    for _ in range(steps):
        it.run()
    dt = time.perf_counter() - t0
    value = n_envs * T_STEPS * steps / dt
    sample = (f"each step = one full PPO iteration at the metric's config ({n_envs} envs x {T_STEPS} steps) on {cores} torch threads "
              f"(fastest of a probe up to all {host_cores} host cores); {steps} timed steps")
    print(json.dumps({
        "impl": "reference", "metric": "env-steps/sec (widowGo1, 4096 envs/GPU)", "value": value, "unit": "env-steps/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", 1)), "steps": steps, "warmup": warmup, "ms_per_step": dt / steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": CONFIGS["flat"]["label"] + ", T=40 rollout + GAE + PPO update (5 epochs x 4 mini-batches), CPU torch fp32",
                   "envs_per_gpu": n_envs, "rollout_steps": T_STEPS, "mini_batch_rows": n_envs * T_STEPS // 4, "n_obs": 860},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "reference" if it.alg is not None else "port",
                         "implementation": it.kind, "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="flat", choices=sorted(CONFIGS), help="BASELINE.json configs[1] (flat, the metric's), [2] (rough) or [3] (roa)")
    ap.add_argument("--precision", default="tf32x3", choices=["fp32", "tf32", "tf32x3"],
                    help="ActorCritic GEMM arithmetic: tf32x3 = error-compensated tensor cores (default: fp32-grade, passes the fp32 parity tests), "
                         "tf32 = plain TF32 tensor cores (what the reference's pinned torch 1.10 does on Ampere+, allow_tf32=True), fp32 = CUDA cores")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (losses, parameters, rollout storage, last observation; "
                         "rank 0) as DIR/<name>.npy, at most 64 MB")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
