#!/usr/bin/env python
"""Benchmark of the DQNFlappyBird hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--envs-per-gpu E] [--dump-outputs DIR]

One "step" = one batched ``frame_step`` (physics + render + cv2-exact preprocess into the device
frame ring) over every env of the job, with i.i.d. Bernoulli(0.5) actions (BASELINE.json
configs[1]: "batched frame_step + preprocess only, random actions").  Metric: env frames/s, whole
job.  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.

``--dump-outputs DIR`` writes what the last timed step returned on rank 0 as float32 ``DIR/<name>.npy``
(see ``dump_outputs``).  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

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

BYTES_PER_FRAME = 6400 + 64 + 1 + 4 + 1 + 4          # SURVEY 8(d): obs + state r/w + action + reward + terminal + score
METRIC = "env frames/sec (step+render+preproc)"
WORKLOAD = ("configs[1] op mix (batched frame_step + render + preprocess, random actions p=0.5, Philox gaps) "
            "at configs[4] scale: 1,048,576 envs / 8 GPUs")
UNIT = "frames/s"


_RESULT_OUT = None


def emit(line: dict):
    out = _RESULT_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def recorded_traffic(envs_per_gpu: int):
    """dram read+write bytes per launch of the step kernel from the committed ncu --set full capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_ncu_env_step_kernel_summary.json")) as f:
            d = json.load(f)
        if int(d["envs"]) == envs_per_gpu:
            return float(d["traffic_bytes_per_launch"])
    except Exception:
        pass
    return None


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------ CPU arm

def cpu_port_frames_per_s(n_envs: int, n_steps: int, threads: int, seed: int = 1234):
    """The oracle port (oracle/flappy_oracle.c: full-frame blits + cv2-exact resize, as the reference
    does per frame) on `threads` host threads, one env per reference process, random actions p=0.5."""
    import numpy as np
    from oracle import flappy_oracle as fo
    rng = np.random.default_rng(seed)
    env = fo.OracleEnvs(n_envs, seed=42)
    acts = (rng.random((n_steps + 2, n_envs)) < 0.5).astype(np.uint8)
    env.step(acts[0], want_obs=True, threads=threads)
    env.step(acts[1], want_obs=True, threads=threads)
    t0 = time.perf_counter()
    for t in range(n_steps):
        env.step(acts[2 + t], want_obs=True, threads=threads)
    dt = time.perf_counter() - t0
    return n_envs * n_steps / dt, dt


def cpu_port_updates_per_s(budget_s: float = 6.0):
    """The reference's learner on the host cores: BrainDQNNature's update at ITS OWN minibatch of 32 (BrainDQN.py:22) as the
    torch-CPU restatement of the TF-1.12 graph (oracle/qnet_oracle.py, float64 like the oracle; TensorFlow 1.12 is not
    installable) -- target forward, online forward, backward, Adam, all host threads."""
    import numpy as np
    from oracle import qnet_oracle as qo
    B = 32
    rng = np.random.default_rng(0)
    p = qo.init_params(512, False, seed=1); t = qo.init_params(512, False, seed=2)
    x = (rng.random((B, 5, 80, 80)) < 0.2).astype(np.uint8) * 255
    a = rng.integers(0, 2, B).astype(np.uint8)
    r = rng.choice(np.array([0.1, 3.0, -3.0], np.float32), B); term = (r == -3.0).astype(np.uint8)
    adam = qo.AdamTF1(len(p))
    qo.loss_and_grads(1, p, t, x[:, 0:4], x[:, 1:5], a, r, term)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s:
        _, g, *_ = qo.loss_and_grads(1, p, t, x[:, 0:4], x[:, 1:5], a, r, term)
        p = adam.step(p, g.astype(np.float32))
        n += 1
    dt = time.perf_counter() - t0
    return n / dt, n, dt


def cpu_reference_figures(budget_s: float):
    """The three labelled CPU figures of SURVEY 8(d) for the env half of the path, on this box's host cores:
    as shipped (30 frames/s/process), the reference verbatim on the pygame shim (clock neutralised, one process per core),
    and the C port (what SDL + cv2 would do natively).  None for the verbatim figure when oracle/_ref was not staged."""
    from oracle import ref_verbatim as rv
    cores = os.cpu_count() or 1
    out = {"as_shipped_frames_per_s_per_process": 30.0,
           "as_shipped_note": "FPSCLOCK.tick(FPS) sleeps every frame to 30 frames/s (wrapped_flappy_bird.py:14,179); one env per process"}
    if rv.available():
        procs = min(cores, 64)
        fps, dt = rv.env_frames_per_s(procs, 16)
        n_steps = max(16, int(fps / procs * budget_s))
        fps, dt = rv.env_frames_per_s(procs, n_steps)
        out["ref_verbatim"] = {"value": fps, "unit": UNIT, "cores": procs, "kind": "reference",
                               "sample": f"{procs} processes x {n_steps} frame_steps ({dt:.1f} s): game/wrapped_flappy_bird.py + flappy_bird_utils.py "
                                         "UNMODIFIED on the pygame shim (oracle/pygame_shim), game.FPSCLOCK replaced by a no-op object, real cv2 "
                                         "resize / cvtColor / threshold (FlappyBirdDQN.py:31-34); NumPy blits are slower than SDL's"}
        try:
            sample_ms, store_ms = rv.per_sample_ms(calls=2)
            out["per_verbatim"] = {"memory_sample_32_ms": sample_ms, "memory_store_ms": store_ms, "capacity": 50000, "kind": "reference",
                                   "sample": "BrainPrioritizedReplyDQN.py SumTree / Memory classes executed verbatim (AST-extracted), full 50,000-leaf tree"}
        except Exception as e:                              # pragma: no cover
            out["per_verbatim"] = {"error": str(e)[:200]}
    return out


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's own CPU implementation of the path for the same metric / config on the box's host
    cores.  With oracle/_ref staged (build() does it whenever a reference checkout is present) this is the reference's
    game/wrapped_flappy_bird.py run VERBATIM on the pygame shim, one process per core, the 30 frames/s clock neutralised,
    plus the real cv2 preprocess (kind "reference"); the C port's figure (kind "port": what SDL's C blits would cost) and the
    as-shipped 30 frames/s/process are reported beside it.  Without oracle/_ref: the C port alone."""
    if rank != 0:
        return
    import numpy as np
    from oracle import flappy_oracle as fo
    from oracle import ref_verbatim as rv
    cores = os.cpu_count() or 1
    threads = min(cores, 256)

    # ---- the C port (fair CPU figure), ~6 s
    n_envs = threads * 4
    port_fps, _ = cpu_port_frames_per_s(n_envs, 2, threads)
    port_steps = max(4, int(port_fps * 6.0 / n_envs))
    port_fps, port_dt = cpu_port_frames_per_s(n_envs, port_steps, threads)
    port = {"value": port_fps, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{n_envs} envs x {port_steps} frame_steps ({port_dt:.1f} s), oracle/flappy_oracle.c (full 288x512 blits + cv2-exact resize / gray / threshold) on {threads} threads"}
    if rv.available():
        procs = min(cores, 64)
        rate, _ = rv.env_frames_per_s(procs, 16)                     # calibration
        seg_s = min(4.0, args.reference_budget_s / (args.steps + args.warmup))
        n_steps = max(1, int(rate / procs * seg_s))
        segs = rv.env_segments(procs, n_steps, args.warmup + args.steps)
        timed = segs[args.warmup:]
        total_t = sum(timed)
        value = procs * n_steps * args.steps / total_t
        kind, used = "reference", procs
        sample = (f"each bench step = {procs} reference processes x {n_steps} frame_steps of the same workload: game/wrapped_flappy_bird.py + "
                  "flappy_bird_utils.py UNMODIFIED on the pygame shim (pygame / SDL are not installable), FPSCLOCK.tick neutralised, real cv2 "
                  "preprocess (FlappyBirdDQN.py:31-34)")
    else:
        rng = np.random.default_rng(1234)
        env = fo.OracleEnvs(n_envs, seed=42)

        def run(n):
            acts = (rng.random((n, n_envs)) < 0.5).astype(np.uint8)
            t0 = time.perf_counter()
            for t in range(n):
                env.step(acts[t], want_obs=True, threads=threads)
            return time.perf_counter() - t0
        budget_s = min(1.0, args.reference_budget_s / (args.steps + 0.25 * args.warmup))
        n_steps = max(1, int(port_fps * budget_s / n_envs))
        for _ in range(args.warmup):
            run(max(1, n_steps // 4))
        total_t = sum(run(n_steps) for _ in range(args.steps))
        value = n_envs * n_steps * args.steps / total_t
        kind, used = "port", threads
        sample = f"each bench step = {n_envs} envs x {n_steps} frame_steps of the C port (oracle/_ref not staged: no reference checkout at build time)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs_per_gpu": args.envs_per_gpu, "envs_total": args.envs_per_gpu * max(args.gpus, 1),
                   "cpu_sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": kind, "sample": sample,
                         "c_port": port,
                         "as_shipped": "30 frames/s/process: FPSCLOCK.tick(FPS) sleeps every frame (wrapped_flappy_bird.py:14,179)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------ GPU arm

DUMP_MAX_ENVS = 1 << 18            # reward / terminal / score / state of at most this many envs: 20 MB
DUMP_OBS_ENVS = 512                # 80x80 observations of this many envs: 13 MB


def dump_outputs(out_dir: str, gs, reward, terminal, score):
    """What ``frame_step`` hands its caller after the last timed step, as float32 .npy files: reward, terminal and score
    per env (every env up to DUMP_MAX_ENVS, else a fixed seeded sample, listed in env_index), the 80x80 observation of a
    fixed seeded sample of DUMP_OBS_ENVS envs (listed in obs_env_index), and the 16-int env state after the step
    (``GameState.export_state``) of the envs in env_index.  The state carries what every earlier step did: with random
    actions at p = 0.5 every env crashes on the same step, once every 50 steps, and none ever scores, so the last step
    alone usually holds no crash and no score.  The samples depend only on the env count."""
    import numpy as np
    import torch
    E = gs.num_envs
    rng = np.random.default_rng(0)
    envs = np.arange(E) if E <= DUMP_MAX_ENVS else np.sort(rng.choice(E, DUMP_MAX_ENVS, replace=False))
    obs_envs = np.sort(rng.choice(E, min(E, DUMP_OBS_ENVS), replace=False))
    pick = lambda t, idx: t[torch.from_numpy(idx).to(t.device)].cpu().numpy()
    arrays = {"reward": pick(reward, envs), "terminal": pick(terminal, envs), "score": pick(score, envs), "env_index": envs,
              "obs": pick(gs.ring[:, gs.slot], obs_envs), "obs_env_index": obs_envs, "state": pick(gs.export_state(), envs)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def run_ours(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist
    from dqnflappybird_b200.game import GameState

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    E = args.envs_per_gpu
    gs = GameState(num_envs=E, device=dev, seed=42, history=4, first_env_id=rank * E)
    rew = torch.empty(E, dtype=torch.float32, device=dev)
    term = torch.empty(E, dtype=torch.uint8, device=dev)
    score = torch.empty(E, dtype=torch.int32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step():
        gs.step_random(1, 0.5, 1234, None, rew, term, score)

    # decorrelate episode phases (SURVEY 8d) without drawing, then warm up the real step
    gs.step_random(min(args.decorrelate, 1000), 0.5, 1234, draw=False)
    for _ in range(max(args.warmup, 3)):
        one_step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        one_step()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    gs.check_errors()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, gs, rew, term, score)

    # ---- e2e: the reference-facing call with HOST buffers (actions in, reward/terminal/score out EVERY step).
    # Measured twice: strictly synchronous (one step in flight), and as a user would drive a throughput job --
    # fb_env_step_host_submit / _wait with two steps in flight and two sets of pinned buffers, so that the copies of
    # step t overlap the kernel of step t+1.  Every step's results are waited for inside the timed region.
    def pinned_set():
        return ((torch.rand(E) < 0.5).to(torch.uint8).pin_memory(), torch.zeros(E, dtype=torch.float32).pin_memory(),
                torch.zeros(E, dtype=torch.uint8).pin_memory(), torch.zeros(E, dtype=torch.int32).pin_memory())
    bufs = [pinned_set(), pinned_set()]
    for _ in range(3):
        gs.frame_step_host(*bufs[0])
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        gs.frame_step_host(*bufs[0])
    torch.cuda.synchronize()
    e2e_sync_s = time.perf_counter() - t0
    barrier()
    t0 = time.perf_counter()
    gs.frame_step_host_submit(*bufs[0])
    for k in range(1, args.steps):
        gs.frame_step_host_submit(*bufs[k & 1])
        gs.frame_step_host_wait()                    # results of step k-1 are on the host now
    gs.frame_step_host_wait()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert abs(float(bufs[0][1].abs().max()) - 3.0) < 1e-6 or abs(float(bufs[0][1].abs().max()) - 0.1) < 1e-6, "host rewards not delivered"
    te = torch.tensor([e2e_s, e2e_sync_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s, e2e_sync_s = float(te[0]), float(te[1])

    learner = None
    if not args.no_learner:
        learner = bench_learner(args, rank, world, dev)
    # ---- BASELINE.json configs as written, through the reference's own loop (act -> frame_step -> setPerception + update)
    loops = None
    if not args.no_learner and not args.no_closed_loop:
        del gs
        torch.cuda.empty_cache()
        loops = {}
        # configs[4]: BrainDoubleDQN + BrainDuelingDQN acting on 1,048,576 envs over 8 GPUs = 131,072 per GPU (weak scaling)
        for m in ("ddqn", "duelingdqn"):
            loops[f"configs4_{m}"] = closed_loop(m, E, args.learner_batch * world, 1, 8, dev, rank, world)
        if world == 1:
            # configs[4] on ONE GPU (strong-scaling anchor): all 1,048,576 envs, ring u8[1048576][5][80][80] = 33.6 GB
            loops["configs4_ddqn_1M_envs_one_gpu"] = closed_loop("ddqn", 1048576, args.learner_batch, 1, 3, dev, rank, world)
            # configs[2] closed loop: BrainDQNNature, 16,384 envs, minibatch 256
            loops["configs2_dqnnature"] = closed_loop("dqnnature", args.learner_envs, args.learner_batch, 28, 40, dev, rank, world)
            # configs[0]: the reference's own case -- 1 env, BrainDQN, minibatch 32, replay 50,000 (BrainDQN.py:19-28; OBSERVE as
            # shipped is 1000, BASELINE.json says 10000: neither matters for a rate, the loop is timed past it)
            loops["configs0_dqn_1_env"] = closed_loop("dqn", 1, 32, 50000, 300, dev, rank, world, observe_steps=40)
    if rank != 0:
        return
    total_envs = E * world
    value = total_envs * args.steps / (ms_max * 1e-3)
    peak, peak_src = measured_peak_hbm()
    achieved = BYTES_PER_FRAME * E / (ms_max * 1e-3 / args.steps) / 1e9         # per GPU, per launch
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        threads = min(cores, 256)
        n_envs = threads * 4
        fps, _ = cpu_port_frames_per_s(n_envs, 2, threads)
        n_steps = max(4, int(fps * 8.0 / n_envs))            # ~8 s of CPU work
        fps, dt = cpu_port_frames_per_s(n_envs, n_steps, threads)
        port = {"value": fps, "unit": UNIT, "cores": threads, "kind": "port",
                "sample": f"{n_envs} envs x {n_steps} frame_steps ({dt:.1f} s) of the same workload, oracle/flappy_oracle.c on {threads} threads "
                          "(full 288x512 blits + cv2-exact resize, what SDL + cv2 do natively)"}
        figs = cpu_reference_figures(10.0)
        if "ref_verbatim" in figs:                            # the reference itself, verbatim; the fair C figure and the 30 fps fact beside it
            cpu = dict(figs["ref_verbatim"])
            cpu["c_port"] = port
        else:
            cpu = port
        cpu["as_shipped"] = figs["as_shipped_note"]
        if "per_verbatim" in figs:
            cpu["per_verbatim"] = figs["per_verbatim"]
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "envs_per_gpu": E, "envs_total": total_envs, "ring": f"u8[{E}][4][80][80] = {E * 25600 / 1e9:.2f} GB per GPU",
                   "l2": "inputs larger than L2 (ring >> 126 MB; every frame is written once and not re-read)",
                   "parallelism": f"env-sharded x{world}, no collective"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": recorded_traffic(E), "traffic_source": "profiles/r02_ncu_env_step_kernel_summary.json (dram read + write bytes per launch, ncu --set full of this round's kernel)",
                     "achieved_bytes_per_launch": BYTES_PER_FRAME * E, "peak_source": peak_src, "kernel": "env_step_kernel",
                     "algorithmic_bytes_per_frame": BYTES_PER_FRAME},
        "cpu_baseline": cpu,
        "e2e": {"value": total_envs * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": E * 1, "d2h_bytes_per_step": E * 9,
                "in_flight": 2, "value_synchronous": total_envs * args.steps / e2e_sync_s,
                "note": "fb_env_step_host_submit/_wait: pinned host actions in, reward/terminal/score out and waited for EVERY step, two "
                        "steps in flight (copies of step t overlap the kernel of step t+1); value_synchronous = fb_env_step_host, one "
                        "step in flight; the 80x80 observation stays in the device ring by design"},
        "gpu_launches": args.steps,
        "clocks": clocks,
        # the second half of BASELINE.json's metric, at top level (details under "learner"): DQN updates/s of configs[2]
        "updates_per_s": learner and learner["updates_per_s"],
        "learner_ms_per_update": learner and learner["ms_per_update"],
        "learner_transitions_per_s": learner and learner["transitions_per_s"],
        "learner_frac_of_tensor_peak": learner and learner["frac_of_bf16_tensor_peak"],
        "learner_precision": args.learner_precision,
        "learner_weak_efficiency": learner and learner["weak_efficiency_in_run"],
        "exchange_us": learner and learner["exchange_us"],
        "learner_checks": learner and learner["checks"],
        "learner": learner,
        "closed_loop": loops,
    }
    emit(line)


FLOP_FWD, FLOP_BWD = 11675648, 16797696            # SURVEY 2.2 / 8(d), per sample


def verify_and_time_exchange(brain, dev, world, K, sync):
    """N > 1, inside the bench run (the driver's scaling runs are then also the multi-GPU parity runs):
      * every rank holds bit-identical parameters / Adam slots after the timed updates (all-gather of two checksums);
      * ONE exchange step (gradient sum over NVLink peer memory fused with Adam, csrc/fb_dist.cu) equals NCCL all-reduce + the same
        Adam kernel on copies: summed gradients to 1e-6 relative (NCCL's ring order differs from the rank order of the fused
        kernel), parameters to 1e-9 absolute (|update| ~ lr = 1e-6);
      * replicas are still bit-identical after it.
    Then the same update WITHOUT the exchange (each rank's own gradients, on scratch copies of the state): its time against
    the exchanged update's gives the in-run weak-scaling efficiency and the exchange's cost.  Raises on any mismatch."""
    import torch
    import torch.distributed as dist
    from dqnflappybird_b200 import _lib
    net = brain.net
    L = _lib.lib()

    def checksums():
        h = net.params.view(torch.int32).to(torch.int64)
        w = (torch.arange(h.numel(), device=dev, dtype=torch.int64) % 1000003) + 1
        m = net.adam_m.view(torch.int32).to(torch.int64)
        c = torch.stack([h.sum(), (h * w).sum(), (m * w).sum()])
        out = [torch.empty_like(c) for _ in range(world)]
        dist.all_gather(out, c)
        return all(torch.equal(out[0], o) for o in out)

    sync()
    ok_before = checksums()
    assert ok_before, "replicas diverged during the timed updates"
    res = {"replicas_bitwise_equal_after_timed_updates": True}
    if net.exchange is not None:
        mb = brain.replayMemory.sample(brain.local_batch)
        net.loss_backward(brain.variant, mb.frames, mb.actions, mb.rewards, mb.terminals, None, brain.gamma, brain.loss_sum,
                          brain.local_batch * world)
        g_nccl = net.grads.clone()
        dist.all_reduce(g_nccl, op=dist.ReduceOp.SUM)
        p_ref, m_ref, v_ref = net.params.clone(), net.adam_m.clone(), net.adam_v.clone()
        import numpy as np
        one = np.float32(1)
        alpha = np.float32(net.lr * np.sqrt(one - net.beta2_power) / (one - net.beta1_power))
        ref_net_adam = lambda p, g, m, v: _lib.check(L.fb_qnet_adam(net._h, p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), float(alpha),
                                                                 float(net.beta1), float(net.beta2), float(net.adam_eps), 1.0,
                                                                 torch.cuda.current_stream().cuda_stream), "fb_qnet_adam")
        ref_net_adam(p_ref, g_nccl, m_ref, v_ref)
        reduced = torch.empty_like(net.grads)
        net.exchange.adam(net, alpha, 1.0, reduced_out=reduced, wait=True)
        net.grads = net.exchange.grads
        net._advance_powers()
        _lib.check(L.fb_qnet_invalidate(net._h), "fb_qnet_invalidate")     # the reference Adam re-packed operands from p_ref
        sync()
        gmax = g_nccl.abs().max().item()
        rel = ((reduced - g_nccl).abs().max() / max(gmax, 1e-30)).item()
        dp = (net.params - p_ref).abs().max().item()
        assert rel <= 1e-6, f"fused exchange: summed gradient differs from the NCCL all-reduce by {rel:.2e} (relative to max |g|)"
        assert dp <= 1e-9, f"fused exchange + Adam: parameters differ from NCCL all-reduce + Adam by {dp:.2e}"
        assert checksums(), "replicas diverged after the checked exchange step"
        res.update({"exchange_step_vs_nccl_allreduce_plus_adam": {"grad_max_rel": rel, "param_max_abs": dp},
                    "replicas_bitwise_equal_after_checked_step": True})
    # ---- the same update without the exchange, on scratch state (replicas must not diverge)
    saved = (net.params.clone(), net.adam_m.clone(), net.adam_v.clone(), net.beta1_power, net.beta2_power, net.adam_steps)
    ex, net.exchange = net.exchange, None
    in_step, net.exchange_in_step = net.exchange_in_step, False
    _lib.check(L.fb_qnet_attach_exchange(net._h, None), "fb_qnet_attach_exchange")
    grads_saved = net.grads
    net.grads = torch.zeros_like(saved[0])
    world_saved, brain.world = brain.world, 1
    import torch.cuda
    for _ in range(5):
        brain._update(brain.variant)
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        brain._update(brain.variant)
    e1.record(); sync()
    ms_local = e0.elapsed_time(e1) / K
    brain.world = world_saved
    net.exchange, net.grads, net.exchange_in_step = ex, grads_saved, in_step
    _lib.check(L.fb_qnet_attach_exchange(net._h, ex._h if (ex is not None and in_step) else None), "fb_qnet_attach_exchange")
    net.params.copy_(saved[0]); net.adam_m.copy_(saved[1]); net.adam_v.copy_(saved[2])
    net.beta1_power, net.beta2_power, net.adam_steps = saved[3], saved[4], saved[5]
    _lib.check(L.fb_qnet_invalidate(net._h), "fb_qnet_invalidate")
    t = torch.tensor([ms_local], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    assert checksums(), "replicas diverged after restoring the state"
    return res, float(t[0])


def closed_loop(model, n_envs, batch, replay_per_env, steps, dev, rank, world, observe_steps=4, max_act_batch=4096):
    """The reference's own loop (FlappyBirdDQN.py:72-76) on the device: getAction -> frame_step -> setPerception with one
    minibatch update per step once past OBSERVE -- acting with the Q-network, stepping every env, appending to replay (no copy:
    the env draws into the Brain's ring) and training.  Returns env frames/s and updates/s of this rank."""
    import torch
    from dqnflappybird_b200.brains import MODELS
    from dqnflappybird_b200.game import GameState
    brain = MODELS[model](2, "bird", num_envs=n_envs, device=dev, seed=0, first_env_id=rank * n_envs, replay_memory_per_env=replay_per_env,
                          batch_size=batch, observe=observe_steps, max_act_batch=max_act_batch)
    gs = GameState(num_envs=n_envs, device=dev, seed=17, first_env_id=rank * n_envs, history=brain.ring.shape[1], ring=brain.ring)
    a0 = torch.zeros(n_envs, dtype=torch.uint8, device=dev) if n_envs > 1 else [1, 0]
    obs, *_ = gs.frame_step(a0)
    brain.setInitState(obs)

    def one():
        action = brain.getAction()
        out = brain.next_rows()[1:] if n_envs > 1 else None
        nxt, reward, terminal, score = gs.frame_step(action, out=out)
        brain.setPerception(nxt, action, reward, terminal, score)
    for _ in range(observe_steps + 8):
        one()
    torch.cuda.synchronize()
    upd0 = brain.net.adam_steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        one()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    gs.check_errors()
    res = {"model": model, "envs_per_gpu": n_envs, "envs_total": n_envs * world, "minibatch": batch, "steps": steps,
           "env_frames_per_s": n_envs * world * steps / (ms * 1e-3), "updates_per_s": (brain.net.adam_steps - upd0) / (ms * 1e-3),
           "ms_per_loop_step": ms / steps, "precision": brain.net.precision}
    del brain, gs
    torch.cuda.empty_cache()
    return res


def bench_learner(args, rank, world, dev):
    """Second half of BASELINE.json's metric: DQN updates/s (configs[2]: BrainDQNNature, 16384 envs, minibatch 256).
    One update = sample + gather + 2 forwards + backward (+ gradient all-reduce at N > 1) + Adam.  Also times acting
    (one forward + epsilon-greedy for every env).  Replay is pre-filled from a random-action rollout."""
    import torch
    import torch.distributed as dist
    from dqnflappybird_b200.brains import BrainDQNNature
    from dqnflappybird_b200.game import GameState
    # weak scaling like the env leg: every GPU keeps configs[2]'s minibatch of 256, the global minibatch is 256 x world
    # (--learner-scaling strong splits ONE minibatch of 256 over the ranks instead)
    N, C = args.learner_envs, 28
    B = args.learner_batch * (world if args.learner_scaling == "weak" else 1)
    brain = BrainDQNNature(2, "bird", num_envs=N, device=dev, replay_memory_per_env=C, batch_size=B, observe=1e18, seed=0,
                           first_env_id=rank * N, max_act_batch=4096, precision=args.learner_precision)
    gs = GameState(num_envs=N, device=dev, seed=42, history=C + 4, first_env_id=rank * N, ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device=dev))
    brain.setInitState(obs)
    for k in range(1, C + 9):                       # pre-fill the replay ring with random-action transitions
        a_row, r_row, t_row = brain.replayMemory.rows(k)
        gs.step_random(1, 0.5, 1234, a_row, r_row, t_row, None)
        brain._k = k
        brain.replayMemory.appended(k)
    brain.timeStep = 1                              # no target sync inside the timed loop except every 500th update
    K, W = args.learner_updates, 5

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(W):
        brain._trainQNetwork(); brain.timeStep += 1
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        brain._trainQNetwork(); brain.timeStep += 1
    e1.record()
    sync()
    ms_upd = e0.elapsed_time(e1) / K
    checks, ms_local = None, None
    if world > 1:
        checks, ms_local = verify_and_time_exchange(brain, dev, world, K, sync)
    for _ in range(2):
        brain.getAction()
    sync()
    e0.record()
    for _ in range(5):
        brain.getAction()
    e1.record()
    sync()
    ms_act = e0.elapsed_time(e1) / 5
    t = torch.tensor([ms_upd, ms_act], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_upd, ms_act = float(t[0]), float(t[1])
    # ---- the dominant GEMM of the update in isolation: conv1 forward (56 % of the forward FLOPs), re-launched on the
    # workspace contents.  At the update's own batch its operands are L2-resident by construction; at the acting chunk
    # (2048 samples: 116 MB of operands + 58 MB of output > L2) they stream from HBM.
    kern = None
    if args.learner_precision in ("bf16", "fp16"):
        from dqnflappybird_b200 import _lib
        L = _lib.lib()
        st = torch.cuda.current_stream().cuda_stream
        kern = {}
        for kb, reps in ((brain.local_batch, 50), (min(2048, brain.net.max_batch), 20)):
            fbv = brain._act_view()
            fbv.batch = kb
            brain.net.forward(fbv)                                   # fills the workspace at this batch
            _lib.check(L.fb_debug_tc_kernel(brain.net._h, 10, kb, 3, brain.net.params.data_ptr(), st), "probe")
            sync()
            e0.record()
            _lib.check(L.fb_debug_tc_kernel(brain.net._h, 10, kb, reps, brain.net.params.data_ptr(), st), "probe")
            e1.record(); sync()
            us = e0.elapsed_time(e1) * 1e3 / reps
            kern[kb] = {"us": us, "tflops": 6553600 * kb / (us * 1e-6) / 1e12,
                        "hbm_gbs": kb * (441 * (128 + 64) + 49 * 256) / (us * 1e-6) / 1e9}
    # ---- the other DQN-family agents of BASELINE.json's configs on the same workload (same envs, replay and minibatch):
    # Double (configs[4]), Dueling (configs[4]), prioritized replay with the device sum-tree (configs[3])
    variants = {"dqnnature": {"updates_per_s": 1e3 / ms_upd, "ms_per_update": ms_upd}}
    if not args.no_learner_variants:
        from dqnflappybird_b200.brains import BrainDoubleDQN, BrainDuelingDQN, BrainPrioritizedReplyDQN
        ring_shared = brain.ring
        for name, cls in (("ddqn", BrainDoubleDQN), ("duelingdqn", BrainDuelingDQN), ("prioritydqn", BrainPrioritizedReplyDQN)):
            vb = cls(2, "bird", num_envs=N, device=dev, ring=ring_shared, replay_memory_per_env=C, batch_size=B, observe=1e18, seed=0,
                     first_env_id=rank * N, max_act_batch=4096, precision=args.learner_precision)
            vb._k = brain._k
            for k in range(max(1, brain._k - C + 1), brain._k + 1):      # the ring already holds the rollout: register its steps
                a_row, r_row, t_row = vb.replayMemory.rows(k)
                a0, r0, t0 = brain.replayMemory.rows(k)
                a_row.copy_(a0); r_row.copy_(r0); t_row.copy_(t0)
                vb.replayMemory.appended(k)
            vb.timeStep = 1
            for _ in range(W):
                vb._trainQNetwork(); vb.timeStep += 1
            sync()
            e0.record()
            for _ in range(K):
                vb._trainQNetwork(); vb.timeStep += 1
            e1.record(); sync()
            tv = torch.tensor([e0.elapsed_time(e1) / K], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tv, op=dist.ReduceOp.MAX)
            variants[name] = {"updates_per_s": 1e3 / float(tv[0]), "ms_per_update": float(tv[0])}
            del vb
    # ---- the same update at the three precisions of the library, side by side (fixed minibatch of the configured size; one
    # graph launch each on the tensor-core paths): fp32 = CUDA-core FMA (the strict anchor), bf16 = 8-bit significand, fp16 =
    # 11-bit significand (TF32's), the default
    by_precision = {}
    if not args.no_learner_variants and world == 1:
        from dqnflappybird_b200.qnet import QNetwork
        mbp = brain.replayMemory.sample(brain.local_batch)
        fr, ac, rw, tm = mbp.frames.clone(), mbp.actions.clone(), mbp.rewards.clone(), mbp.terminals.clone()
        for prec in ("fp32", "bf16", "fp16"):
            netp = QNetwork(device=dev, max_batch=brain.local_batch, precision=prec, seed=0)
            for _ in range(4):
                netp.train_step("nature", fr, ac, rw, tm)
            sync()
            Kp = K if prec != "fp32" else max(5, K // 5)
            e0.record()
            for _ in range(Kp):
                netp.train_step("nature", fr, ac, rw, tm)
            e1.record(); sync()
            msp = e0.elapsed_time(e1) / Kp
            by_precision[prec] = {"updates_per_s": 1e3 / msp, "ms_per_update": msp, "compute_path": netp.compute_path,
                                  "includes": "update on a fixed minibatch (no sampling / gather)"}
            del netp
    # ---- minibatch sweep (BrainDQNNature): the 256 of configs[2] is launch/latency-bound on a B200; the same step at
    # larger minibatches shows what the kernels sustain
    sweep = {str(B): {"updates_per_s": 1e3 / ms_upd, "transitions_per_s": B * 1e3 / ms_upd, "includes": "sample + gather + update"}}
    if not args.no_learner_variants and world == 1:
        from dqnflappybird_b200.qnet import QNetwork
        for mb_size in (1024, 4096):
            parts = [brain.replayMemory.sample(brain.local_batch) for _ in range(1)]
            fr, ac, rw, tm = [], [], [], []
            for _ in range(mb_size // brain.local_batch):
                mbp = brain.replayMemory.sample(brain.local_batch)
                fr.append(mbp.frames.clone()); ac.append(mbp.actions.clone()); rw.append(mbp.rewards.clone()); tm.append(mbp.terminals.clone())
            fr, ac, rw, tm = torch.cat(fr), torch.cat(ac), torch.cat(rw), torch.cat(tm)
            netv = QNetwork(device=dev, max_batch=mb_size, precision=args.learner_precision, seed=0)
            for _ in range(3):
                netv.train_step("nature", fr, ac, rw, tm)
            sync()
            Kv = max(10, K // 4)
            e0.record()
            for _ in range(Kv):
                netv.train_step("nature", fr, ac, rw, tm)
            e1.record(); sync()
            msv = e0.elapsed_time(e1) / Kv
            sweep[str(mb_size)] = {"updates_per_s": 1e3 / msv, "transitions_per_s": mb_size * 1e3 / msv,
                                   "tflops": (2 * FLOP_FWD + FLOP_BWD) * mb_size / (msv * 1e-3) / 1e12,
                                   "includes": "update only on a fixed minibatch (the CPython-exact sampler is one CTA, <= 512 draws)"}
            del netv, fr
    cpu_upd = None
    if world == 1 and not args.no_cpu_baseline:
        ups, n_done, dt = cpu_port_updates_per_s()
        cpu_upd = {"value": ups, "unit": "updates/s", "minibatch": 32, "cores": os.cpu_count() or 1, "kind": "port",
                   "sample": f"{n_done} BrainDQNNature updates of minibatch 32 in {dt:.1f} s: oracle/qnet_oracle.py (torch CPU float64 "
                             "restatement of the TF-1.12 graph; TensorFlow 1.12 is not installable), all host threads"}
    flop_upd = (2 * FLOP_FWD + FLOP_BWD) * B
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            tc_peak = float(json.load(f)["bf16_tflops"])
    except Exception:
        tc_peak = 1590.0
    return {"metric": "DQN updates/sec", "model": "BrainDQNNature (target net), fc512, one max-pool (as coded)", "envs_per_gpu": N,
            "minibatch_global": B, "minibatch_per_gpu": brain.local_batch, "updates_per_s": 1e3 / ms_upd, "ms_per_update": ms_upd,
            "flop_per_update": flop_upd, "tflops": flop_upd / (ms_upd * 1e-3) / 1e12 / max(world, 1) * 1.0,
            "frac_of_bf16_tensor_peak": flop_upd / world / (ms_upd * 1e-3) / 1e12 / tc_peak, "tensor_peak_tflops": tc_peak,
            "compute_path": brain.net.compute_path if hasattr(brain.net, "compute_path") else "fp32 CUDA-core implicit GEMM",
            "act_envs_per_s": N * world / (ms_act * 1e-3), "ms_per_act": ms_act,
            "act_tflops_per_gpu": N * FLOP_FWD / (ms_act * 1e-3) / 1e12,
            "transitions_per_s": B * 1e3 / ms_upd, "scaling": args.learner_scaling, "cpu_baseline": cpu_upd, "variants": variants, "minibatch_sweep": sweep,
            "by_precision": by_precision, "precision": args.learner_precision,
            "ms_per_update_without_exchange": ms_local,
            "exchange_us": None if ms_local is None else (ms_upd - ms_local) * 1e3,
            "weak_efficiency_in_run": None if ms_local is None else ms_local / ms_upd,
            "checks": checks,
            "gradient_exchange": ("none (1 GPU)" if world == 1 else
                                  "inside the step's graph: NVLink peer-memory sum fused with Adam, W_fc1's bucket beside the conv gradients "
                                  "(adam_xbucket_kernel)" if brain.net.exchange_in_step else
                                  "fused into Adam over NVLink peer memory (fb_dist_adam)" if brain.net.exchange is not None else "NCCL all-reduce"),
            "roofline": None if not kern else {
                "bound": "tensor", "kernel": "tc_conv1_fused_kernel<6,true> (conv1 forward of the training step: TMA slab + tcgen05.mma, N = 32, "
                                             "bias + ReLU + 2x2 max-pool in the epilogue, Z1 and P2 out)",
                "algorithmic_flop_per_sample": 6553600, "unit": "TFLOP/s", "peak": tc_peak,
                "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops, cuBLAS burst)",
                # quoted at the CONFIGURED minibatch (configs[2]: 256); the larger batch is there for the kernel's own ceiling
                "batch": brain.local_batch,
                "achieved": kern[brain.local_batch]["tflops"],
                "frac": kern[brain.local_batch]["tflops"] / tc_peak,
                "whole_step_frac": flop_upd / world / (ms_upd * 1e-3) / 1e12 / tc_peak,
                "whole_step_tensor_pipe_active_pct_ncu": 3.1,
                "whole_step_source": "profiles/r02_ncu_learner_step_summary.json (ncu --set full of every kernel of one update)",
                "by_batch": {str(k): v for k, v in kern.items()},
                "note": "per launch, CUDA events over back-to-back launches; a tcgen05.mma of N = 32 is bound by its operand reads from "
                        "shared memory at 16/40 of the math rate (profiles/r01_tcgen05_mma_rate_b200.txt), so 0.40 is this layer's ceiling; "
                        "at batch 2048 the operands (X2 read 56 KB + Z1 write 28 KB + P2 6 KB per sample) exceed L2 and stream at "
                        "hbm_gbs; ncu traffic and pipe utilisation: profiles/r01_ncu_tc_kernels_summary.json"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=131072)
    ap.add_argument("--decorrelate", type=int, default=1000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-learner", action="store_true")
    ap.add_argument("--learner-envs", type=int, default=16384)
    ap.add_argument("--learner-batch", type=int, default=256)
    ap.add_argument("--learner-updates", type=int, default=50)
    ap.add_argument("--learner-precision", default="fp16", choices=["fp16", "bf16", "fp32"])
    ap.add_argument("--learner-scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-learner-variants", action="store_true")
    ap.add_argument("--no-closed-loop", action="store_true")
    ap.add_argument("--reference-budget-s", type=float, default=120.0, help="--impl reference: CPU seconds for warm-up + all steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl ours: write the last timed step's reward / terminal / score / observations / env state (rank 0) "
                         "as float32 DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the device path's outputs: it needs --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries the one JSON line and nothing else: file descriptor 1 is pointed at stderr for everything libraries
    # print on their own (NCCL writes "NCCL version ..." to stdout), and the line goes out through the saved descriptor
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
