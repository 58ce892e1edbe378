#!/usr/bin/env python
"""Benchmark of the FurnitureEnv.step() hot path (BASELINE.json metric: aggregate env-steps/s, FurnitureSawyerEnv +
table_lack_0825, 4096 envs per GPU; one env-step = one env.step() = 50 mj_steps + action mapping + connect check +
obs + reward, SURVEY.md 8d).

  python bench.py --gpus N --steps K --warmup W            this repo's CUDA engine (one process per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  the CPU restatement of the reference loop (oracle/ref_env.py
                                                           over oracle/fe_oracle.c) on all host cores; rank 0 only
  python bench.py ... --dump-outputs DIR                   also write what the last timed step returned (DIR/<name>.npy):
                                                           the inputs are seeded, so two builds can be compared output for output

Prints ONE JSON line (see the contract in the task statement / DESIGN.md "Measurement").
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "aggregate env-steps/sec, Sawyer+table_lack @4096 envs/GPU"
UNIT = "env-steps/s"
ENVS_PER_GPU = 4096
B_ENV = 58700  # algorithmic bytes per env-step, SURVEY.md 8d: 50 * 4*(2 nq + 5 nv + nu) + 4*(obs_dim + act_dim) + 8
WORKLOAD = "FurnitureSawyerEnv + table_lack_0825, control_type=impedance, 50 mj_steps per env-step, random actions U(-1,1)"


def b_env(model, obs_dim, act_dim, nsub=50):
    """SURVEY.md 8d: B_sub = 4 (2 nq + 5 nv + nu) per mj_step; B_env = nsub B_sub + 4 (obs + act) + 8"""
    return nsub * 4 * (2 * model.nq + 5 * model.nv + model.nu) + 4 * (obs_dim + act_dim) + 8


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return {"hbm_gbs": 6650.0}, "fallback 6.65 TB/s (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons through NVML while the timed region runs"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        names = {0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost", 0x20: "sw_thermal_slowdown",
                 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
        while not self._halt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._halt.wait(0.05)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def dump_outputs(tensors, out_dir, max_bytes=64 << 20):
    """<out_dir>/<name>.npy of every tensor: floats as float32, the integer and boolean ones as float64 (exact for int32).  Above
    `max_bytes` in all, every array keeps the same fixed, seeded fraction of its rows."""
    import numpy as np

    arrays = {n: t.cpu().numpy() for n, t in tensors.items()}
    arrays = {n: a.astype(np.float32 if a.dtype.kind == "f" else np.float64) for n, a in arrays.items()}
    frac = min(1.0, (max_bytes - 128 * len(arrays)) / sum(a.nbytes for a in arrays.values()))  # 128: an .npy header
    os.makedirs(out_dir, exist_ok=True)
    for n, a in arrays.items():
        if frac < 1.0:
            a = a[np.sort(np.random.RandomState(0).choice(len(a), int(len(a) * frac), replace=False))]
        np.save(os.path.join(out_dir, n + ".npy"), a)


def build_id():
    """identifies the kernel build a profile belongs to: sha256 over the SASS of the stock kernels' cubin (__graft_entry__.sass_id)"""
    import __graft_entry__ as ge

    return ge.sass_id()


def host_cores():
    """cores this process may really use: the affinity mask capped by the cgroup CPU quota (a 128-thread box with
    cpu.max = '1600000 100000' gives 16: running 128 busy processes there measures the scheduler, not the code)"""
    aff = len(os.sched_getaffinity(0))
    quota = None
    try:
        a, b = open("/sys/fs/cgroup/cpu.max").read().split()
        if a != "max":
            quota = float(a) / float(b)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    cores = aff if quota is None else max(1, min(aff, int(quota)))
    return cores, aff, quota


def cpu_env_rate(seconds, seed=0):
    """env-steps/s of the CPU oracle env on ONE core for about `seconds` of work (reset excluded, like fps.py:119-127)"""
    import numpy as np

    from furniture_b200 import mjcf
    from oracle.ref_env import OracleFurnitureEnv

    m = mjcf.load_scene("Sawyer", "table_lack_0825")
    env = OracleFurnitureEnv(m)
    env.reset()
    rng = np.random.RandomState(seed)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        _, _, done, _ = env.step(rng.uniform(-1, 1, env.dof))
        if done:
            env.reset()
        n += 1
    return n / (time.perf_counter() - t0), n


def _ref_worker(idx, nrounds, slice_s, start, finish, counts):
    """one reference env per process (make_vec_env / SubprocVecEnv, env/base.py:55-80): free-running for `slice_s` seconds per
    bench step, so that a bench step is not a barrier on the slowest worker's fixed chunk"""
    import numpy as np

    from furniture_b200 import mjcf
    from oracle.ref_env import OracleFurnitureEnv

    m = mjcf.load_scene("Sawyer", "table_lack_0825")
    env = OracleFurnitureEnv(m)
    env.cfg.seed = 123 + idx
    env.reset()
    rng = np.random.RandomState(idx)
    for r in range(nrounds):
        start.wait()
        n, t_end = 0, time.perf_counter() + slice_s
        while time.perf_counter() < t_end:
            _, _, done, _ = env.step(rng.uniform(-1, 1, env.dof))
            if done:
                env.reset()
            n += 1
        counts[idx] = n
        finish.wait()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp

    for v in ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = "1"  # one thread per env process, as a SubprocVecEnv worker (inherited by the spawned workers)
    cores, aff, quota = host_cores()
    one_core, _ = cpu_env_rate(4.0)
    slice_s = args.ref_slice
    ctx = mp.get_context("spawn")
    start, finish = ctx.Barrier(cores + 1), ctx.Barrier(cores + 1)
    counts = ctx.Array("l", cores)
    W, K = max(args.warmup, 1), args.steps
    procs = [ctx.Process(target=_ref_worker, args=(i, W + K, slice_s, start, finish, counts), daemon=True) for i in range(cores)]
    for p in procs:
        p.start()
    total, dt = 0, 0.0
    for r in range(W + K):
        start.wait()
        t0 = time.perf_counter()
        finish.wait()
        t1 = time.perf_counter()
        if r >= W:
            total += sum(counts[:])
            dt += t1 - t0
    for p in procs:
        p.join(timeout=10)
    value = total / dt
    sample = ("%d processes (affinity %d, cgroup quota %s), one env each, free-running %.1f s per bench step; %d env.step() in %.1f s; "
              "reset excluded" % (cores, aff, "none" if quota is None else "%.1f cpus" % quota, slice_s, total, dt))
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs": cores, "note": "CPU restatement of the reference loop (mujoco-py/MuJoCo 2.0 absent): oracle/ref_env.py over oracle/fe_oracle.c; "
                   "published anchor 225 env-steps/s on one Xeon 6154 core (docs/more_info.md:35)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "per_core": value / cores, "one_core_alone": one_core,
                         "parallel_efficiency": value / cores / one_core},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


def run_ours(args):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, world)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    from furniture_b200.env import BatchedFurnitureEnv, ShardedFurnitureEnv

    n_local = args.envs_per_gpu
    K, W = args.steps, args.warmup

    mixed = None
    if args.furniture == "mixed":  # BASELINE.json config 5: every furniture model of the asset tree the compiler accepts, ragged nv / nefc
        from furniture_b200 import mjcf
        from furniture_b200.env import MixedFurnitureEnv, shard_furniture

        cdir = os.path.join(ROOT, "furniture_b200", "compiled")
        names = sorted(f[len(args.agent) + 1 : -4] for f in os.listdir(cdir) if f.startswith(args.agent + "_") and f.endswith(".npz"))
        models = {n: mjcf.load_scene(args.agent, n) for n in names}
        # the same number of envs of every furniture model; whole buckets per GPU, balanced on the measured cost of the models;
        # ranks then own different numbers of envs and pad their shard to the largest (the all-gather wants equal shards)
        from furniture_b200.env import model_costs

        per_model = max(1, (n_local * world) // len(names))
        owned = shard_furniture(names, per_model, world, nv=[models[n].nv for n in names], cost_per_env=model_costs() or None)
        n_real = [sum(c for _, c in o) for o in owned]
        n_local = max(n_real)
        wide = max(7 * len(models[n].meta["part_names"]) for n in names)
        mixed = {"models": len(names), "per_rank": [len(o) for o in owned], "nv_range": [min(m.nv for m in models.values()), max(m.nv for m in models.values())],
                 "envs_per_model": per_model, "envs_per_rank": n_real, "global_envs": sum(n_real)}

    def make_env():
        # the two timed legs (device-resident `value`, host-buffer `e2e`) run on two envs built alike -- same seeds, same
        # reset draws, same actions, same step range -- so that their numbers are comparable
        if mixed is not None:
            mine = owned[rank]
            e = MixedFurnitureEnv([n for n, _ in mine], [c for _, c in mine], agent=args.agent, device=local, object_ob_dim=wide, pad_to=n_local,
                                  seed=ShardedFurnitureEnv.shard_seed(123, rank, n_local))
            return (ShardedFurnitureEnv(n_local, env=e), e) if world > 1 else (e, e)
        if world > 1:
            e = ShardedFurnitureEnv(n_local, agent=args.agent, furniture_name=args.furniture)
            return e, e.env
        if args.reward == "dense":  # IKEASawyerDense-v0: the phase-based reward inside the step kernel, the dense env's own config
            from furniture_b200.env import split_dense_config

            _, over, dense, _ = split_dense_config(dict(furniture_name=args.furniture, seed=123))
            e = BatchedFurnitureEnv(args.agent, args.furniture, n_local, device=local, dense=dense, control_type=args.control_type, **over)
        else:
            e = BatchedFurnitureEnv(args.agent, args.furniture, n_local, device=local, seed=123, control_type=args.control_type)
        return e, e

    env, benv = make_env()
    env2, benv2 = make_env()
    env.reset()
    env2.reset()
    gen = torch.Generator().manual_seed(1000 + rank)
    a_host = [(torch.rand((n_local, benv.act_dim), generator=gen) * 2 - 1).pin_memory() for _ in range(K + W)]
    if args.actions == "settled":  # SURVEY.md 8d "settled" variant: zero arm action, gripper open, no connect request
        for a in a_host:
            a.zero_()
            a[:, -2:] = -1.0
    acts = [a.to(dev) for a in a_host]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > L2 (126 MB)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- leg 1: device-resident actions, CUDA events per step
    for i in range(W):
        env.step(acts[i])
    barrier()
    if world > 1:
        env.timing = True
    sampler = ClockSampler(local)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for k in range(K):
        flush.fill_(float(k))  # evict L2 between timed iterations (not timed)
        ev[k][0].record()
        last = env.step(acts[W + k])
        ev[k][1].record()
    barrier()
    clocks = sampler.stop()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], device=dev, dtype=torch.float64)
    rank_ms = float(total_ms.item()) / K
    per_rank = None
    if world > 1:
        km, gm = env.pop_timing()
        env.timing = False
        mine = torch.tensor([rank_ms, sum(km) / len(km), sum(gm) / len(gm)], device=dev, dtype=torch.float64)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = [{"rank": r, "step_ms": float(t[0]), "kernel_ms": float(t[1]), "gather_wait_ms": float(t[2])} for r, t in enumerate(allr)]
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    n_global = mixed["global_envs"] if mixed is not None else n_local * world  # padding rows of a mixed batch are not envs
    value = n_global * K / (total_ms * 1e-3)
    # kernels launched by this repo inside the timed region, per step: fe_env_step_kernel + fe_order_kernel (block packing for
    # the next step); N > 1 adds NCCL's all-gather kernel (a library kernel, not counted)
    launches = 2 * K * (len(owned[rank]) if mixed is not None else 1)

    # ---- leg 2: end to end through the public API with HOST buffers, same actions and step range on the twin env:
    # pinned actions -> H2D -> step (-> all_gather) -> D2H of this rank's results
    n_out = n_local
    obs_host = torch.empty((n_out, benv2.obs_dim)).pin_memory()
    rew_host = torch.empty(n_out).pin_memory()
    done_host = torch.empty(n_out, dtype=torch.bool if world > 1 else torch.uint8).pin_memory()
    for i in range(W):
        env2.step(a_host[i])
    barrier()
    e2e_s = 0.0
    for k in range(K):
        flush.fill_(float(k))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        od, rew, done, _ = env2.step(a_host[W + k])
        if world > 1:  # every rank holds the gathered tensors on the device; its host side reads its own shard
            ob_o, ob_r, rew, done = env2.local_slice(od["object_ob"]), env2.local_slice(od["robot_ob"]), env2.local_slice(rew), env2.local_slice(done)
        else:
            ob_o, ob_r = od["object_ob"], od["robot_ob"]
        obs_host[:, : benv2.object_ob_dim].copy_(ob_o, non_blocking=True)
        obs_host[:, benv2.object_ob_dim :].copy_(ob_r, non_blocking=True)
        rew_host.copy_(rew, non_blocking=True)
        done_host.copy_(done, non_blocking=True)
        torch.cuda.synchronize()
        e2e_s += time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e = n_global * K / float(e2e_t.item())
    h2d = n_local * benv.act_dim * 4
    d2h = obs_host.numel() * 4 + rew_host.numel() * 4 + done_host.numel()

    if rank == 0:
        peaks, peak_src = load_peaks()
        kernel_ms = total_ms / K  # one env-step = one launch of fe_env_step_kernel (+ the all_gather when N > 1)
        if mixed is not None:
            benv_bytes = benv.algorithmic_bytes_per_step() / n_local  # this rank's buckets, per row of its (padded) shard
        else:
            benv_bytes = b_env(benv.model, benv.obs_dim, benv.act_dim, nsub=150 if args.control_type == "ik" else 50)  # ik: three _do_simulation per env step
        assert args.furniture != "table_lack_0825" or args.agent != "Sawyer" or args.control_type != "impedance" or args.reward != "sparse" or benv_bytes == B_ENV
        achieved = benv_bytes * n_local / (kernel_ms * 1e-3) / 1e9
        act_txt = "random actions U(-1,1)" if args.actions == "random" else "settled (zero arm action, gripper open)"
        default_case = args.agent == "Sawyer" and args.furniture == "table_lack_0825" and args.actions == "random" and n_local == ENVS_PER_GPU and args.reward == "sparse" and args.control_type == "impedance"
        workload = WORKLOAD if default_case else "Furniture%sEnv + %s, control_type=impedance, 50 mj_steps per env-step, %s" % (args.agent, args.furniture, act_txt)
        if args.reward == "dense":
            workload = "FurnitureSawyerDenseRewardEnv (IKEASawyerDense-v0) + %s, phase-based reward inside the step kernel, episodes of 150 steps, %s" % (args.furniture, act_txt)
        if args.control_type == "ik":
            workload = workload.replace("control_type=impedance, 50 mj_steps per env-step", "control_type=ik (in-kernel inverse kinematics), 3 x 50 mj_steps per env-step") + " [control_type=ik]"
        if mixed is not None:
            workload = ("Furniture%sEnv, mixed-furniture batch: %d furniture models (nv %d..%d) x %d envs each, whole buckets per GPU balanced on measured model cost "
                        "(%s models / %s envs per rank, shards padded to %d rows), one kernel-module instance and stream per bucket, 50 mj_steps per env-step, %s"
                        % (args.agent, mixed["models"], mixed["nv_range"][0], mixed["nv_range"][1], mixed["envs_per_model"], mixed["per_rank"], mixed["envs_per_rank"], n_local, act_txt))
        # measured DRAM traffic and instruction counts come from an ncu capture of exactly this kernel build
        # (tools/ncu_extract.py writes profiles/traffic.json with the build id); a stale capture is refused
        traffic, secondary, prof_note = None, None, None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        bid = build_id()
        if os.path.exists(tp) and default_case:
            prof = json.load(open(tp))
            if prof.get("build_id") == bid:
                traffic = prof.get("dram_bytes_per_launch")
                if prof.get("warp_instructions_per_launch") and clocks.get("sm_mhz"):
                    slots = kernel_ms * 1e-3 * clocks["sm_mhz"] * 1e6 * 148 * 4  # warp-issue slots of the chip during one launch
                    ipc = prof["warp_instructions_per_launch"] / (kernel_ms * 1e-3 * clocks["sm_mhz"] * 1e6 * 148)
                    lanes = prof.get("lanes_active_per_instruction")
                    secondary = {"bound": "fp32-issue", "ipc": ipc, "ipc_peak": 4.0, "lanes_active": lanes,
                                 "frac": prof["warp_instructions_per_launch"] * lanes / 32.0 / slots,
                                 "note": "warp instructions x active lanes of the ncu capture of this build (%s) over the lane-issue slots of the live launch" % prof.get("source", "profiles/")}
            else:
                prof_note = "profiles/traffic.json belongs to build %s, this is build %s: traffic not reported" % (prof.get("build_id"), bid)
        out = {
            "metric": METRIC if default_case else "aggregate env-steps/sec, %s+%s @%d envs/GPU (%s actions)" % (args.agent, args.furniture, n_local, args.actions),
            "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": total_ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "envs_per_gpu": n_local, "global_envs": n_global, "parallelism": "env-shards x%d" % world,
                       "l2": "flushed before every timed step of both legs (256 MiB write, not timed)",
                       "timing": "value: CUDA events per step on the launch stream, max over ranks; e2e: wall clock per step around the public call with "
                                 "host buffers, same actions and step range on a twin env", "build_id": bid},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": traffic,
                         "kernel": "fe_env_step_kernel", "algorithmic_bytes_per_launch": benv_bytes * n_local, "peak_source": peak_src,
                         "note": "state stays in shared memory for the 50 mj_steps of a launch; the path is latency/issue bound, not HBM bound (DESIGN.md)"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": K},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        if secondary:
            out["roofline_secondary"] = secondary
        if prof_note:
            out["roofline"]["traffic_note"] = prof_note
        if per_rank:
            out["per_rank"] = per_rank
        if world == 1 and not args.no_cpu_baseline and default_case:
            for v in ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS"):
                os.environ.setdefault(v, "1")
            v, n = cpu_env_rate(args.cpu_seconds)
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
                                   "sample": "%d env.step() of one CPU oracle env (oracle/ref_env.py over oracle/fe_oracle.c) in %.0f s" % (n, args.cpu_seconds)}
        if args.dump_outputs:  # leg 1's env is not stepped after its timed window: its buffers still hold that window's last step
            od, rew, done, info = last
            dump_outputs(dict(od, reward=rew, done=done, info=info), args.dump_outputs)
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--furniture", default="table_lack_0825", help="other furniture = parity-test configs timed for DESIGN.md, not the bench line")
    ap.add_argument("--agent", default="Sawyer")
    ap.add_argument("--control-type", default="impedance", choices=["impedance", "ik"], help="ik = the reference's default control type: inverse kinematics + 3 x 50 mj_steps "
                    "per env step inside the kernel; one GPU, not the bench line")
    ap.add_argument("--reward", default="sparse", choices=["sparse", "dense"], help="dense = FurnitureSawyerDenseRewardEnv (IKEASawyerDense-v0), one GPU, not the bench line")
    ap.add_argument("--ref-slice", type=float, default=1.0, help="--impl reference: seconds every worker runs free per bench step")
    ap.add_argument("--actions", default="random", choices=["random", "settled"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the observations, rewards, dones and infos of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
