#!/usr/bin/env python
"""Headline benchmark: agent-env-steps/s of the batched rollout hot path.

    python bench.py [--gpus N --steps K --warmup W]            # this engine
    python bench.py --impl reference [...]                      # the CPU path on host cores
    torchrun --nproc-per-node N bench.py --gpus N ...           # one rank per GPU, weak scaling

Headline workload = BASELINE.json configs[1] (MAWaterWorld 5 pursuers / 5 evaders / 10 poison /
30 sensors, 4096 envs per B200).  One bench "step" = one 1024-step horizon of every env in the
batch = 4 rollout launches of 256 lockstep env steps (SURVEY.md 8d times 1000 steps, the env's
`timestep_limit`; 4 x 256 keeps one launch's observation tensor at 4.5 GB).  The same line carries,
under "workloads", short measurements of the other BASELINE configs (Pursuit C3, Waterworld C4 shape
-- at --gpus 8 that is config 4: 32 768 envs over 8 GPUs --, Hostage C5), each with its own roofline
fractions.  Prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WW_CFG = dict(n_pursuers=5, n_evaders=5, n_poison=10, n_sensors=30)   # class defaults otherwise
METRIC = "agent_env_steps_per_sec"
UNIT = "agent-env-steps/s"

PE_C3 = dict(n_evaders=30, n_pursuers=8, obs_range=7, surround=True, n_catch=2, flatten=True,
             reward_mech='local', catchr=0.1, term_pursuit=5.0, sample_maps=True, include_id=True)
HW_C5 = (10, 16, 16, 4, 2)

# name -> the BASELINE.json config it measures; t = lockstep env steps per rollout launch (one
# launch's observation tensor stays around 3-5 GB: larger than L2 by 30x, small next to 180 GB)
WORKLOADS = {
    "waterworld": dict(desc="MAWaterWorld 5p/5e/10po/30 sensors", envs=4096, agents=5, family="ww", cfg=WW_CFG,
                       t=256, kernel="ww_kernel<float,1,1,30>", key="ww_c2"),
    "waterworld_c4": dict(desc="MAWaterWorld 20p/50e/50po/30 sensors", envs=4096, agents=20, family="ww",
                          cfg=dict(n_pursuers=20, n_evaders=50, n_poison=50, n_sensors=30), t=64,
                          kernel="ww_kernel<float,4,1,30>", key="ww_c4"),
    "pursuit": dict(desc="PursuitEvade 16x16 map_pool16, 8p/30e, obs_range 7, surround", envs=65536, agents=8,
                    family="pe", cfg=PE_C3, t=16, kernel="pe_kernel<1,2,7>", key="pe_c3"),
    "hostage": dict(desc="ContinuousHostageWorld 10 rescuers/16 hostages/16 criminals/30 sensors", envs=8192,
                    agents=10, family="hw", cfg=HW_C5, t=64, kernel="hw_kernel<float,1,1,30>", key="hw_c5"),
}
LAUNCHES_PER_STEP = 4


def ww_bytes_per_env_step(Np, Ne, Npo, K):
    """Algorithmic (compulsory) bytes per env-step, SURVEY.md 8(d) / BASELINE.md section 5."""
    return 4 * (8 * (Np + Ne + Npo) + 2 * Np + Np * (7 * K + 3) + Np) + 41


def bytes_per_env_step(wl):
    """Algorithmic (compulsory) bytes per env-step, SURVEY.md 8(d)."""
    w = WORKLOADS[wl]
    if w["family"] == "ww":
        c = w["cfg"]
        return ww_bytes_per_env_step(c["n_pursuers"], c["n_evaders"], c["n_poison"], c["n_sensors"])
    if w["family"] == "pe":
        Np, Ne, R = 8, 30, 7
        return 2 * (2 * Np + 2 * Ne + (Ne + 7) // 8 + 1 + 8) + 4 * Np + 4 * Np * (3 * R * R + 1) + 4 * Np + 1 + 4
    Nr, Nh, Nc, K = 10, 16, 16, 30
    return 4 * (2 * 4 * Nr + 2 * 4 * Nc + 2 * Nh + 4) + 2 * ((Nh + 7) // 8 + 12 + 8) + 4 * 2 * Nr + \
        4 * Nr * (5 * K + 6) + 4 * Nr + 9


def make_engine(wl, E, dev, rank):
    from madrl_b200 import BatchedHostageWorld, BatchedMAWaterWorld, BatchedPursuitEvade
    w = WORKLOADS[wl]
    if w["family"] == "ww":
        return BatchedMAWaterWorld(E, device=dev, seed=0, env_id_base=rank * E, **w["cfg"])
    if w["family"] == "pe":
        maps = np.load(os.path.join(ROOT, "maps", "map_pool16.npy"))
        return BatchedPursuitEvade(E, maps, device=dev, seed=0, env_id_base=rank * E, max_path_length=500, **w["cfg"])
    return BatchedHostageWorld(E, *w["cfg"], device=dev, seed=0, env_id_base=rank * E)


def act_spec(wl):
    """(per-step action shape after [T, E], torch dtype name)"""
    w = WORKLOADS[wl]
    return ((w["agents"],), "int32") if w["family"] == "pe" else ((w["agents"], 2), "float32")


def make_actions(wl, T, E, dev, g, host=False):
    import torch
    w = WORKLOADS[wl]
    d = "cpu" if host else dev
    gg = None if host else g
    if w["family"] == "pe":
        return torch.randint(0, 5, (T, E, w["agents"]), dtype=torch.int32, device=d, generator=gg)
    return torch.randn(T, E, w["agents"], 2, device=d, generator=gg) * 0.5


def make_oracle(wl, seed):
    from oracle.philox import Stream
    w = WORKLOADS[wl]
    if w["family"] == "ww":
        from oracle.waterworld_oracle import WaterworldOracle
        return WaterworldOracle(rng=Stream(seed, seed), **w["cfg"])
    if w["family"] == "pe":
        from oracle.pursuit_oracle import PursuitOracle
        maps = np.load(os.path.join(ROOT, "maps", "map_pool16.npy"))
        return PursuitOracle(maps, rng=Stream(seed, seed), **w["cfg"])
    from oracle.hostage_oracle import HostageOracle
    return HostageOracle(*w["cfg"], rng=Stream(seed, seed))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def measured_traffic():
    """DRAM bytes per env-step of each kernel from the committed ncu captures
    (profiles/r2_traffic.json, written by scripts/ncu_traffic.py from `ncu --set full`:
    dram__bytes_read.sum + dram__bytes_write.sum per launch / env-steps per launch).  Only trusted
    for the binary it was captured on: the file records the source hash of that build."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        from madrl_b200.build import kernel_hash
        d = json.load(open(p))["kernels"]
        return {k: v for k, v in d.items() if v.get("kernel_hash") == kernel_hash(k.split("_")[0])}
    except Exception:
        return {}


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled DURING the timed region (NVML, ~1 ms per sample;
    nvidia-smi polling as the fallback)."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.mode = index, [], False, "nvml"
        self.sm_max = None
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[index])
                except Exception:
                    idx = index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.mode = "nvidia-smi"

    def run(self):
        if self.mode == "nvml":
            nv = self.nv
            while not self.stop_flag:
                try:
                    self.samples.append((float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)),
                                         int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                                         if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons")
                                         else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))))
                except Exception:
                    pass
                time.sleep(0.002)
            return
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip().split(",")
                self.sm_max = float(out[1])
                self.samples.append((float(out[0]), int(out[2].strip(), 16)))
            except Exception:
                pass
            time.sleep(0.02)

    def window(self, t0, t1):
        pass

    def summary(self, note):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["unavailable"], "window": note}
        sm = sorted(s[0] for s in self.samples)
        bits = 0
        for s in self.samples:
            bits |= s[1]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.sm_max,
                "reasons": [n for n, b in self.REASONS if bits & b], "samples": len(self.samples),
                "source": self.mode, "window": note}


# ----------------------------------------------------------------------------- CPU baseline
def _cpu_worker(args):
    seconds, seed, wl = args
    w = WORKLOADS[wl]
    env = make_oracle(wl, seed)
    env.reset()
    rs = np.random.RandomState(seed)
    if w["family"] == "pe":
        acts = rs.randint(0, 5, size=(4096, w["agents"]))
    else:
        acts = rs.randn(4096, w["agents"] * 2) * 0.5
    for i in range(50):
        env.step(acts[i])
    n, last_reset, t0 = 0, 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        _, _, done, _ = env.step(acts[n % 4096])
        n += 1
        if done or n - last_reset >= 500:
            env.reset()
            last_reset = n
    return n, time.perf_counter() - t0


def cpu_baseline(seconds, procs, wl="waterworld"):
    """The CPU path (float64 NumPy oracle port of the reference step(), one env per process the
    way rllab's StatefulPool parallelises; rllab/rllab/sampler/stateful_pool.py:102-157)."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        res = pool.map(_cpu_worker, [(seconds, 100 + i, wl) for i in range(procs)])
    env_steps_per_s = sum(n / dt for n, dt in res)
    return env_steps_per_s * WORKLOADS[wl]["agents"]


# ----------------------------------------------------------------------------- NUMA placement
def bind_to_gpu_numa(dev_index):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off BEFORE the pinned staging
    buffers are allocated, so device->host traffic lands in local DRAM (at N = 8 the round-1 e2e fell
    from 62 to 45 M agent-steps/s per GPU with every rank's buffers wherever the launcher ran)."""
    try:
        import torch
        p = torch.cuda.get_device_properties(dev_index)
        bus = "%04x:%02x:%02x.0" % (getattr(p, "pci_domain_id", 0), p.pci_bus_id, p.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


# ----------------------------------------------------------------------------- device-resident run
class Runner(object):
    """One workload on this rank's GPU: engine, output buffers, optional per-rollout exchange."""

    def __init__(self, wl, E, T, dev, rank, world, exchange, n_act):
        import torch
        self.torch, self.wl, self.E, self.T, self.dev, self.rank, self.world = torch, wl, E, T, dev, rank, world
        self.W = WORKLOADS[wl]
        self.Np = self.W["agents"]
        self.eng = make_engine(wl, E, dev, rank)
        self.D = self.eng.obs_dim
        self.eng.reset()
        g = torch.Generator(device=dev)
        g.manual_seed(1234 + rank)
        # synthetic actions 0.5*N(0,1) (waterworld.py:486) / uniform {0..4}; a different tensor per launch
        self.actions = [make_actions(wl, T, E, dev, g) for _ in range(n_act)]
        self.info_w = 1 if self.W["family"] == "pe" else 2
        from madrl_b200.dist import AsyncRootGather, PackedTrajectory
        self.mode, self.note, self.agather = ("none" if world == 1 else exchange), None, None
        if world > 1 and self.mode in ("overlap", "overlap-nccl"):
            try:   # agrees on success across ranks internally and raises on ALL ranks
                self.agather = AsyncRootGather(T, E, self.Np, self.info_w, dev,
                                               completion="auto" if self.mode == "overlap" else "nccl")
                self.completion = self.agather.completion
            except Exception as ex:   # e.g. no peer access between the GPUs of this box
                self.mode, self.note = "nccl", "overlap unavailable (%s)" % type(ex).__name__
        self.packed = PackedTrajectory(T, E, self.Np, self.info_w, dev)
        self.obs_buf = torch.empty((T, E, self.Np, self.D), device=dev)
        self.k = 0

    def rollout(self, i):
        k = self.k
        self.k += 1
        a = self.actions[i % len(self.actions)]
        if self.agather is not None:
            self.agather.before_reuse(k)
            rew_b, done_b, info_b = self.agather.buffers(k)
            self.eng.rollout(a, auto_reset=True, out=(self.obs_buf, rew_b, done_b, info_b))
        else:
            self.eng.rollout(a, auto_reset=True, out=(self.obs_buf, self.packed.rew, self.packed.done, self.packed.info))
        return k

    def exchange(self, k):
        if self.world > 1:
            if self.agather is not None:
                self.agather.submit(k)
            elif self.mode == "nccl":
                self.packed.gather_raw()

    def drain(self):
        if self.agather is not None:   # the timed region ends when the last exchange has landed
            self.torch.cuda.current_stream(self.dev).wait_stream(self.agather.comm)

    def verify_exchange(self):
        """Driver-visible proof of the default multi-GPU data plane: for two rollouts (both buffer
        sets) the root's gathered buffer must equal a plain NCCL all_gather of the ranks' packed
        buffers.  Returns 1.0 / 0.0 (agreed over ranks by the caller)."""
        import torch.distributed as dist
        torch = self.torch
        ok = True
        for _ in range(3):
            k = self.rollout(self.k)
            self.exchange(k)
            self.drain()
            torch.cuda.synchronize()
            if self.agather is not None:
                local = self.agather.packed(k).buf
                ref = torch.empty(self.world * local.numel(), dtype=torch.uint8, device=self.dev)
                dist.all_gather_into_tensor(ref, local)
                got = self.agather.result(k)
                if got is not None:
                    ok = ok and bool(torch.equal(got.reshape(-1), ref))
        return 1.0 if ok else 0.0

    def close(self):
        if self.agather is not None:
            self.agather.close()
        self.agather = None
        del self.eng, self.actions, self.obs_buf, self.packed
        self.torch.cuda.empty_cache()


def time_runner(r, steps, warmup, sampler=None):
    """W warm-up steps, then `steps` bench steps (= LAUNCHES_PER_STEP rollout launches each) between
    barrier + synchronize; device time, max over ranks.  Returns (ms_total, kernel_ms, launches)."""
    import torch
    import torch.distributed as dist
    from madrl_b200 import launch_count

    def barrier():
        if r.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(warmup * LAUNCHES_PER_STEP):
        r.exchange(r.rollout(i))
    r.drain()
    barrier()
    n = steps * LAUNCHES_PER_STEP
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    l0 = launch_count()
    if sampler:
        sampler.start()
    barrier()
    ev0.record()
    for i in range(n):
        kev[i][0].record()
        k_ = r.rollout(i)
        kev[i][1].record()
        r.exchange(k_)
    r.drain()
    ev1.record()
    barrier()
    if sampler:
        sampler.stop_flag = True
    launches = launch_count() - l0
    ms = ev0.elapsed_time(ev1)
    kern_ms = float(np.mean([s.elapsed_time(e) for s, e in kev]))
    r.kernel_ms_per_rank = [kern_ms]
    if r.world > 1:
        per = torch.zeros(r.world, device=r.dev)
        dist.all_gather_into_tensor(per, torch.tensor([kern_ms], device=r.dev))
        r.kernel_ms_per_rank = [float(x) for x in per.tolist()]
        t = torch.tensor([ms, kern_ms], device=r.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, kern_ms = float(t[0].item()), float(t[1].item())
    return ms, kern_ms, launches


def dump_outputs(r, d, budget=60 << 20):
    """Writes what the last rollout returned to its caller (obs, rew, done, info: [T, E, ...]) as d/<name>.npy,
    float32 (info: float64), for a fixed seeded sample of the envs that keeps the data within `budget` bytes;
    d/env_ids.npy lists the sampled envs.  Engine seeds and actions are fixed, so the same arguments give the
    same inputs on every run and two builds can be compared output for output."""
    torch = r.torch
    last = r.agather.buffers(r.k - 1) if r.agather is not None else (r.packed.rew, r.packed.done, r.packed.info)
    outs = dict(zip(("obs", "rew", "done", "info"), (r.obs_buf,) + tuple(last)))
    dtypes = {k: np.float64 if k == "info" else np.float32 for k in outs}
    per_env = sum(x[:, 0].numel() * np.dtype(dtypes[k]).itemsize for k, x in outs.items())
    n = max(1, min(r.E, budget // per_env))
    ids = np.sort(np.random.RandomState(0).choice(r.E, n, replace=False))
    idx = torch.as_tensor(ids, device=r.dev)
    torch.cuda.synchronize()
    os.makedirs(d, exist_ok=True)
    for k, x in outs.items():
        np.save(os.path.join(d, k + ".npy"), x.index_select(1, idx).cpu().numpy().astype(dtypes[k]))
    np.save(os.path.join(d, "env_ids.npy"), ids.astype(np.float64))


def roofline_of(wl, E, T, kern_ms):
    bpe = bytes_per_env_step(wl)
    peak, peak_kind = measured_peak_gbs()
    achieved = bpe * E * T / (kern_ms * 1e-3) / 1e9
    key = WORKLOADS[wl]["key"]
    dram = measured_traffic().get(key, {}).get("dram_bytes_per_env_step")
    out = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
           "peak_kind": peak_kind, "kernel": WORKLOADS[wl]["kernel"], "kernel_ms": kern_ms,
           "algorithmic_bytes_per_env_step": bpe,
           # bytes DRAM actually moved (ncu dram__bytes_read.sum + dram__bytes_write.sum of the same
           # kernel and launch shape, profiles/r2_traffic.json), scaled to this launch; null when
           # the capture belongs to another build of the library
           "traffic": (dram * E * T) if dram else None,
           "traffic_unit": "bytes per launch (algorithmic: %d)" % (bpe * E * T),
           "frac_dram": (dram * E * T / (kern_ms * 1e-3) / 1e9 / peak) if dram else None,
           "dram_bytes_per_env_step": dram}
    if dram is None:
        out["traffic_note"] = "no ncu capture of this kernel's current source in profiles/r2_traffic.json"
    return out


def e2e_of(r, steps, obs_last):
    """The same rollout through the host-buffer C-ABI entry point with pinned host tensors: H2D of the
    actions and D2H of the results inside the timed region (wall clock around the blocking calls)."""
    import torch
    import torch.distributed as dist
    E, Np, D, T = r.E, r.Np, r.D, r.T
    Te = max(1, min(T, (1 << 30) // (E * Np * D * 4))) if not obs_last else T    # <= 1 GB of obs per call
    h_act = [make_actions(r.wl, Te, E, r.dev, None, host=True).pin_memory() for _ in range(2)]
    h_out = (torch.empty((E, Np, D) if obs_last else (Te, E, Np, D)).pin_memory(), torch.empty((Te, E, Np)).pin_memory(),
             torch.empty((Te, E), dtype=torch.uint8).pin_memory(),
             torch.empty((Te, E, 2) if r.info_w == 2 else (Te, E), dtype=torch.int32).pin_memory())
    for i in range(2):
        r.eng.rollout_host(h_act[i % 2], *h_out, obs_last=obs_last)
    if r.world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    n = max(3, min(steps, 10))
    t0 = time.perf_counter()
    for i in range(n):
        r.eng.rollout_host(h_act[i % 2], *h_out, obs_last=obs_last)     # returns after results are in host memory
    dt = time.perf_counter() - t0
    if r.world > 1:
        t = torch.tensor([dt], device=r.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    h2d = int(h_act[0].numel() * h_act[0].element_size())
    d2h = int(sum(x.numel() * x.element_size() for x in h_out))
    fam = {"ww": "ww", "pe": "pursuit", "hw": "hostage"}[r.W["family"]]
    return {"value": r.world * E * Np * Te * n / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "t_inner": Te, "pcie_gbs": (h2d + d2h) * n / dt / 1e9,
            "api": "madrl_%s_rollout_host2%s (pinned host buffers, chunked copy/compute overlap)"
                   % (fam, ", MADRL_HOST_OBS_LAST" if obs_last else "")}


def closed_loop_of(r, steps):
    """Closed-loop rollouts with the reference's hand-written policy evaluated INSIDE the rollout kernel
    (madrl_ww_rollout_heuristic / madrl_pursuit_rollout_heuristic through the Batched* classes): no action
    tensor exists at all; per rollout the actions taken, rewards, dones and infos are copied to pinned host
    memory inside the timed region (what a learner on the host consumes), the observations stay in HBM."""
    import torch
    import torch.distributed as dist
    if not hasattr(r.eng, "rollout_heuristic"):
        return None
    E, Np, T = r.E, r.Np, r.T
    obs0 = r.eng.reset()
    out = (r.obs_buf, r.packed.rew, r.packed.done, r.packed.info)
    shp, dt_name = act_spec(r.wl)
    act_buf = torch.empty((T, E) + shp, dtype=getattr(torch, dt_name), device=r.dev)
    host = None

    def one(obs_prev):
        # copies on the same stream as the rollouts: issuing them on a side stream, double-buffered against the next
        # rollout, was measured and is SLOWER (1.2-1.6 vs 1.8 G agent-env-steps/s on the B200 box), so the
        # learner-side transfer is simply serialised here
        nonlocal host
        act, obs, rew, done, info = r.eng.rollout_heuristic(T, obs_prev, auto_reset=True, out=out, actions_out=act_buf)
        if host is None:
            host = [torch.empty(x.shape, dtype=x.dtype).pin_memory() for x in (act, rew, done, info)]
        for h, x in zip(host, (act, rew, done, info)):
            h.copy_(x, non_blocking=True)
        return obs[-1]
    prev = obs0
    for _ in range(2):
        prev = one(prev)
    if r.world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    n = max(3, min(steps, 10))
    t0 = time.perf_counter()
    for _ in range(n):
        prev = one(prev)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if r.world > 1:
        t = torch.tensor([dt], device=r.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    d2h = int(sum(h.numel() * h.element_size() for h in host))
    return {"value": r.world * E * Np * T * n / dt, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": d2h,
            "t_inner": T, "api": "Batched%s.rollout_heuristic (policy of heuristics/%s.py in the rollout kernel; actions, "
                                 "rewards, dones, infos copied to pinned host memory per rollout)"
                                 % ({"ww": "MAWaterWorld", "pe": "PursuitEvade"}[r.W["family"]],
                                    {"ww": "waterworld", "pe": "pursuit"}[r.W["family"]])}


def pcie_d2h_gbs(dev):
    """Live pinned device->host copy rate of this box (the ceiling of the full-observation e2e)."""
    import torch
    src = torch.empty(1 << 29, dtype=torch.uint8, device=dev)
    dst = torch.empty(1 << 29, dtype=torch.uint8).pin_memory()
    dst.copy_(src)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    return 3 * (1 << 29) / (time.perf_counter() - t0) / 1e9


# ----------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="waterworld", choices=sorted(WORKLOADS),
                    help="headline workload (default = BASELINE.json configs[1])")
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (weak scaling); 0 = the config's")
    ap.add_argument("--t-inner", type=int, default=0, help="lockstep env steps per rollout launch (0 = the config's)")
    ap.add_argument("--cpu-seconds", type=float, default=8.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--exchange", default="overlap", choices=["overlap", "overlap-nccl", "nccl", "none"],
                    help="multi-GPU per-rollout exchange of rewards / dones / infos (see DESIGN.md 7)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed rollout (rank 0) as DIR/<name>.npy, at most 64 MB")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    WL = WORKLOADS[a.workload]
    E = a.envs if a.envs > 0 else WL["envs"]
    T = a.t_inner if a.t_inner > 0 else WL["t"]
    host_cores = os.cpu_count() or 1
    warmup = max(3, a.warmup)

    if a.impl == "reference":
        if rank != 0:
            return
        procs = host_cores
        per = max(2.0, min(10.0, 60.0 / max(1, a.steps + a.warmup)))
        for _ in range(a.warmup):
            cpu_baseline(0.5, procs, a.workload)
        t0 = time.perf_counter()
        vals = [cpu_baseline(per, procs, a.workload) for _ in range(a.steps)]
        dt = time.perf_counter() - t0
        v = float(np.mean(vals))
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * dt / a.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": WL["desc"] + ", one env per host process", "envs_per_gpu": E},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": procs, "kind": "port",
                             "sample": "%d processes x %.1f s of step() per bench step, float64 NumPy "
                                       "oracle port of the reference step() (the reference tree cannot "
                                       "travel to the GPU box)" % (procs, per)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- headline: device-resident rollouts -------------------------------------------------------
    r = Runner(a.workload, E, T, dev, rank, world, a.exchange, n_act=4)
    exchange_ok = None
    if world > 1 and r.agather is not None:
        v = torch.tensor([r.verify_exchange()], device=dev)
        dist.all_reduce(v, op=dist.ReduceOp.MIN)
        exchange_ok = bool(v.item() == 1.0)
        if not exchange_ok:
            if rank == 0:
                sys.stderr.write("bench.py: the per-rollout exchange does not reproduce an NCCL all_gather\n")
            dist.destroy_process_group()
            sys.exit(3)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms, kern_ms, launches = time_runner(r, a.steps, warmup, sampler)
    if sampler:
        sampler.join(timeout=2)
    if a.dump_outputs and rank == 0:
        dump_outputs(r, a.dump_outputs)
    agent_steps_per_step = world * E * WL["agents"] * T * LAUNCHES_PER_STEP
    value = agent_steps_per_step * a.steps / (ms * 1e-3)
    mode, note, completion = r.mode, r.note, getattr(r, "completion", None)
    # where a multi-GPU run loses time: the rollout kernel's mean duration on every rank with the per-rollout
    # exchange running behind it, and again with the exchange switched off (same engines, same actions)
    probe = None
    if world > 1:
        probe = {"kernel_ms_per_rank": r.kernel_ms_per_rank}
        keep = (r.agather, r.mode, r.k)
        r.agather, r.mode = None, "none"
        time_runner(r, 5, 1)
        probe["kernel_ms_per_rank_no_exchange"] = r.kernel_ms_per_rank
        r.agather, r.mode, r.k = keep          # the exchange's sequence numbers continue where they stopped
        probe["note"] = ("mean rollout-kernel duration per rank (CUDA events around each launch); `value` uses the "
                         "max over ranks, so rank-to-rank spread of the GPUs costs efficiency even without an exchange")

    # ---- e2e through the host-buffer C ABI ----------------------------------------------------------
    e2e = None
    if not a.no_e2e:
        e2e = e2e_of(r, a.steps, obs_last=False)
        lite = e2e_of(r, a.steps, obs_last=True)
        if rank == 0:
            pcie = pcie_d2h_gbs(dev)
            e2e.update(pcie_peak_gbs=pcie, frac_of_pcie=e2e["pcie_gbs"] / pcie, numa_node=numa,
                       pcie_note="peak = pinned 512 MB device->host copies measured in this run")
        e2e["policy_on_device"] = dict(lite, note="MADRL_HOST_OBS_LAST: rewards / dones / infos of every step + "
                                       "the last observations return to the host; the per-step observations "
                                       "stay in HBM for a policy that runs on the GPU")
        cl = closed_loop_of(r, a.steps)
        if cl is not None:
            e2e["closed_loop_heuristic"] = cl
    r.close()

    # ---- the other BASELINE configs, short (5 steps each) ------------------------------------------
    extra = {}
    if not a.no_extra:
        for wl in ("pursuit", "waterworld_c4", "hostage"):
            if wl == a.workload:
                continue
            w = WORKLOADS[wl]
            rr = Runner(wl, w["envs"], w["t"], dev, rank, world, a.exchange, n_act=2)
            xms, xk, xl = time_runner(rr, 5, 3)
            rec = {"config": "%s, %d envs per GPU, %d lockstep env steps per launch" % (w["desc"], w["envs"], w["t"]),
                   "value": world * w["envs"] * w["agents"] * w["t"] * LAUNCHES_PER_STEP * 5 / (xms * 1e-3), "unit": UNIT,
                   "steps": 5, "ms_per_step": xms / 5, "gpu_launches": int(xl),
                   "roofline": roofline_of(wl, w["envs"], w["t"], xk)}
            if not a.no_e2e and world == 1:
                rec["e2e"] = e2e_of(rr, 3, obs_last=False)
            extra[{"pursuit": "pursuit_c3", "waterworld_c4": "waterworld_c4", "hostage": "hostage_c5"}[wl]] = rec
            rr.close()

    # ---- full-trajectory gather (obs + actions + rewards + dones + infos), one NCCL all_gather -----
    full = None
    if world > 1:
        from madrl_b200.dist import PackedTrajectory
        Tf = 32
        eng = make_engine(a.workload, E, dev, rank)
        eng.reset()
        shp, dt_name = act_spec(a.workload)
        pk = PackedTrajectory(Tf, E, WL["agents"], 1 if WL["family"] == "pe" else 2, dev, obs_dim=eng.obs_dim,
                              act_shape=shp, act_dtype=getattr(torch, dt_name))
        g = torch.Generator(device=dev)
        g.manual_seed(99 + rank)
        pk.act.copy_(make_actions(a.workload, Tf, E, dev, g))
        gbuf = torch.empty(world * pk.nbytes, dtype=torch.uint8, device=dev)
        for _ in range(2):
            eng.rollout(pk.act, auto_reset=True, out=(pk.obs, pk.rew, pk.done, pk.info))
            dist.all_gather_into_tensor(gbuf, pk.buf)
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        nf = 5
        for _ in range(nf):
            eng.rollout(pk.act, auto_reset=True, out=(pk.obs, pk.rew, pk.done, pk.info))
            dist.all_gather_into_tensor(gbuf, pk.buf)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        fms = float(t.item()) / nf
        ingress = (world - 1) * pk.nbytes / (fms * 1e-3) / 1e9
        full = {"value": world * E * WL["agents"] * Tf / (fms * 1e-3), "unit": UNIT, "ms_per_rollout": fms,
                "bytes_per_rank": pk.nbytes, "nvlink_ingress_gbs_per_gpu": ingress,
                "frac_of_nvlink": ingress / 770.0,
                "note": "ONE NCCL all_gather per rollout of the packed [obs | actions | rewards | dones | infos] "
                        "buffer (%d lockstep steps); every rank ends with the whole trajectory.  Bound by the "
                        "NVLink ingress of each GPU (measured peer-copy reference 770 GB/s per direction): "
                        "4 3xx bytes of observations per env-step x (N-1) ranks" % Tf}
        del eng, pk, gbuf
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": warmup, "ms_per_step": ms / a.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": ("u8/int32 + f32 obs" if WL["family"] == "pe" else "f32"),
        "data": "synthetic",
        "config": {"workload": WL["desc"] + ", %d envs per GPU; one bench step = %d rollout launches of %d lockstep "
                               "env steps (a %d-step horizon of every env), auto-reset (VecEnvExecutor semantics)"
                               % (E, LAUNCHES_PER_STEP, T, LAUNCHES_PER_STEP * T),
                   "envs_per_gpu": E, "t_inner": T, "launches_per_step": LAUNCHES_PER_STEP,
                   "actions": ("uniform {0..4}" if WL["family"] == "pe" else "0.5*N(0,1)") + ", HBM-resident",
                   "l2": "outputs per launch (%.0f MB) exceed L2" % (T * E * WL["agents"] * 4 * (1 + 213) / 1e6),
                   "parallelism": "env-shard x%d" % world,
                   "gather": {"none": "none",
                              "overlap": "packed rew/done/info copied to rank 0 over NVLink by the copy engines on "
                                         "a side stream, overlapped with the next rollout; completion + buffer "
                                         "release by stream memory operations on mailbox words (no SM, no "
                                         "collective kernel)",
                              "overlap-nccl": "as overlap, completion by a 4-byte NCCL all-reduce per rollout",
                              "nccl": "one packed NCCL all_gather of rew/done/info per rollout"}[mode]
                             + (" [completion: %s]" % completion if completion else "")
                             + (" [%s]" % note if note else ""),
                   "exchange_verified": exchange_ok},
        "roofline": roofline_of(a.workload, E, T, kern_ms),
        "gpu_launches": int(launches),
        "clocks": sampler.summary("sampled every ~2 ms between the barriers of the timed region") if sampler else None,
    }
    if e2e:
        line["e2e"] = e2e
    if extra:
        line["workloads"] = extra
    if full:
        line["full_gather"] = full
    if probe:
        line["scaling_probe"] = probe
    if world == 1 and not a.no_cpu:
        procs = host_cores
        v = cpu_baseline(a.cpu_seconds, procs, a.workload)
        v1 = cpu_baseline(min(4.0, a.cpu_seconds), 1, a.workload)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": procs, "kind": "port",
                                "single_core_value": v1,
                                "sample": "%d processes x %.0f s of step() (one env each), float64 NumPy "
                                          "oracle port of the reference step()" % (procs, a.cpu_seconds)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
