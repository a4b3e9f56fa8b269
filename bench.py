#!/usr/bin/env python
"""Benchmark of the search-and-target hot path (BASELINE.json metric: MCTS node expansions/sec).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
  python bench.py --impl reference [--gpus N] [--steps K] ...    # the reference's CPU path (port)

A "step" is one move for every game: initial_inference + root expansion + Dirichlet noise +
num_simulations x (descent -> batched recurrent_inference -> expand + backup) + root statistics +
action selection (the body of Actor.play_game, actors.py:131-153).  Workload (configs[3] of
BASELINE.json, "C4"): 18 actions, 4096 games x 50 simulations per GPU, FCNetwork(128 -> 50),
synthetic observations, random-init weights.

Prints ONE JSON line on rank 0.  See DESIGN.md section "Measurement" for how every field is defined.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
  sys.path.insert(0, REPO)

METRIC = "mcts_node_expansions_per_sec"
UNIT = "expansions/s"


def FC_FLOPS_PER_EXPANSION(A):
  """2 * MACs of FCNetwork.recurrent_inference (SURVEY.md section 8 a9): 0.375 MFLOP for A=18."""
  return 2 * (2 * (50 + A) * 512 + 512 * 31 + 512 * 50 + 2 * 50 * 512 + 512 * 31 + 512 * A)


def parse():
  p = argparse.ArgumentParser()
  p.add_argument("--gpus", type=int, default=1)
  p.add_argument("--steps", type=int, default=200)  # ~0.2 s of timed moves: enough NVML clock samples under load
  p.add_argument("--warmup", type=int, default=5)
  p.add_argument("--impl", choices=["b200", "reference"], default="b200")
  p.add_argument("--games", type=int, default=4096, help="concurrent games per GPU")
  p.add_argument("--sims", type=int, default=50)
  p.add_argument("--actions", type=int, default=18)
  p.add_argument("--obs-dim", type=int, default=128)
  p.add_argument("--cpu-baseline-seconds", type=float, default=12.0)
  p.add_argument("--no-cpu-baseline", action="store_true")
  p.add_argument("--no-graph", action="store_true")
  p.add_argument("--streams", type=int, default=4,
                 help="game slices run on separate CUDA streams inside the move graph")
  p.add_argument("--precision", choices=["bf16", "f32", "tf32x3"], default="bf16",
                 help="network kernel: bf16 tcgen05 tensor cores (default), float32 CUDA cores, or float32 accuracy on "
                      "the tensor cores (three TF32 products per multiply)")
  p.add_argument("--wide-step-max-games", type=int, default=None,
                 help="diagnostics: mz_tree_set_wide_step_max_games (trees with <= 16 actions)")
  p.add_argument("--no-conv", action="store_true", help="skip the C5 MuZeroNetwork section")
  p.add_argument("--no-sweep", action="store_true", help="skip the larger-batch throughput probe")
  p.add_argument("--conv-games", type=int, default=4096, help="C5: concurrent games per GPU")
  p.add_argument("--fused", choices=["auto", "0", "1"], default="auto",
                 help="1: the whole move in one persistent kernel (mz_fc_search); 0: one tree + one network launch per "
                      "simulation; auto: FCSearch's default (MZ_FUSED in the environment)")
  p.add_argument("--no-f32", action="store_true", help="skip the float32-network throughput line")
  p.add_argument("--no-selfplay", action="store_true", help="skip the self-play driver section")
  p.add_argument("--no-concurrent", action="store_true", help="skip the search + concurrent learner section")
  p.add_argument("--ref-moves-per-step", type=int, default=2,
                 help="reference arm: moves each worker plays per step")
  p.add_argument("--dump-outputs", metavar="DIR", default=None,
                 help="after the timed steps, write what the last timed move returned for rank 0's games (actions, "
                      "root_value, child_visits, init_value) as DIR/<name>.npy, to compare two builds output for output")
  args = p.parse_args()
  if args.dump_outputs is not None and args.impl != "b200":
    p.error("--dump-outputs needs --impl b200")
  return args


def search_config(args):
  import types
  return types.SimpleNamespace(
      num_simulations=args.sims, action_space=args.actions, two_players=False, discount=0.997,
      pb_c_base=19652, pb_c_init=1.25, init_value_score=0.0, known_bounds=[None, None],
      root_dirichlet_alpha=0.25, root_exploration_fraction=0.25, value_support=[-15, 15],
      reward_support=[-15, 15], no_support=False, no_target_transform=False)


def synthetic_inputs(args, rank, games, as_bytes=False):
  """Observations are `obs_dim` bytes per game (Breakout-ram style, README.md:56); the float32 form is
  the reference's `--obs_range 0 255 --norm_obs` normalisation of the same bytes."""
  rng = np.random.default_rng(1234 + rank)
  obs = rng.integers(0, 256, size=(games, args.obs_dim)).astype(np.uint8)
  if not as_bytes:
    obs = obs.astype(np.float32) / np.float32(255.0)
  noise = rng.dirichlet([0.25] * args.actions, size=games)
  uniforms = rng.random(games)
  temperature = np.ones(games)
  return obs, noise, uniforms, temperature


# ------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the pure-Python port of the reference path (oracle/search_ref.py)
# ------------------------------------------------------------------------------------------------
_WORKER_STATE = {}


def _cpu_worker(job):
  """Plays moves of independent games with the python port until the deadline / move budget.  The network,
  its weights and the search object live as long as the worker process (an Actor builds them once,
  actors.py:29-47), so a timed step measures moves only."""
  (wid, args_d, seconds, max_moves) = job
  key = (args_d["actions"], args_d["sims"], args_d["obs_dim"])
  if key not in _WORKER_STATE:
    os.environ["OMP_NUM_THREADS"] = "1"  # train.py:63
    import torch
    torch.set_num_threads(1)
    from oracle.fcnet_ref import FCNetworkRef, random_state_dict
    from oracle.search_ref import FlatSearch
    A, S, D = key
    net = FCNetworkRef(D, A)
    net.load_state_dict(random_state_dict(D, A))
    _WORKER_STATE[key] = (net, FlatSearch(S, A), np.random.default_rng(99 + wid + 1000 * os.getpid()))
  import torch
  from oracle.search_ref import play_move
  A, S, D = key
  net, search, rng = _WORKER_STATE[key]
  moves, t0 = 0, time.perf_counter()
  with torch.inference_mode():
    while True:
      obs = (rng.integers(0, 256, size=D).astype(np.float32) / 255.0)
      play_move(search, net, obs, rng.dirichlet([0.25] * A), 1.0, rng.random())
      moves += 1
      if max_moves is not None and moves >= max_moves:
        break
      if max_moves is None and time.perf_counter() - t0 >= seconds:
        break
  return moves, time.perf_counter() - t0


def host_cores():
  try:
    return len(os.sched_getaffinity(0))
  except AttributeError:
    return os.cpu_count() or 1


def run_cpu_port(args, seconds=None, moves_per_worker=None, pool=None, cores=None):
  """Returns (expansions/s aggregate, cores, moves, elapsed) for one bounded sample."""
  import multiprocessing as mp
  cores = cores or host_cores()
  args_d = dict(actions=args.actions, sims=args.sims, obs_dim=args.obs_dim)
  jobs = [(w, args_d, seconds, moves_per_worker) for w in range(cores)]
  own = pool is None
  if own:
    pool = mp.get_context("fork").Pool(cores)
  t0 = time.perf_counter()
  res = pool.map(_cpu_worker, jobs)
  elapsed = time.perf_counter() - t0
  if own:
    pool.close()
    pool.join()
  moves = sum(r[0] for r in res)
  return moves * args.sims / elapsed, cores, moves, elapsed


def run_reference(args):
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  import multiprocessing as mp
  cores = host_cores()
  pool = mp.get_context("fork").Pool(cores)
  for _ in range(args.warmup):
    run_cpu_port(args, moves_per_worker=1, pool=pool, cores=cores)
  total_moves, t0 = 0, time.perf_counter()
  for _ in range(args.steps):
    _, _, moves, _ = run_cpu_port(args, moves_per_worker=args.ref_moves_per_step, pool=pool, cores=cores)
    total_moves += moves
  elapsed = time.perf_counter() - t0
  pool.close()
  pool.join()
  value = total_moves * args.sims / elapsed
  sample = "%d worker processes x %d moves x %d sims per step (A=%d, FCNetwork %d->50, B=1 torch CPU)" % (
      cores, args.ref_moves_per_step, args.sims, args.actions, args.obs_dim)
  line = {
      "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
      "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * elapsed / max(1, args.steps),
      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64 tree / f32 net",
      "data": "synthetic",
      "config": workload_config(args, 1, cpu=True),
      "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
      "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
      "l2": "n/a (CPU)",
  }
  emit(line)


def workload_config(args, n_gpus, cpu=False):
  """Identical in both arms (the driver compares them key by key)."""
  return {"workload": "C4 synthetic Atari-scale search sweep: A=%d, %d games x %d sims per GPU, "
                      "FCNetwork(%d->50), Dirichlet root noise, temperature 1" %
                      (args.actions, args.games, args.sims, args.obs_dim),
          "games_per_gpu": args.games, "num_simulations": args.sims, "action_space": args.actions,
          "obs_dim": args.obs_dim, "parallelism": "independent games, sharded across GPUs, no search collective"}


L2_POLICY = "L2 flushed (512 MiB memset) between timed steps, outside the per-step event pairs"


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
  Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
       "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
       "clocks_event_reasons.sw_power_cap")
  NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

  def __init__(self, index):
    self.rows, self.proc, self.index = [], None, index

  def _nvml_loop(self):
    """Samples through NVML every 2 ms: the timed region of the default run lasts ~50 ms, which
    `nvidia-smi -lms 100` sees once."""
    nv, h = self.nv, self.handle
    bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
    get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
    mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
    while not self.stop_flag:
      try:
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        mask = int(get_reasons(h))
        row = [str(sm), str(mx), ""] + ["Active" if mask & b else "Not Active" for b in
                                        (bits[n] for n in self.NAMES)]
        self.rows.append(row)
      except Exception:
        pass
      time.sleep(0.002)

  def start(self):
    self.stop_flag, self.nv = False, None
    try:
      import pynvml as nv
      nv.nvmlInit()
      self.handle = nv.nvmlDeviceGetHandleByIndex(self.index)
      self.nv = nv
      self.how = "nvml, 2 ms"
      self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
      self.thread.start()
      return
    except Exception:
      self.nv = None
    self.how = "nvidia-smi -lms 100"
    try:
      self.proc = subprocess.Popen(
          ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
           "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
          stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._read, daemon=True)
      self.thread.start()
    except OSError:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append([c.strip() for c in line.split(",")])

  def stop(self):
    if self.nv is not None:
      self.stop_flag = True
      self.thread.join(timeout=1)
    elif self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    else:
      time.sleep(0.15)
      self.proc.terminate()
      try:
        self.proc.wait(timeout=2)
      except subprocess.TimeoutExpired:
        self.proc.kill()
    sm, mx, reasons = [], [], set()
    for r in self.rows:
      try:
        sm.append(float(r[0]))
        mx.append(float(r[1]))
      except (ValueError, IndexError):
        continue
      for name, cell in zip(self.NAMES, r[3:7]):
        if cell.lower().startswith("active"):
          reasons.add(name)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "samples": len(sm), "sampler": self.how, "reasons": sorted(reasons)}


def measured_peaks():
  path = os.path.join(REPO, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    d = json.load(open(path))
    return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
            "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
  return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local = int(os.environ.get("LOCAL_RANK", "0"))

  cpu_baseline = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    # before CUDA is initialised (fork-safe); bounded sample of the same workload
    v, cores, moves, el = run_cpu_port(args, seconds=args.cpu_baseline_seconds)
    cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                    "sample": "%d moves (= %d expansions) of the C4 workload in %.1f s on %d worker "
                              "processes, python port of mcts.py + torch CPU FCNetwork at B=1" %
                              (moves, moves * args.sims, el, cores)}

  import torch
  import torch.distributed as dist
  from model_based_rl_b200 import _lib
  from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict
  if not torch.cuda.is_available():
    raise RuntimeError("GPU was requested but torch.cuda.is_available() is False.")
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
  _lib.load()
  if args.wide_step_max_games is not None:
    _lib.load().mz_tree_set_wide_step_max_games(args.wide_step_max_games)

  cfg = search_config(args)
  G, S, A = args.games, args.sims, args.actions
  net = FCNetwork(args.obs_dim, A, dev, cfg, precision=args.precision)
  sd = {k: v.to(dev) for k, v in random_state_dict(args.obs_dim, A, seed=1234 + rank).items()}
  if world > 1:  # learner -> self-play ranks weight hand-off over NCCL (rank 0 plays the learner)
    from model_based_rl_b200 import parallel
    parallel.broadcast_weights(sd, src=0)
  net.load_weights(sd)
  fused = {"auto": None, "0": False, "1": True}[args.fused]
  fs = FCSearch(cfg, net, G, use_graph=not args.no_graph, num_streams=args.streams, fused=fused)
  obs, noise, uniforms, temperature = synthetic_inputs(args, rank, G)
  pin = lambda a: torch.from_numpy(a).pin_memory()
  h_obs, h_noise, h_u, h_t = pin(obs), pin(noise), pin(uniforms), pin(temperature)
  # end to end the observations cross PCIe as the bytes the emulator produces; the device normalises them
  h_obs_u8 = pin(synthetic_inputs(args, rank, G, as_bytes=True)[0])
  fs.search_host(h_obs_u8, h_noise, h_u, h_t)
  obs_from_bytes = fs.obs.clone()
  fs.search_host(h_obs, h_noise, h_u, h_t)  # also leaves the inputs resident in HBM
  assert torch.equal(obs_from_bytes, fs.obs), "device-side normalisation differs from numpy's"

  flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
  # learner side at N > 1 (BASELINE config C4 "with learner allreduce"): one gradient-sized
  # all-reduce per step on a side stream; the search itself has no collective.
  grad = torch.zeros(sum(v.numel() for v in net.state_dict().values()), device=dev) if world > 1 else None
  side = torch.cuda.Stream(device=dev) if world > 1 else None

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def timed(fn, steps):
    pairs = []
    for _ in range(steps):
      flush.zero_()
      if side is not None:
        with torch.cuda.stream(side):
          dist.all_reduce(grad)
      s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      s.record()
      fn()
      e.record()
      pairs.append((s, e))
    if side is not None:
      torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    return sum(s.elapsed_time(e) for s, e in pairs)

  clocks = ClockSampler(local)
  if rank == 0:
    clocks.start()  # sampled from the warm-up on: the GPU is under the same load there
  for _ in range(args.warmup):
    fs.run()
  barrier()
  ms_total = timed(fs.run, args.steps)
  barrier()
  # later sections run fs again (the concurrent learner also hands it new weights): keep this move's outputs now
  outputs = search_outputs(fs) if args.dump_outputs is not None and rank == 0 else None
  # end-to-end: host buffers in, host buffers out, through the public call
  pinned = fs.pinned_inputs()  # the engine's own pinned staging views: the host writes a move's inputs here
  for name, src in (("obs_u8", h_obs_u8), ("noise", h_noise), ("uniforms", h_u), ("temperature", h_t)):
    pinned[name].copy_(src)
  for _ in range(args.warmup):
    fs.search_pinned()
  ms_e2e = timed(fs.search_pinned, args.steps)
  barrier()
  clock_info = clocks.stop() if rank == 0 else None

  # per-kernel durations (CUDA events around each launch of one un-graphed move), at the launch shape the
  # timed graph uses: the games of ONE slice (G / streams) per launch, and for reference all G games in one
  n_slices = 1 if fs.fused is not None else len(fs.lanes)
  g_slice = (G + n_slices - 1) // n_slices
  kern, kern_full = None, None
  for gk in sorted({g_slice, G}):
    fs1 = FCSearch(cfg, net, gk, use_graph=False, num_streams=1, fused=False)  # un-graphed, one stream
    for name in ("obs", "noise", "uniforms", "temperature"):
      getattr(fs1, name).copy_(getattr(fs, name)[:gk])
    k = kernel_breakdown(fs1, torch)
    k["games_per_launch"] = gk
    if gk == g_slice:
      kern = k
    if gk == G:
      kern_full = k
    del fs1
  fused_us = None
  if fs.fused is not None:  # the persistent kernel alone: CUDA events around its launch in an un-graphed move
    fsu = FCSearch(cfg, net, G, use_graph=False, num_streams=1, fused=True)
    for name in ("obs", "noise", "uniforms", "temperature"):
      getattr(fsu, name).copy_(getattr(fs, name))
    fused_us = fused_kernel_us(fsu, torch)
    del fsu
  f32_line = None
  if rank == 0 and world == 1 and args.precision == "bf16" and not args.no_f32:
    # the same move with the reference-precision (float32, CUDA-core) network kernel
    net32 = FCNetwork(args.obs_dim, A, dev, cfg, precision="f32")
    net32.load_weights(sd)
    fs32 = FCSearch(cfg, net32, G, use_graph=not args.no_graph, num_streams=args.streams)
    fs32.search_host(h_obs, h_noise, h_u, h_t)
    for _ in range(args.warmup):
      fs32.run()
    torch.cuda.synchronize()
    n32 = max(3, min(args.steps, 10))
    ms32 = timed(fs32.run, n32)
    f32_line = {"value": G * S * n32 / (ms32 * 1e-3), "unit": UNIT, "ms_per_step": ms32 / n32, "steps": n32,
                "network": "fc_recurrent_f32_kernel (float32 CUDA cores; parity bar vs the reference's torch module: "
                           "1e-4, tests/test_gpu_fcnet.py)", "same_workload": True}
    del fs32, net32
    # and with the float32-accurate TENSOR-CORE network kernel (three TF32 products per multiply)
    net3 = FCNetwork(args.obs_dim, A, dev, cfg, precision="tf32x3")
    net3.load_weights(sd)
    fs3 = FCSearch(cfg, net3, G, use_graph=not args.no_graph, num_streams=args.streams)
    fs3.search_host(h_obs, h_noise, h_u, h_t)
    for _ in range(args.warmup):
      fs3.run()
    torch.cuda.synchronize()
    ms3 = timed(fs3.run, n32)
    f32_line["tensor_core"] = {
        "value": G * S * n32 / (ms3 * 1e-3), "unit": UNIT, "ms_per_step": ms3 / n32, "steps": n32,
        "network": "fc_recurrent_tf32x3_kernel (mma.sync TF32 x 3 on split operands, float32 accumulate; same parity "
                   "bars as the CUDA-core kernel + 2e-5 against it, tests/test_gpu_fcnet.py)"}
    del fs3, net3

  t = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device=dev)
  if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms_total, ms_e2e = t.tolist()
  sweep = None
  if rank == 0 and world == 1 and not args.no_sweep:
    # the same move at larger batches: at 4096 games a step is bound by the latency of the two
    # per-simulation kernels in series; the kernels' own throughput shows when more games are in flight
    sweep = {}
    for g2 in (4 * G,):
      fs2 = FCSearch(cfg, net, g2, use_graph=not args.no_graph, num_streams=args.streams)
      o2, n2, u2, t2 = synthetic_inputs(args, rank, g2)
      fs2.search_host(pin(o2), pin(n2), pin(u2), pin(t2))
      for _ in range(args.warmup):
        fs2.run()
      torch.cuda.synchronize()
      ms2 = timed(fs2.run, 5)
      sweep[str(g2)] = {"expansions_per_s": g2 * S * 5 / (ms2 * 1e-3), "ms_per_step": ms2 / 5}
      del fs2
      # the two kernels' own rooflines at this batch (one slice, un-graphed, CUDA events per launch)
      fs3 = FCSearch(cfg, net, g2, use_graph=False, num_streams=1)
      for name, src in (("obs", o2), ("noise", n2), ("uniforms", u2), ("temperature", t2)):
        getattr(fs3, name).copy_(torch.from_numpy(src).to(dev))
      k2 = kernel_breakdown(fs3, torch)
      del fs3
      pk = measured_peaks()
      tb = g2 * (k2["mean_depth"] * (28 * A + 33) + 16 * A + 86)
      sweep[str(g2)]["kernels"] = {
          "tree_step_us": k2["tree_step_us"], "fc_recurrent_us": k2["fc_recurrent_us"],
          "tree_hbm_frac": tb / (k2["tree_step_us"] * 1e-6) / 1e9 / pk["hbm_gbs"],
          "fc_tensor_frac": g2 * FC_FLOPS_PER_EXPANSION(A) / (k2["fc_recurrent_us"] * 1e-6) / 1e12 /
                            pk["bf16_tflops_sustained"]}
  others = bench_other_configs(args, torch, dev, timed) if rank == 0 and world == 1 and not args.no_sweep else None
  targets = bench_targets(torch, _lib, dev) if rank == 0 else None
  replay = bench_replay(torch, _lib, dev, cpu_baseline=not args.no_cpu_baseline) if rank == 0 else None
  selfplay = (bench_selfplay(args, torch, dev, cpu_baseline["value"] if cpu_baseline else None)
              if rank == 0 and world == 1 and not args.no_selfplay else None)
  learner = bench_learner(torch, _lib, dev, world, barrier)  # every rank: the step all-reduces at N > 1
  concurrent = (bench_concurrent(args, torch, dev, world, fs, net, barrier, flush)
                if not args.no_concurrent else None)  # every rank: gradient all-reduce + weight broadcast
  conv = bench_conv(args, torch, _lib, dev) if rank == 0 and not args.no_conv else None

  if rank == 0:
    peaks = measured_peaks()
    expansions = world * G * S * args.steps
    value = expansions / (ms_total * 1e-3)
    e2e = expansions / (ms_e2e * 1e-3)
    # algorithmic bytes / flops per launch (SURVEY.md section 8d, DESIGN.md "Kernels")
    d = kern["mean_depth"]
    gl = kern["games_per_launch"]  # the launch shape of the timed region
    per_game_bytes = d * (28 * A + 33) + 16 * A + 86
    tree_bytes = gl * per_game_bytes
    fc_flops = gl * FC_FLOPS_PER_EXPANSION(A)
    tree_t, fc_t = kern["tree_step_us"] * 1e-6, kern["fc_recurrent_us"] * 1e-6
    tree_name = "tree_step_w32_kernel"
    fc_name = {"bf16": "fc_recurrent_tc_kernel", "f32": "fc_recurrent_f32_kernel",
               "tf32x3": "fc_recurrent_tf32x3_kernel"}[args.precision]
    roof_tree = {"kernel": tree_name, "bound": "hbm", "achieved": tree_bytes / tree_t / 1e9,
                 "peak": peaks["hbm_gbs"], "unit": "GB/s",
                 "traffic": ncu_traffic(tree_name, gl, A, S),
                 "games_per_launch": gl, "algorithmic_bytes_per_launch": tree_bytes,
                 "avg_launch_us": kern["tree_step_us"]}
    roof_fc = {"kernel": fc_name, "bound": "tensor", "achieved": fc_flops / fc_t / 1e12,
               "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
               "traffic": ncu_traffic(fc_name, gl, A, S),
               "games_per_launch": gl, "algorithmic_flops_per_launch": fc_flops,
               "avg_launch_us": kern["fc_recurrent_us"]}
    roofs = [roof_tree, roof_fc]
    if fused_us is not None:  # one launch = the whole move: both resources against the same duration
      move_bytes, move_flops = S * G * per_game_bytes, S * G * FC_FLOPS_PER_EXPANSION(A)
      roof_fused = {"kernel": "fc_search_kernel", "bound": "hbm", "achieved": move_bytes / (fused_us * 1e-6) / 1e9,
                    "peak": peaks["hbm_gbs"], "unit": "GB/s", "traffic": ncu_traffic("fc_search_kernel", G, A, S),
                    "games_per_launch": G, "algorithmic_bytes_per_launch": move_bytes, "avg_launch_us": fused_us,
                    "tensor_tflops": move_flops / (fused_us * 1e-6) / 1e12,
                    "tensor_frac": move_flops / (fused_us * 1e-6) / 1e12 / peaks["bf16_tflops_sustained"]}
      roofs = [roof_fused] + roofs
    for r in roofs:
      r["frac"] = r["achieved"] / r["peak"]
      r["peak_source"] = peaks["source"]
    dominant = roofs[0] if fused_us is not None else (roof_fc if fc_t >= tree_t else roof_tree)
    # the whole timed step against both roofs (algorithmic bytes / FLOPs of all S simulations of all games)
    step_s = ms_total * 1e-3 / args.steps
    whole_step = {"hbm_gbs": S * G * per_game_bytes / step_s / 1e9,
                  "hbm_frac": S * G * per_game_bytes / step_s / 1e9 / peaks["hbm_gbs"],
                  "tensor_tflops": S * G * FC_FLOPS_PER_EXPANSION(A) / step_s / 1e12,
                  "tensor_frac": S * G * FC_FLOPS_PER_EXPANSION(A) / step_s / 1e12 / peaks["bf16_tflops_sustained"],
                  "note": "per GPU; the step is %d dependent simulations, not one roofline-bound kernel" % S}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 (tree) / %s (network)" % {"bf16": "bf16 tcgen05, f32 accumulate", "f32": "f32",
                                                 "tf32x3": "tf32 x 3 mma.sync, f32 accumulate"}[args.precision],
        "data": "synthetic", "config": workload_config(args, world),
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": fs.h2d_blob_bytes(),
                "inputs": "pinned host blob, one copy per direction: uint8 observations (normalised on the device), "
                          "float64 noise / uniforms / temperatures, legal masks, to_play",
                "d2h_bytes_per_step": fs.d2h_bytes(), "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": fs.launches_per_move * args.steps,
        "clocks": clock_info, "roofline": dominant, "roofline_all": roofs, "whole_step": whole_step,
        "kernel_share": kern, "kernel_share_all_games_one_launch": kern_full,
        "fused_search_kernel": fs.fused is not None, "l2": L2_POLICY,
        "cuda_graph": not args.no_graph, "streams": n_slices, "f32_network": f32_line,
        "games_sweep": sweep, "other_configs": others, "targets": targets, "replay": replay, "selfplay": selfplay, "learner": learner,
        "concurrent_learner": concurrent,
        "conv": conv,
    }
    if cpu_baseline is not None:
      line["cpu_baseline"] = cpu_baseline
    if outputs is not None:
      dump_outputs(args.dump_outputs, outputs)
    emit(line)
  if world > 1:
    dist.destroy_process_group()


DUMP_BYTES = 60 << 20  # under 64 MB with the .npy headers


def search_outputs(fs):
  """The arrays FCSearch.search_host returns for the move in fs's device buffers, as float64 / float32 numpy arrays
  (the int32 actions as float64, exactly)."""
  return {"actions": fs.actions.cpu().numpy().astype(np.float64), "root_value": fs.root_value.cpu().numpy(),
          "child_visits": fs.child_visits.cpu().numpy(), "init_value": fs.init_value.cpu().numpy()}


def dump_outputs(path, outputs):
  """Writes every per-game array as path/<name>.npy.  Past DUMP_BYTES in all, a fixed seeded sample of the games is
  written instead: the same games in every array, their indices as game_index.npy."""
  games = len(outputs["actions"])
  row_bytes = sum(a[:1].nbytes for a in outputs.values())
  if games * row_bytes > DUMP_BYTES:
    keep = np.sort(np.random.default_rng(0).choice(games, DUMP_BYTES // (row_bytes + 8), replace=False))
    outputs = {name: a[keep] for name, a in outputs.items()}
    outputs["game_index"] = keep.astype(np.float64)
  os.makedirs(path, exist_ok=True)
  for name, a in outputs.items():
    np.save(os.path.join(path, name + ".npy"), a)


def bench_other_configs(args, torch, dev, timed):
  """The FCNetwork configurations of BASELINE.json besides C4, same move, resident inputs (parity-test
  shapes; reported for orientation): C1 Tic-Tac-Toe (two players, known bounds -1 1), C2 LunarLander,
  C3 Breakout-ram."""
  import argparse
  from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict
  out = {}
  for name, G, A, S, D, two, bounds in (("C1_tictactoe", 4096, 9, 30, 9, True, [-1, 1]),
                                        ("C2_lunarlander", 1024, 4, 30, 8, False, [None, None]),
                                        ("C3_breakout_ram", 4096, 4, 50, 128, False, [None, None])):
    a2 = argparse.Namespace(**vars(args))
    a2.games, a2.actions, a2.sims, a2.obs_dim = G, A, S, D
    cfg = search_config(a2)
    cfg.two_players, cfg.known_bounds = two, bounds
    if two:
      cfg.discount = 1.0
    net = FCNetwork(D, A, dev, cfg, precision=args.precision)
    net.load_weights({k: v.to(dev) for k, v in random_state_dict(D, A, seed=99).items()})
    fs = FCSearch(cfg, net, G, use_graph=not args.no_graph, num_streams=args.streams)
    obs, noise, u, t = synthetic_inputs(a2, 0, G)
    fs.search_host(obs, noise, u, t)
    for _ in range(3):
      fs.run()
    torch.cuda.synchronize()
    ms = timed(fs.run, 5)
    out[name] = {"games": G, "actions": A, "sims": S, "obs_dim": D, "expansions_per_s": G * S * 5 / (ms * 1e-3),
                 "ms_per_move": ms / 5}
    del fs
  return out


def _source_sha16(names):
  """sha256 over the kernel's source files ('a.cu+b.cuh': concatenated in that order), first 16 hex digits."""
  import hashlib
  h = hashlib.sha256()
  for name in names.split("+"):
    path = os.path.join(REPO, "model-based-rl_b200", "csrc", name)
    if not os.path.exists(path):
      return None
    h.update(open(path, "rb").read())
  return h.hexdigest()[:16]


def ncu_traffic(kernel, games, A, S):
  """dram__bytes_read.sum + dram__bytes_write.sum per launch from an `ncu --set full` capture of THIS kernel
  source at THIS launch shape (profiles/traffic.json, written by tests/ncu_traffic.py from the capture;
  an entry only counts while the kernel's .cu file is byte-identical to the captured one), else null."""
  path = os.path.join(REPO, "profiles", "traffic.json")
  if not os.path.exists(path):
    return None
  for e in json.load(open(path)).get("entries", []):
    if (e.get("kernel") == kernel and e.get("games") == games and e.get("actions") == A and e.get("sims") == S and
        e.get("source_sha16") == _source_sha16(e.get("source", ""))):
      return e.get("dram_bytes_per_launch")
  return None


def fused_kernel_us(fs, torch):
  """Device time of the persistent search kernel alone (CUDA events around the launch, un-graphed move)."""
  fs.run()
  torch.cuda.synchronize()
  plan = fs._fused_plan
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  total = 0.0
  for _ in range(3):
    plan[0][0](*plan[0][1])
    a.record()
    rc = plan[1][0](*plan[1][1])
    b.record()
    assert rc == 0, rc
    plan[2][0](*plan[2][1])
    torch.cuda.synchronize()
    total += a.elapsed_time(b) * 1e3
  return total / 3


def kernel_breakdown(fs, torch):
  """Average device time of the two per-simulation kernels: CUDA events on the launching stream
  around every launch of one un-graphed move (pre-marshalled launch list, so the host keeps ahead
  of the device)."""
  ln = fs.lanes[0]
  S = fs.S
  plan = ln._plan(fs.use_noise, fs.noise_frac, torch.cuda.current_stream().cuda_stream)
  ev = lambda: torch.cuda.Event(enable_timing=True)
  depth_sum = torch.zeros((), dtype=torch.float64, device=ln.eng.path_len.device)
  for i, (fn, args) in enumerate(plan):  # warm-up pass; also collects the mean path length
    fn(*args)
    if 2 <= i < 2 + 2 * S and (i - 2) % 2 == 0:
      depth_sum += ln.eng.path_len.double().mean()
  torch.cuda.synchronize()
  marks = [ev() for _ in range(len(plan) + 1)]
  marks[0].record()
  for i, (fn, args) in enumerate(plan):
    rc = fn(*args)
    assert rc == 0, (fn.__name__, rc)
    marks[i + 1].record()
  torch.cuda.synchronize()
  dur = [marks[i].elapsed_time(marks[i + 1]) * 1e3 for i in range(len(plan))]
  fc_us = sum(dur[3 + 2 * s] for s in range(S)) / S
  tree_us = sum(dur[4 + 2 * s] for s in range(S)) / S
  move_us = marks[0].elapsed_time(marks[-1]) * 1e3
  mean_depth = float(depth_sum.item()) / S
  return {"fc_recurrent_us": fc_us, "tree_step_us": tree_us, "fc_initial_us": dur[0],
          "ungraphed_move_us": move_us, "fc_share": fc_us * S / move_us,
          "tree_share": tree_us * S / move_us, "mean_depth": mean_depth}


def bench_conv(args, torch, _lib, dev):
  """C5 (BASELINE.json configs[4]): MuZeroNetwork residual conv tower, synthetic 96x96 frames with 32 stacked
  channels (and 64: `stack_actions`, utils.py:28-32), A=18, 50 simulations, bf16 tensor-core recurrent_inference.
  Reports whole-move expansions/s through ConvSearch.search (initial_inference -- representation tower included --
  and the search in one CUDA graph), the same with the two parts timed separately, and the tensor roofline of the
  conv kernel."""
  from model_based_rl_b200.muzero import CH, ROWS, ConvSearch, MuZeroNetwork, random_state_dict
  cfg = search_config(args)
  G, S, A = args.conv_games, args.sims, args.actions
  rng = np.random.default_rng(77)
  noise, u = rng.dirichlet([0.25] * A, size=G), rng.random(G)
  a, b, c = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
  res = {}
  for C_in in (32, 64):
    net = MuZeroNetwork(C_in, A, dev, cfg)
    net.load_weights(random_state_dict(C_in, A))
    cs = ConvSearch(cfg, net, G)
    obs = torch.from_numpy(rng.random((G, C_in, 96, 96), dtype=np.float32)).to(dev)
    for _ in range(2):
      cs.search(obs, noise, u)
    torch.cuda.synchronize()
    steps = 3
    ms_graph = 0.0
    for _ in range(steps):  # the public call: one graph per move
      a.record()
      cs.search(obs)
      b.record()
      torch.cuda.synchronize()
      ms_graph += a.elapsed_time(b)
    cs.set_roots(obs)
    cs.run()
    torch.cuda.synchronize()
    ms_move = ms_search = 0.0
    for _ in range(steps):  # the two halves apart: eager initial_inference, then the search graph
      a.record()
      cs.set_roots(obs)
      b.record()
      cs.run()
      c.record()
      torch.cuda.synchronize()
      ms_move += a.elapsed_time(c)
      ms_search += b.elapsed_time(c)
    res[C_in] = {"expansions_per_s": G * S * steps / (ms_graph * 1e-3), "ms_per_move": ms_graph / steps,
                 "expansions_per_s_search_only": G * S * steps / (ms_search * 1e-3),
                 "ms_per_move_two_parts": ms_move / steps, "ms_representation_eager": (ms_move - ms_search) / steps,
                 "recurrent_tflops_useful": G * S * steps * 0.705e9 / (ms_search * 1e-3) / 1e12}
    if C_in == 32:
      # one convolution launch alone (the dominant kernel: 65 of the 70 launches per simulation)
      x = torch.rand((G * ROWS, CH), device=dev).to(torch.bfloat16)
      out = net.buffers(G)["x"][0]
      n = 20
      for _ in range(3):
        net._conv(G, net.dyn_tower[0], x, 3, out, residual=x)
      a.record()
      for _ in range(n):
        net._conv(G, net.dyn_tower[0], x, 3, out, residual=x)
      b.record()
      torch.cuda.synchronize()
      us_conv = a.elapsed_time(b) * 1e3 / n
    del cs, net, obs
  peaks = measured_peaks()
  flops = 2.0 * G * 36 * 128 * 1152  # algorithmic: interior pixels only (the padded rows are overhead)
  roof = {"kernel": "conv_pair_tc_kernel", "bound": "tensor", "achieved": flops / us_conv / 1e6,
          "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
          "traffic": ncu_traffic("conv_pair_tc_kernel", G, A, S),
          "algorithmic_flops_per_launch": flops, "avg_launch_us": us_conv,
          "issued_tflops": 2.0 * G * ROWS * 128 * 1152 / us_conv / 1e6, "peak_source": peaks["source"]}
  roof["frac"] = roof["achieved"] / roof["peak"]
  out = {"workload": "C5 MuZeroNetwork residual conv (16+16 blocks, 128 ch, 6x6 state), %d games x %d "
                     "sims, A=%d, synthetic 96x96x32 frames, bf16 tcgen05 initial_inference (representation "
                     "tower included) and recurrent_inference; one CUDA graph per move" % (G, S, A),
         "gpu_launches_per_move": cs_launches(G, S), "roofline": roof}
  out.update(res[32])
  out["stack_actions_64_channels"] = res[64]
  return out


def cs_launches(G, S):
  return 4 + S * (2 + 70)  # set_root, first descent, per sim: row base + 69 network + tree step, stats, action


def _targets_case(torch, _lib, dev, rng, P, A, K, T, B, E, obs_u8, n_sets, reps, discount=0.997):
  """Times mz_build_targets (supports fused) on one synthetic replay window; returns (seconds per launch,
  algorithmic bytes per sampled row: SURVEY.md section 8d's formula)."""
  lib = _lib.load()
  lens = rng.integers(200, 800, size=P // 200)
  lens = lens[np.cumsum(lens) <= P]
  starts = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
  t = lambda a: torch.from_numpy(a).to(dev)
  if obs_u8:
    obs = t(rng.integers(0, 256, size=(P, E), dtype=np.uint8))
  else:
    obs = t(rng.normal(size=(P, E)).astype(np.float32))
  rewards = t(np.sign(rng.normal(size=P) * (rng.random(P) < 0.1)).astype(np.float32))
  actions = t(rng.integers(0, A, size=P, dtype=np.int32))
  to_play = torch.ones(P, dtype=torch.int8, device=dev)
  root_values = t(rng.normal(0, 2, size=P))
  cv = rng.random((P, A)).astype(np.float32)
  child_visits = t(cv / cv.sum(1, keepdims=True))
  win = _lib.Window(A, E, 1 if obs_u8 else 0, 0, obs.data_ptr(), actions.data_ptr(), rewards.data_ptr(),
                    to_play.data_ptr(), root_values.data_ptr(), child_visits.data_ptr())
  discounts = t(np.array([discount**n for n in range(K + T)], np.float32))
  tc = _lib.TargetCfg(B, K, T, 1, -15, 15, -15, 15, 0, 0, discount**T, discounts.data_ptr(), None, None)
  sets = []
  for _ in range(n_sets):
    ci = rng.integers(0, len(lens), size=B)
    step = (rng.random(B) * lens[ci]).astype(np.int64)
    sets.append((t(starts[ci] + step), t(starts[ci]), t(lens[ci].astype(np.int32)),
                 t(rng.integers(0, A, size=(B, K), dtype=np.int32))))
  out = [torch.zeros((B, E), device=dev), torch.zeros((B, K), dtype=torch.int32, device=dev),
         torch.zeros((B, K + 1), device=dev), torch.zeros((B, K + 1), device=dev),
         torch.zeros((B, K + 1, A), device=dev), torch.zeros((B, K + 1, 31), device=dev),
         torch.zeros((B, K + 1, 31), device=dev)]
  stream = _lib.current_stream()

  def launch(s):
    _lib.check(lib.mz_build_targets(win, tc, _lib.ptr(s[0]), _lib.ptr(s[1]), _lib.ptr(s[2]),
                                    _lib.ptr(s[3]), *[_lib.ptr(o) for o in out], stream), "targets")
  for s in sets[:4]:
    launch(s)
  torch.cuda.synchronize()
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record()
  for _ in range(reps):
    for s in sets:
      launch(s)
  b.record()
  torch.cuda.synchronize()
  sec = a.elapsed_time(b) * 1e-3 / (n_sets * reps)
  in_bytes = E * (1 if obs_u8 else 4)
  bytes_per_sample = (in_bytes + 5 * (T + K) + (K + 1) * (8 + 4 * A) + 4 * K) + \
                     (4 * E + 4 * K + (K + 1) * (4 * A + 8)) + (K + 1) * 2 * 31 * 4
  return sec, bytes_per_sample


def bench_targets(torch, _lib, dev):
  """targets/s of the fused target kernel.  Headline: the C3 (Breakout-ram) learner batch -- window 200k
  positions, B=512, K=5, td=10, A=4, obs 128 x u8, supports fused (one launch per batch: launch bound).
  `bulk`: the same kernel producing 128 learner batches (65 536 rows) per launch, outputs larger than L2 --
  the regime where HBM bounds it -- for the C3 shape and the C2 (LunarLander, td_steps=1000) shape."""
  rng = np.random.default_rng(5)
  peaks = measured_peaks()
  hbm = peaks["hbm_gbs"]
  P, A, K, T, B, E = 200_000, 4, 5, 10, 512, 128
  sec, bps = _targets_case(torch, _lib, dev, rng, P, A, K, T, B, E, True, 64, 1)
  res = {"samples_per_s": B / sec, "target_positions_per_s": B * (K + 1) / sec, "us_per_batch": sec * 1e6,
         "workload": "C3 Breakout-ram: window 200000, B=512, K=5, td=10, A=4, obs 128 u8, supports fused",
         "algorithmic_bytes_per_sample": bps, "achieved_gbs": B * bps / sec / 1e9}
  bulk = {}
  for name, (A2, T2, E2, u8, disc) in {"C3_breakout_ram": (4, 10, 128, True, 0.997),
                                       "C2_lunarlander_td1000": (4, 1000, 8, False, 0.997)}.items():
    Bb = 128 * 512
    sec, bps = _targets_case(torch, _lib, dev, rng, P, A2, K, T2, Bb, E2, u8, 4, 5, disc)
    gbs = Bb * bps / sec / 1e9
    rows_kernel = T2 <= 64  # mz_build_targets picks the TMA-staged lane-per-position kernel for K + 1 <= 16, td_steps <= 64
    bulk[name] = {"rows_per_launch": Bb, "us_per_launch": sec * 1e6, "samples_per_s": Bb / sec,
                  "algorithmic_bytes_per_sample": bps,
                  "roofline": {"kernel": "build_targets_tma_kernel" if rows_kernel else "build_targets_kernel",
                               "bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                               "traffic": ncu_traffic("build_targets_tma_kernel" if rows_kernel else
                                                      "build_targets_kernel", Bb, A2, T2),
                               "peak_source": peaks["source"]}}
  res["bulk"] = bulk
  return res


def bench_replay(torch, _lib, dev, cpu_baseline=True):
  """The replay facade end to end on the C3 (Breakout-ram) shape: PrioritizedReplay filled through
  save_history with synthetic 500-step chunks (window 200 000, B = 512, K = 5, td = 10, A = 4, 128-byte
  observations), then `sample_batch()` (the reference's numpy tuple: sum-tree sampling + target kernel +
  device-to-host copies), `sample_batch_device()` (nothing leaves the GPU) and `update()`.  Beside it the
  CPU port of the same row loop (oracle SumTree + oracle insert_target, one process -- the reference's
  replay buffer is a single Ray actor)."""
  import types
  from model_based_rl_b200.replay_buffer import PrioritizedReplay
  from model_based_rl_b200.selfplay import HistorySlice
  rng = np.random.default_rng(9)
  W, A, K, T, B, E, L = 200_000, 4, 5, 10, 512, 128, 500
  cfg = types.SimpleNamespace(batch_size=B, beta_increment_per_sampling=0.001, epsilon=0.01, alpha=1.0, beta=0.4,
                              num_unroll_steps=K, td_steps=T, discount=0.997, action_space=A, obs_space=(E,),
                              window_size=W, window_step=None, max_history_length=L, seed=3)
  rb = PrioritizedReplay(cfg, device=dev)
  hist = []
  n_chunks = W // L
  for _ in range(n_chunks):
    obs = list(rng.integers(0, 256, size=(L + 1, E), dtype=np.uint8))
    cv = rng.random((L, A))
    h = HistorySlice(obs, (cv / cv.sum(1, keepdims=True)).tolist(), rng.normal(0, 2, size=L).tolist(),
                     rng.integers(0, A, size=L).tolist(),
                     np.sign(rng.normal(size=L) * (rng.random(L) < 0.1)).astype(np.int64).tolist(),
                     np.abs(rng.normal(size=L)).tolist(), [False] * L, list(range(L)), [None] * L, [1] * L)
    rb.save_history(h, ignore=None, terminal=True)
    if len(hist) < 40:
      hist.append(h)
  torch.cuda.synchronize()

  def wall(fn, n):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
      fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n
  t_host = wall(rb.sample_batch, 20)
  t_dev0 = wall(lambda: rb.sample_batch_device(True), 50)
  t_dev = wall(lambda: rb.sample_batch_device(True, ring=4), 200)
  _, idxs, _ = rb.sample_batch()
  errs = np.abs(rng.normal(size=B)).astype(np.float32)
  t_upd0 = wall(lambda: rb.update(idxs, errs), 20)
  d_idx, d_err = torch.tensor(idxs, dtype=torch.int64, device=dev), torch.from_numpy(errs).to(dev)
  t_upd = wall(lambda: rb.update(d_idx, d_err), 200)
  out = {"workload": "C3 Breakout-ram replay: window %d filled by save_history, B=%d, K=%d, td=%d, A=%d, obs %d u8" % (W, B, K, T, A, E),
         "size": rb.size(),
         "sample_batch_samples_per_s": B / t_host, "sample_batch_ms": t_host * 1e3,
         "sample_batch_device_samples_per_s": B / t_dev, "sample_batch_device_ms": t_dev * 1e3,
         "sample_batch_device_fresh_outputs_ms": t_dev0 * 1e3,
         "update_ms": t_upd * 1e3, "update_host_arrays_ms": t_upd0 * 1e3,
         "note": "sample_batch_device: ring of 4 preallocated output sets, pinned staging, one library call "
                 "(mz_replay_sample_targets); update: CUDA idxs + float32 errors (mz_sumtree_update_errors); the "
                 "*_fresh_outputs / *_host_arrays figures are the same calls with per-call allocations / numpy inputs"}
  if cpu_baseline:
    import oracle
    from oracle import replay_ref
    tree = replay_ref.SumTreeRef(len(hist) * L, len(hist) * L)
    for i, h in enumerate(hist):
      tree.add(replay_ref.get_priorities(np.asarray(h.errors), cfg.epsilon, cfg.alpha), i)
    arrs = [(np.asarray(h.rewards, np.float64), np.asarray(h.to_play, np.int8), np.asarray(h.root_values),
             np.asarray(h.child_visits)) for h in hist]
    t0, rows = time.perf_counter(), 0
    while time.perf_counter() - t0 < 2.0:
      picks, _ = replay_ref.sample_indices(tree, B, rng.random(B), 0.4)
      for (_, _, step, hid) in picks:
        r, tp, rv, cv = arrs[hid]
        oracle.insert_target(r, tp, rv, cv, K, T, cfg.discount, step)
        np.float32(hist[hid].observations[step])
      rows += B
    dt = time.perf_counter() - t0
    out["cpu_baseline"] = {"value": rows / dt, "unit": "samples/s", "cores": 1, "kind": "port",
                           "sample": "%d rows in %.1f s: python SumTree descent + C insert_target per row "
                                     "(the reference's sample_batch is a per-row Python loop in one Ray actor)" % (rows, dt)}
  return out


def bench_selfplay(args, torch, dev, cpu_expansions_per_s=None):
  """The actor replacement end to end (SURVEY.md section 8 f-2 / f-3): `DeviceActor.play_move` at the C4 shape --
  4096 games, A = 18, 50 simulations, 128-byte observations from a synthetic vector environment -- with the
  trajectories written on the device into a Breakout-sized replay window (200 000 memories, 500-step chunks with
  the K + td overlap) and priorities added per finished chunk.  Wall clock per move, everything included: host
  environment step, noise / uniform draws, the search call with its copies, the append launch, chunk commits.
  `list_path` is the same move through BatchedActor (per-game Python lists, HistorySlice upload)."""
  import types
  from model_based_rl_b200.environments import SyntheticRam
  from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict
  from model_based_rl_b200.replay_buffer import PrioritizedReplay
  from model_based_rl_b200.selfplay import BatchedActor, DeviceActor
  G, A, S, D = args.games, args.actions, args.sims, args.obs_dim
  cfg = search_config(args)
  for k, v in dict(num_unroll_steps=5, td_steps=10, max_history_length=500, max_steps=27000, batch_size=512,
                   beta_increment_per_sampling=0.001, epsilon=0.01, alpha=1.0, beta=0.4, obs_space=(D,),
                   window_size=200_000, window_step=None, seed=None, clip_rewards=True).items():
    setattr(cfg, k, v)
  net = FCNetwork(D, A, dev, cfg, precision=args.precision)
  net.load_weights({k: v.to(dev) for k, v in random_state_dict(D, A, seed=5).items()})
  out = {"workload": "self-play move: %d games, A=%d, %d sims, obs %d u8, episodes of 600 steps, replay window 200000 "
                     "(chunks of 500 + 15 overlap), clip_rewards" % (G, A, S, D)}
  np.random.seed(0)
  for name in ("device", "list_path"):
    env = SyntheticRam(G, A, D, episode_length=600, seed=1)
    rb = PrioritizedReplay(cfg, device=dev, window_positions=int(200_000 * 1.3) + 3 * G * 515)
    fs = FCSearch(cfg, net, G)
    if name == "device":
      actor = DeviceActor(cfg, env, rb, fs)
    else:
      actor = BatchedActor(cfg, net, env, replay_buffer=rb, device=dev, search=fs)
    # stagger the games so that chunk commits are spread over the moves like in steady state
    env.elapsed[:] = np.arange(G) % 600
    moves = 30 if name == "device" else 6
    for _ in range(3):
      actor.play_move()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(moves):
      actor.play_move()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / moves
    out[name] = {"ms_per_move": dt * 1e3, "moves_per_s": 1.0 / dt, "expansions_per_s": G * S / dt,
                 "experiences_per_s": G / dt, "games_finished": actor.games_played, "replay_size": rb.size()}
    del actor, rb, fs
  # two actors of G games each taking turns on the GPU (the reference runs several Ray actors beside each other):
  # one actor's search runs on the device while the host does the other's environment step / append / staging
  from model_based_rl_b200.selfplay import PipelinedActors
  rb = PrioritizedReplay(cfg, device=dev, window_positions=int(200_000 * 1.3) + 6 * G * 515)
  actors = []
  for k in range(2):
    env = SyntheticRam(G, A, D, episode_length=600, seed=1 + k)
    actors.append(DeviceActor(cfg, env, rb, FCSearch(cfg, net, G)))
    env.elapsed[:] = np.arange(G) % 600  # (after the actor's reset) chunk commits spread over the moves
  pipe = PipelinedActors(actors)
  for _ in range(3):
    pipe.play_round()
  torch.cuda.synchronize()
  rounds = 30
  t0 = time.perf_counter()
  for _ in range(rounds):
    pipe.play_round()
  torch.cuda.synchronize()
  dt = (time.perf_counter() - t0) / rounds
  pipe.drain()
  out["pipelined_two_actors"] = {
      "actors": 2, "games_per_actor": G, "ms_per_round": dt * 1e3, "ms_per_actor_move": dt * 1e3 / 2,
      "expansions_per_s": 2 * G * S / dt, "experiences_per_s": 2 * G / dt, "replay_size": rb.size(),
      "games_finished": sum(a.games_played for a in actors),
      "note": "PipelinedActors: the same DeviceActor moves, each actor's next search enqueued before the other's host "
              "work starts"}
  del pipe, actors, rb
  out["speedup_vs_list_path"] = out["list_path"]["ms_per_move"] / out["device"]["ms_per_move"]
  if cpu_expansions_per_s:
    out["cpu_baseline"] = {"value": cpu_expansions_per_s / S, "unit": "game-moves/s", "kind": "port",
                           "sample": "the cpu_baseline leg of this run (the reference's actor spends its time in the "
                                     "search: moves/s = expansions/s / num_simulations)"}
    out["device"]["game_moves_per_s"] = G / (out["device"]["ms_per_move"] * 1e-3)
  return out


def bench_concurrent(args, torch, dev, world, fs, net, barrier, flush):
  """BASELINE config C4 "with learner allreduce" as it runs in training: while the search plays its moves on the
  main stream, a real learner (`Learner.update_weights` on batches from `PrioritizedReplay.sample_batch_device`,
  priorities fed back on the device) trains on a side stream of the same GPU -- at N > 1 with the NCCL gradient
  all-reduce of the data-parallel step every step -- and hands its weights to the search network every
  `send_weights_frequency` steps (learners.py:115-148, actors.py:81-85; rank 0's weights are broadcast).  One
  learner step is enqueued per move.  Reported: both rates alone and together, max over ranks."""
  import types
  import torch.distributed as dist
  from model_based_rl_b200 import fused_learner
  from model_based_rl_b200.replay_buffer import PrioritizedReplay
  from model_based_rl_b200.selfplay import HistorySlice
  G, S, A, D = args.games, args.sims, args.actions, args.obs_dim
  B, K, T, L, W = 512, 5, 10, 500, 30_000
  cfg = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=False, no_target_transform=False,
                              num_unroll_steps=K, td_steps=T, optimizer="AdamW", lr_init=0.0008, momentum=0.9,
                              weight_decay=1e-4, clip_grad=0, lr_scheduler=None, norm_obs=False, batch_size=B,
                              beta_increment_per_sampling=0.001, epsilon=0.01, alpha=1.0, beta=0.4, discount=0.997,
                              action_space=A, obs_space=(D,), window_size=W, window_step=None, max_history_length=L,
                              seed=None, clip_rewards=True)
  rng = np.random.default_rng(21)
  rb = PrioritizedReplay(cfg, device=dev)
  for _ in range(W // L):
    cv = rng.random((L, A))
    rb.save_history(HistorySlice(list(rng.integers(0, 256, size=(L + 1, D), dtype=np.uint8)),
                                 (cv / cv.sum(1, keepdims=True)).tolist(), rng.normal(0, 2, size=L).tolist(),
                                 rng.integers(0, A, size=L).tolist(),
                                 np.sign(rng.normal(size=L) * (rng.random(L) < 0.1)).astype(np.int64).tolist(),
                                 np.abs(rng.normal(size=L)).tolist(), [False] * L, list(range(L)), [None] * L, [1] * L),
                    ignore=None, terminal=True)
  torch.manual_seed(3)
  learner = fused_learner.FusedLearner(cfg, fused_learner.FusedFCNetwork(D, A, dev, cfg), replay_buffer=rb,
                                       search_network=net, use_graph=True, precision="bf16")
  main, side = torch.cuda.current_stream(), torch.cuda.Stream(device=dev)
  send_every = 25

  def learner_step():
    (obs, act, t_r, t_v, t_p), idx, isw = rb.sample_batch_device(False, ring=4)
    learner.update_weights(((obs, act, (t_r, t_v, t_p)), idx, isw))

  def hand_off():  # between two moves: the search never sees half-written weights
    main.wait_stream(side)
    learner.send_weights()
    side.wait_stream(main)

  with torch.cuda.stream(side):
    for _ in range(6):
      learner_step()
  torch.cuda.synchronize()
  hand_off()
  for _ in range(3):
    fs.run()
  barrier()
  n = max(20, min(args.steps, 100))
  ev = lambda: torch.cuda.Event(enable_timing=True)

  def run(with_search, with_learner):
    pairs, a, b = [], ev(), ev()
    a.record(side)
    for i in range(n):
      flush.zero_()
      if with_learner:
        with torch.cuda.stream(side):
          learner_step()
        if (i + 1) % send_every == 0:
          hand_off()
      if with_search:
        s, e = ev(), ev()
        s.record()
        fs.run()
        e.record()
        pairs.append((s, e))
    b.record(side)
    torch.cuda.synchronize()
    t = torch.tensor([sum(s.elapsed_time(e) for s, e in pairs), a.elapsed_time(b)], dtype=torch.float64, device=dev)
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    barrier()
    return t.tolist()

  ms_search_alone, _ = run(True, False)
  _, ms_learner_alone = run(False, True)
  ms_search, ms_learner = run(True, True)
  n_params = sum(p.numel() for p in learner.network.parameters())
  rate = lambda ms: world * G * S * n / (ms * 1e-3)
  return {
      "workload": "C4 search (%d games x %d sims, A=%d per GPU) + C3-shaped learner (B=%d, K=%d, td=%d, AdamW, FCNetwork; "
                  "FusedLearner: bf16 tensor-core forward / backward, bucketed gradient all-reduce overlapped with the "
                  "recurrent backward) on a side stream of the same GPU, one learner step enqueued per move, %d moves" % (G, S, A, B, K, T, n),
      "ranks": world,
      "collectives": ("gradient all-reduce of %d float32 per learner step + weight broadcast every %d steps (NCCL)"
                      % (n_params, send_every)) if world > 1 else "none at one rank (weights handed to the search network "
                                                                   "on the device every %d steps)" % send_every,
      "search_alone_expansions_per_s": rate(ms_search_alone),
      "learner_alone_steps_per_s": world * n / (ms_learner_alone * 1e-3),
      "search_expansions_per_s": rate(ms_search),
      "learner_steps_per_s": world * n / (ms_learner * 1e-3),
      "search_kept": ms_search_alone / ms_search,
      "learner_kept": ms_learner_alone / ms_learner,
      "weight_handoffs": n // send_every,
      "note": "search time = sum of per-move CUDA-event pairs (L2 flushed between moves, like the headline); learner "
              "time = first enqueue to last completion on the side stream (it includes the waits at the hand-offs); "
              "learner steps/s is the aggregate over ranks of data-parallel steps x ranks; together the learner is paced "
              "at one step per move, so its rate cannot exceed moves/s (alone it runs back to back)",
  }


def bench_learner(torch, _lib, dev, world, barrier):
  """Learner.update_weights (SURVEY.md section 8 f-4) on the C3 shape: B=512, K=5, A=4, 128-float
  observations, AdamW; device-resident synthetic batch.  Reports whole steps/s of FusedLearner (network forward +
  backward on the library's tensor-core kernels, the fused loss, the AdamW kernel, the gradient all-reduce at
  N > 1; max over ranks), the same step on the float32 kernels and on torch modules (cuBLAS) beside it, and the
  fused loss kernel alone against HBM."""
  import types
  import torch.distributed as dist
  from model_based_rl_b200 import learners
  B, K, A, E = 512, 5, 4, 128
  cfg = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=False,
                              no_target_transform=False, num_unroll_steps=K, optimizer="AdamW", lr_init=0.0008,
                              momentum=0.9, weight_decay=1e-4, clip_grad=0, lr_scheduler=None, norm_obs=False)
  g = torch.Generator(device=dev).manual_seed(7)
  r = lambda *shape: torch.rand(*shape, device=dev, generator=g)
  pol = r(B, K + 1, A)
  batch = ((r(B, E), torch.randint(0, A, (B, K), device=dev, generator=g),
            ((r(B, K + 1) < 0.1).float(), 4 * torch.randn(B, K + 1, device=dev, generator=g),
             pol / pol.sum(-1, keepdim=True))), None, r(B).double())
  from model_based_rl_b200 import fused_learner
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ms = {}
  for mode in ("torch_eager", "torch_graph", "fused_f32_graph", "fused_bf16_graph"):
    torch.manual_seed(11)
    if mode.startswith("torch"):
      lr = learners.Learner(cfg, learners.FCNetworkTrain(E, A, dev, cfg), use_graph=mode.endswith("graph"))
    else:
      lr = fused_learner.FusedLearner(cfg, fused_learner.FusedFCNetwork(E, A, dev, cfg), use_graph=True,
                                      precision=mode.split("_")[1])
    lr.send_weights()
    for _ in range(5):
      lr.update_weights(batch)
    barrier()
    steps = 100 if mode == "fused_bf16_graph" else 30
    a.record()
    for _ in range(steps):
      lr.update_weights(batch)
    b.record()
    torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms[mode] = float(t.item()) / steps
    del lr
  ms_step = ms["fused_bf16_graph"]
  # the loss kernel alone
  V = 31
  vl, rl, pl = torch.randn(K + 1, B, V, device=dev), torch.randn(K, B, V, device=dev), torch.randn(K + 1, B, A, device=dev)
  (_, _, (t_r, t_v, t_p)), _, w = batch
  outs = [torch.empty_like(vl), torch.empty_like(rl), torch.empty_like(pl), torch.empty(3, B, dtype=torch.float64, device=dev),
          torch.empty(3, dtype=torch.float64, device=dev), torch.empty(B, device=dev)]
  c = _lib.LossCfg(B, K, A, -15, 15, -15, 15, 0)
  lib, stream = _lib.load(), _lib.current_stream()

  def launch():
    _lib.check(lib.mz_unroll_loss(c, _lib.ptr(vl), _lib.ptr(rl), _lib.ptr(pl), _lib.ptr(t_v.contiguous()),
                                  _lib.ptr(t_r), _lib.ptr(t_p), _lib.ptr(w), *[_lib.ptr(o) for o in outs], stream),
               "mz_unroll_loss")
  for _ in range(5):
    launch()
  torch.cuda.synchronize()
  a.record()
  for _ in range(100):
    launch()
  b.record()
  torch.cuda.synchronize()
  us = a.elapsed_time(b) * 10.0
  logit_bytes = 4 * (vl.numel() + rl.numel() + pl.numel())
  alg = 2 * logit_bytes + 4 * (2 * B * (K + 1) + t_p.numel()) + 8 * B + 8 * 3 * B + 4 * B
  return {"steps_per_s": 1e3 / ms_step, "samples_per_s": world * B * 1e3 / ms_step, "ms_per_step": ms_step,
          "cuda_graph": True,
          "workload": "C3 learner step: B=512 per GPU, K=5, A=4, obs 128 f32, FCNetwork, AdamW; FusedLearner: forward / "
                      "backward on the library's tensor-core kernels (bf16 operands, f32 accumulation and master "
                      "weights: chain, heads, heads backward, chain backward = 4 launches), fused unroll loss, own AdamW "
                      "kernel; gradient all-reduce over %d rank(s)" % world,
          "variants_ms_per_step": {"fused_bf16_cuda_graph": ms["fused_bf16_graph"], "fused_f32_cuda_graph": ms["fused_f32_graph"],
                                   "torch_modules_cublas_f32_cuda_graph": ms["torch_graph"],
                                   "torch_modules_cublas_f32_eager": ms["torch_eager"]},
          "loss_kernel": {"us_per_launch": us, "algorithmic_bytes": alg, "achieved_gbs": alg / us / 1e3,
                          "launches": 2}}


def emit(line):
  """The ONE JSON line goes to the real stdout; everything else this process (or a library: NCCL prints
  its version banner on fd 1) writes to stdout lands on stderr."""
  _REAL_STDOUT.write(json.dumps(line) + "\n")
  _REAL_STDOUT.flush()


_REAL_STDOUT = sys.stdout


def main():
  global _REAL_STDOUT
  sys.stdout.flush()
  _REAL_STDOUT = os.fdopen(os.dup(1), "w")
  os.dup2(2, 1)
  args = parse()
  if args.impl == "reference":
    run_reference(args)
  else:
    run_b200(args)


if __name__ == "__main__":
  main()
