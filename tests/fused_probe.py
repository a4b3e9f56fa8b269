"""Bring-up / timing probe of the fused search kernel (not a pytest): python tests/fused_probe.py"""
import sys, types, time
import numpy as np
import torch
sys.path.insert(0, ".")
from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict



def cfg_for(S, A):
  return types.SimpleNamespace(
      num_simulations=S, action_space=A, two_players=False, discount=0.997, pb_c_base=19652, pb_c_init=1.25,
      init_value_score=0.0, known_bounds=[None, None], root_exploration_fraction=0.25,
      value_support=[-15, 15], reward_support=[-15, 15], no_support=False, no_target_transform=False)


def compare(G, S, A=18, D=128):
  cfg = cfg_for(S, A)
  net = FCNetwork(D, A, "cuda", cfg)
  net.load_weights(random_state_dict(D, A))
  rng = np.random.default_rng(1)
  obs = rng.random((G, D)).astype(np.float32)
  noise, u, temp = rng.dirichlet([0.25] * A, size=G), rng.random(G), np.ones(G)
  res = []
  for fused in (False, True):
    fs = FCSearch(cfg, net, G, use_graph=False, num_streams=1, fused=fused)
    fs.enable_record()
    r = fs.search_host(obs, noise, u, temp)
    torch.cuda.synchronize()
    res.append((fs, [t.clone() for t in r]))
  (fa, ra), (fb, rb) = res
  ok = True
  for i, name in enumerate(("value", "reward", "logits")):
    x, y = fa.record[i], fb.record[i]
    if not torch.equal(x, y):
      ok = False
      bad = (x != y).reshape(S, G, -1).any(-1)
      s0 = int(bad.any(1).nonzero()[0])
      print("  net %s differs first at sim %d in %d games, max abs %.3g" % (name, s0, int(bad[s0].sum()),
                                                                       float((x - y).abs().max())))
  for i, name in enumerate(("parent", "action", "depth")):
    x, y = fa.trace[i], fb.trace[i]
    if not torch.equal(x, y):
      ok = False
      bad = (x != y)
      s0 = int(bad.any(1).nonzero()[0])
      g0 = int(bad[s0].nonzero()[0])
      print("  trace %s differs first at sim %d (%d games), e.g. game %d: %d vs %d" % (
          name, s0, int(bad[s0].sum()), g0, int(x[s0, g0]), int(y[s0, g0])))
  for name, x, y in (("visits", fa.visits, fb.visits), ("root_value", ra[1], rb[1]), ("actions", ra[0], rb[0]),
                     ("minmax", fa.minmax, fb.minmax)):
    if not torch.equal(x, y):
      ok = False
      print("  %s differs in %d entries" % (name, int((x != y).sum())))
  print("compare G=%d S=%d A=%d: %s (err flag %d)" % (G, S, A, "IDENTICAL" if ok else "MISMATCH",
                                                      int(fb.fused.error_flag.item())))
  return ok


def timing(G, S=50, A=18, D=128, moves=20):
  cfg = cfg_for(S, A)
  net = FCNetwork(D, A, "cuda", cfg)
  net.load_weights(random_state_dict(D, A))
  rng = np.random.default_rng(2)
  obs = rng.random((G, D)).astype(np.float32)
  noise, u, temp = rng.dirichlet([0.25] * A, size=G), rng.random(G), np.ones(G)
  for fused, streams in ((False, 4), (True, 1)):
    fs = FCSearch(cfg, net, G, use_graph=True, num_streams=streams, fused=fused)
    fs.search_host(obs, noise, u, temp)
    for _ in range(3):
      fs.run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(moves):
      fs.run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / moves
    print("timing G=%d fused=%s: %.3f ms/move  %.1f M expansions/s" % (G, fused, ms, G * S / ms / 1e3))
    if fused:
      fs.fused.enable_timeline()
      fs._fused_plan_key = None
      fs.graph = None
      fs.use_graph = False
      fs.run()
      torch.cuda.synchronize()
      k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      import ctypes as C
      from model_based_rl_b200 import _lib
      plan = fs.fused.plan(fs, fs.use_noise, fs.noise_frac, C.c_void_p(torch.cuda.current_stream().cuda_stream))
      names_ = [fn.__name__ for fn, _ in plan]
      for fn, args in plan:
        if fn.__name__ == "mz_fc_search":
          k0.record()
        fn(*args)
        if fn.__name__ == "mz_fc_search":
          k1.record()
      torch.cuda.synchronize()
      tl = fs.fused.timeline.cpu().numpy().astype(np.int64)
      t0 = tl[0]
      print("   launches of a move: %s" % names_)
      print("   mz_fc_search by CUDA events %.1f us; block 0: entry -> exit %d cycles = %.1f us by globaltimer (%.0f MHz), "
            "entry -> set-up done %d cycles, last stamp -> exit %d cycles" % (
                k0.elapsed_time(k1) * 1e3, t0[28] - t0[27], (t0[30] - t0[29]) / 1e3,
                (t0[28] - t0[27]) / max(1, (t0[30] - t0[29])) * 1e3, t0[13] - t0[27], t0[28] - tl[-1, 15]))
      base = tl[:, 0:1]
      names = {1: "descent", 2: "a1 sent", 3: "a1 ready", 4: "dyn d2", 5: "dyn out", 6: "a3 ready", 7: "pred d2",
               8: "pred out"}
      rel = tl - base
      med = np.median(rel[5:], axis=0)
      print("  timeline (cycles after the start of a simulation's descent, median over sims 5..):")
      print("   ", ", ".join("%s %d" % (names[k], med[k]) for k in sorted(names)))
      print("   kernel body (after set-up) %d cycles = %.1f x the median sim period; root set-up %d; last backup + root stats %d" % (
          tl[-1, 15] - tl[0, 13], (tl[-1, 15] - tl[0, 13]) / np.median(tl[1:, 0] - tl[:-1, 0]), tl[0, 14] - tl[0, 13],
          tl[-1, 15] - tl[-1, 12]))
      nxt = tl[1:, 0] - tl[:-1, 0]
      print("   sim period median %d cycles" % np.median(nxt))
      d = lambda a, b: int(np.median((tl[:, a] - tl[:, b])[5:]))
      print("   descent: reset %d | issue loads %d | rank items %d | winners %d | chase %d" % (
          int(np.median((tl[1:, 16] - tl[:-1, 11])[5:])), d(17, 16), d(18, 17), d(19, 18), d(20, 19)))
      print("   expand+backup: early loads %d | exp + prior sum %d | priors %d | top x2 + meta %d | backup %d | minmax %d" % (
          d(22, 10), d(23, 22), d(24, 23), d(25, 24), d(26, 25), d(11, 26)))
      print("   next sim: wait for outputs %d, expand+backup %d, descent %d" % (
          np.median((tl[:-1, 10] - tl[1:, 0])[5:]), np.median((tl[:-1, 11] - tl[:-1, 10])[5:]),
          np.median((tl[1:, 1] - tl[:-1, 11])[5:])))

if __name__ == "__main__":
  ok = compare(128, 4) and compare(300, 50)
  if ok:
    compare(257, 30, A=4, D=8)
    timing(4096)
    timing(16384, moves=5)
