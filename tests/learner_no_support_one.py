"""Diagnostics (not a test): step time of FusedLearner (bf16 and f32 kernels, CUDA graphs) against learners.Learner
(torch modules, CUDA graph) on the C3 shape (B = 512, K = 5, A = 4, 128 features) for a support network and for
`--no_support` networks trained with the MSE and the Huber scalar loss, all in one process.

  python tests/learner_no_support_one.py [optimizer]
"""
import os, sys, time, types
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from model_based_rl_b200 import fused_learner, learners
dev = torch.device("cuda:0")
B, K, A, E = 512, 5, 4, 128
optimizer = sys.argv[1] if len(sys.argv) > 1 else "AdamW"
g = torch.Generator(device=dev).manual_seed(7)
r = lambda *shape: torch.rand(*shape, device=dev, generator=g)
pol = r(B, K + 1, A)
batch = ((r(B, E), torch.randint(0, A, (B, K), device=dev, generator=g),
          ((r(B, K + 1) < 0.1).float(), 4 * torch.randn(B, K + 1, device=dev, generator=g), pol / pol.sum(-1, keepdim=True))),
         None, r(B).double())
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
print(torch.cuda.get_device_name(dev))
for scalar_loss in (None, "MSE", "Huber"):
  cfg = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=scalar_loss is not None,
                              scalar_loss=scalar_loss or "MSE", no_target_transform=False, num_unroll_steps=K,
                              optimizer=optimizer, lr_init=0.0008, momentum=0.9, weight_decay=1e-4, clip_grad=0,
                              lr_scheduler=None, norm_obs=False)
  for name in ("bf16_graph", "f32_graph", "torch_graph"):
    if name == "torch_graph":
      lr = learners.Learner(cfg, learners.FCNetworkTrain(E, A, dev, cfg), use_graph=True)
    else:
      lr = fused_learner.FusedLearner(cfg, fused_learner.FusedFCNetwork(E, A, dev, cfg), precision=name.split("_")[0])
    for _ in range(5):
      lr.update_weights(batch)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    a.record()
    n = 50
    for _ in range(n):
      lr.update_weights(batch)
    b.record()
    torch.cuda.synchronize()
    print("%-8s %-12s %8.1f us/step device, %8.1f us/step wall, %7.0f steps/s, loss %s" %
          (scalar_loss or "support", name, a.elapsed_time(b) * 1e3 / n, (time.perf_counter() - t0) * 1e6 / n,
           n / (a.elapsed_time(b) * 1e-3), lr.last_losses.cpu().numpy().round(4)))
