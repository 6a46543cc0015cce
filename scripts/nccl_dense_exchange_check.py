"""Multi-rank check of the device-side pooled DENSE adaptor (WelfordCov; run under torchrun, one rank per GPU):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29521 scripts/nccl_dense_exchange_check.py
Every rank feeds its own (theta, alpha) per iteration to ahmc_adapt_exchange_f64 over an ahmc_comm (one NCCL all-gather of the
(2 + 2D + D^2)-double records inside the C ABI); eps, M^-1 and its factor U must equal the host-side pooled adaptors fed the
rank-ordered merge of all ranks' K5 + K5b records (exchanged here through torch.distributed as the independent path), and be
bit-identical on every rank."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

import ahmc_b200 as A
from ahmc_b200 import adaptation as ad

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
D, N, n_adapts = 29, 150 + 23 * rank, 30  # ragged: every rank owns a different number of chains
windows = (5, 4, 6)
comm = ad.Comm.from_torch_distributed(local)
assert comm is not None and comm.nranks == world
dev_ad = ad.PooledDeviceAdaptor(local, D, N, n_adapts, eps0=0.11, init_buffer=windows[0], term_buffer=windows[1],
                                window_size=windows[2], n_min=3, dense=True)
host = ad.StanHMCAdaptor(ad.WelfordCov(D, n_min=3), ad.NesterovDualAveraging(0.8, 0.11), *windows)
host.initialize(n_adapts)
rng = np.random.default_rng(200 + rank)
Lc = np.tril(np.random.default_rng(7).normal(size=(D, D))) * 0.3 + np.eye(D)
worst = 0.0
for i in range(1, n_adapts + 1):
    th = torch.as_tensor(rng.normal(size=(N, D)) @ Lc.T + 0.1 * rank, device=dev)
    al = torch.as_tensor(rng.uniform(0.2, 1.3, N), device=dev)
    dev_ad.exchange(th, al, comm, None, flags=0)
    head = A.adapt_summary(th, al)
    rec = torch.cat([head, A.adapt_cov(th, head[2:2 + D]).reshape(-1)])
    recs = [torch.empty_like(rec) for _ in range(world)]
    dist.all_gather(recs, rec)
    merged = ad.merge_records([r.cpu().numpy() for r in recs], "cov")
    host.adapt(merged)
    if i == n_adapts:
        host.finalize()
    s = dev_ad.state()
    assert s["iteration"] == i and s["failed_iteration"] == 0
    assert np.abs(s["merged_record"] - merged).max() <= 1e-12 * np.abs(merged).max(), (rank, i)
    assert abs(s["eps"] - host.eps) <= 1e-12 * host.eps, (rank, i, s["eps"], host.eps)
    assert np.abs(s["Minv"] - host.Minv).max() <= 1e-12 * np.abs(host.Minv).max(), (rank, i)
    U = s["cholU"]
    assert np.abs(U - np.linalg.cholesky(s["Minv"]).T).max() <= 1e-10 * np.abs(U).max(), (rank, i)
    worst = max(worst, abs(s["eps"] - host.eps) / host.eps)
    # bit-identical on every rank
    mine = torch.as_tensor(np.concatenate([[s["eps"]], s["Minv"].reshape(-1), U.reshape(-1)]), device=dev)
    allv = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allv, mine)
    assert all(torch.equal(allv[0], v) for v in allv), (rank, i)
assert not np.array_equal(s["Minv"], np.eye(D))
dev_ad.destroy()
comm.destroy()
dist.barrier()
if rank == 0:
    print(f"nccl dense exchange ok: {world} ranks, {n_adapts} iterations, max rel eps error vs host adaptors {worst:.2e}, "
          "eps / M^-1 / U identical on all ranks")
dist.destroy_process_group()
