"""Run under torchrun on N GPUs: evaluates a sharded problem (NCCL exchange of the
gradient and cost) and checks every rank's result against an unsharded evaluation on the
same GPU.  Prints one line per rank."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT]
import numpy as np
import torch, torch.distributed as dist
import ceres_b200
from ceres_b200 import binding as B, problems as P

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
def fresh_nccl_id():
    """One ncclUniqueId per communicator, created on rank 0 and broadcast."""
    buf = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        buf.copy_(torch.frombuffer(bytearray(B.nccl_unique_id()), dtype=torch.uint8))
    dist.broadcast(buf, 0)
    return bytes(buf.cpu().numpy().tobytes())


scale = float(sys.argv[1]) if len(sys.argv) > 1 else 0.05
for fmt, kw in ((0, {}), (1, {"subset_manifold": True})):
    spec = P.bal_shape("L", scale=scale, **kw)
    full = B.CudaProblem(spec, jacobian_format=fmt, device=local)
    x = full.initial_state()
    ok, c0, r0, g0, j0 = full.evaluate(x)
    j0 = j0.copy()
    sh = B.CudaProblem(spec, jacobian_format=fmt, device=local, rank=rank, world_size=world, nccl_id=fresh_nccl_id())
    r = np.full(full.num_residuals, np.nan)
    sh.evaluate(x, out_residuals=r)  # first call pays NCCL's lazy initialisation
    ok, c, r, g, j = sh.evaluate(x, out_residuals=r)
    info = sh.shard_info()
    e_cost = abs(c - c0) / abs(c0)
    e_grad = np.max(np.abs(g - g0)) / np.max(np.abs(g0))
    rs = slice(info["residual_begin"], info["residual_end"])
    e_res = np.max(np.abs(r[rs] - r0[rs])) / np.max(np.abs(r0))
    e_jac = max(np.max(np.abs(j[gb:gb + ln] - j0[gb:gb + ln])) for gb, ln, _ in info["segments"]) / np.max(np.abs(j0))
    # device-resident linear algebra on the sharded Jacobian: column-space results are
    # summed over the ranks, so every rank must reproduce the unsharded numbers
    rng = np.random.default_rng(7)
    xv = rng.normal(size=full.num_effective_parameters)
    wv = rng.normal(size=full.num_residuals)
    rel = lambda a, b: float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))
    e_la = max(rel(sh.jacobian_multiply(wv, transpose=True), full.jacobian_multiply(wv, transpose=True)),
               rel(sh.jacobian_squared_column_norm(), full.jacobian_squared_column_norm()),
               rel(sh.jacobian_multiply(xv)[rs], full.jacobian_multiply(xv)[rs]))
    d2 = full.jacobian_squared_column_norm() / 1e4
    y0, s0 = full.cgnr_solve(d2, max_iterations=30, r_tolerance=-1, q_tolerance=-1)
    y1, s1 = sh.cgnr_solve(d2, max_iterations=30, r_tolerance=-1, q_tolerance=-1)
    e_cg = max(rel(y1, y0), abs(s1["jy_dot_b"] - s0["jy_dot_b"]) / abs(s0["jy_dot_b"]))
    print(f"rank {rank}/{world} fmt {fmt}: device linear algebra {e_la:.1e}, 30 CG iterations {e_cg:.1e} "
          f"({s1['ms'] / 30:.3f} ms/iteration sharded, {s0['ms'] / 30:.3f} unsharded) "
          f"{'OK' if e_la <= 1e-11 and e_cg <= 1e-8 else 'MISMATCH'}", flush=True)
    # blockdiag(J'J) is summed over the ranks as well
    y0, s0 = full.cgnr_solve(d2, max_iterations=30, r_tolerance=-1, q_tolerance=-1, preconditioner="jacobi")
    y1, s1 = sh.cgnr_solve(d2, max_iterations=30, r_tolerance=-1, q_tolerance=-1, preconditioner="jacobi")
    e_bj = max(rel(y1, y0), abs(s1["jy_dot_b"] - s0["jy_dot_b"]) / abs(s0["jy_dot_b"]))
    print(f"rank {rank}/{world} fmt {fmt}: 30 block-Jacobi CG iterations {e_bj:.1e} "
          f"{'OK' if e_bj <= 1e-8 else 'MISMATCH'}", flush=True)
    t = sh.timing()
    mode = {0: "single", 1: "nccl all-reduce", 2: "peer exchange"}[sh.exchange_mode()]
    # the other output combinations take the unfused path (PushExclusiveKernel)
    ok2, c2, r2, g2, _ = sh.evaluate(x, jacobian=False)
    e_grad = max(e_grad, np.max(np.abs(g2 - g0)) / np.max(np.abs(g0)))
    ok3, c3, *_ = sh.evaluate(x, gradient=False, jacobian=False)
    e_cost = max(e_cost, abs(c2 - c0) / abs(c0), abs(c3 - c0) / abs(c0))
    print(f"rank {rank}/{world} fmt {fmt}: exchange = {mode}; "
          f"cost {e_cost:.1e} grad {e_grad:.1e} res {e_res:.1e} jac {e_jac:.1e} "
          f"segments {len(info['segments'])} kernel {t['kernel_ms']:.3f} device {t['device_ms']:.3f} ms "
          f"{'OK' if max(e_cost, e_grad) <= 1e-10 and max(e_res, e_jac) <= 1e-12 else 'MISMATCH'}", flush=True)
    full.close(); sh.close()
dist.barrier()
dist.destroy_process_group()
