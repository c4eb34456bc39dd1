"""Multi-process covariance: frames sharded over the ranks (one process per GPU, torchrun) must
reproduce the single-GPU covariance — the camera block on every rank, each rank's board blocks
against its slice of the single-GPU blocks, the residual variance to 1e-12 relative.  Agreement bar
for the blocks: max(1e-10, 64 kappa_c eps) on the correlation-normalised blocks and their diagonals,
kappa_c the condition number of the camera block's correlation matrix (it underestimates that of the
equilibrated J^T J, which tests/test_covariance_gpu.py uses, by 10-100x on these rigs)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
from tscm_calib_b200 import capi, synth

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local = int(os.environ.get("LOCAL_RANK", rank))
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))


def normalised(S):
    d = np.sqrt(np.abs(np.diagonal(S, axis1=-2, axis2=-1)))
    return S / (d[..., :, None] * d[..., None, :])


ok = True
for cfg, frames, loss in ((2, 200, "none"), (5, 200, "huber"), (4, 600, "none")):
    sp = synth.config(cfg, num_frames=frames)
    opt = capi.default_options(loss_type=loss, loss_scale=1.0)
    prob, fr = synth.shard_frames(sp, rank, world)
    s = capi.Solver(prob, opt, device=local)
    capi.attach_ranks(s, rank, world)
    s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt[fr])
    cov = s.covariance()
    s.close()
    one = capi.Solver(sp.problem, opt, device=local)
    one.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    ref = one.covariance()
    one.close()
    ev = np.linalg.eigvalsh(normalised(ref.camera))
    tol = max(1e-10, 64.0 * ev[-1] / ev[0] * np.finfo(np.float64).eps)
    err = max(float(np.max(np.abs(normalised(cov.camera) - normalised(ref.camera)))),
              float(np.max(np.abs(np.diag(cov.camera) / np.diag(ref.camera) - 1))),
              float(np.max(np.abs(normalised(cov.board) - normalised(ref.board[fr])))),
              float(np.max(np.abs(np.diagonal(cov.board, axis1=1, axis2=2) /
                                  np.diagonal(ref.board[fr], axis1=1, axis2=2) - 1))))
    s2 = abs(cov.residual_variance / ref.residual_variance - 1)
    good = err <= tol and s2 < 1e-12 and cov.board.shape[0] == len(fr)
    ok = ok and good
    print(f"rank {rank} cfg{cfg} {loss} world={world}: block err {err:.2e} (bar {tol:.1e}) sigma2 rel {s2:.1e} "
          f"-> {'OK' if good else 'MISMATCH'}", flush=True)
flags = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(flags, op=dist.ReduceOp.MIN)
dist.barrier()
dist.destroy_process_group()
if rank == 0:
    print("DIST COVARIANCE", "PASS" if int(flags.item()) == 1 else "FAIL")
