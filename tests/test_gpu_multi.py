"""2-GPU NCCL test of the sharded commit (skipped on single-GPU boxes): bit-exact cap == single-GPU commit of the whole trace."""
import os
import pathlib
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
pytestmark = pytest.mark.gpu
LOG_H, W, CAP_H = 12, 100, 3


def _worker(rank, world, port, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
        from oracle import p3_oracle as O
        from plonky3_b200 import _lib
        from plonky3_b200.distributed import GpuBackend, column_block, column_starts, commit_bit_exact, commit_column_blocks
        from plonky3_b200.field import KoalaBear as f
        from plonky3_b200.gpu import Gpu
        from plonky3_b200.poseidon2 import default_poseidon2
        gpu = Gpu(rank)
        for w in (16, 24):
            default_poseidon2(f, w).upload(gpu)
        be = GpuBackend(gpu, f, _lib.HASH_POSEIDON2_W24, 1)
        full = O.random_matrix(f.id, 1 << LOG_H, W, seed=9)
        widths = [column_block(W, world, g)[1] - column_block(W, world, g)[0] for g in range(world)]
        c0, c1 = column_block(W, world, rank)
        local = torch.from_numpy(np.ascontiguousarray(full[:, c0:c1]).view(np.int32)).cuda()
        cap, recv, layers = commit_bit_exact(be, local, widths, CAP_H)
        roots, _, _ = commit_column_blocks(be, local)
        ohs = O.poseidon2_hasher(O.default_perm(f.id, 24), O.default_perm(f.id, 16))
        lde_full = O.coset_lde_batch(f.id, full, 1, f.generator, True)
        exp_cap = O.merkle_cap(O.merkle_tree(ohs, [lde_full]), CAP_H)
        ok = np.array_equal(cap.cpu().numpy().view(np.uint32), exp_cap)
        exp_root = O.merkle_tree(ohs, [O.coset_lde_batch(f.id, full[:, c0:c1], 1, f.generator, True)])[-1][0]
        ok2 = np.array_equal(roots[rank].cpu().numpy().view(np.uint32), exp_root)
        # peer-memory mode (no NCCL on the data path): IPC-mapped row blocks, LDE column chunks copied into them on the copy engines
        from plonky3_b200.distributed import PeerGroup
        H = 2 << LOG_H
        grp = PeerGroup(gpu, H // world, W)
        a0, a1 = column_block(W, world, rank, align=8)
        loc8 = torch.from_numpy(np.ascontiguousarray(full[:, a0:a1]).view(np.int32)).cuda()
        for _ in range(3):
            pcap, players, ph = grp.commit(f, _lib.HASH_POSEIDON2_W24, loc8, column_starts(W, world, align=8), 1, CAP_H, phases=True)
        ok = ok and np.array_equal(pcap, exp_cap)
        rows = H // world
        ok = ok and np.array_equal(grp.row_block_dense().cpu().numpy().view(np.uint32), lde_full[rank * rows:(rank + 1) * rows])
        dist.barrier()
        grp.close()
        q.put((rank, bool(ok), bool(ok2), ""))
        dist.destroy_process_group()
    except Exception as e:
        q.put((rank, False, False, repr(e)))


def test_sharded_commit_nccl():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + (os.getpid() % 300)
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs: p.start()
    res = [q.get(timeout=300) for _ in range(world)]
    for p in procs: p.join(timeout=60)
    for rank, ok, ok2, err in res:
        assert ok and ok2, f"rank {rank}: cap ok={ok} block root ok={ok2} {err}"
