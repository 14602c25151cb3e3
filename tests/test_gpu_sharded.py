"""The row-sharded multi-GPU commit (p3gpu_coset_lde_batch_sharded_dev / p3gpu_commit_sharded_dev: peer-memory stores from
the LDE's last pass, flag barrier, peer all-gather of the cap slices) exercised on whatever the box has.

  * test_sharded_lde_scatters_row_blocks: the store addressing of the sharded LDE, `world` ranks simulated inside this process
    on cuda:0 (no barrier involved);
  * test_sharded_commit_equals_single_commit: the full commit with one PROCESS per rank — CUDA IPC mappings, flag barrier,
    peer all-gather — with every rank on cuda:0 when the box has one GPU (the driver's test box; the GPU time-slices between
    the processes) and one GPU per rank when it has enough (tests/test_gpu_multi.py additionally compares with the NCCL path)."""
import numpy as np
import pytest
import torch

from oracle import p3_oracle as O

from plonky3_b200 import _lib
from plonky3_b200.distributed import PeerGroup, column_block, column_starts
from plonky3_b200.field import BabyBear, KoalaBear
from plonky3_b200.gpu import Gpu
from plonky3_b200.poseidon2 import default_poseidon2

pytestmark = pytest.mark.gpu


def host(t):
    return t.cpu().numpy().view(np.uint32)


def _gpus(n):
    out = []
    for _ in range(n):
        g = Gpu(0)
        for f in (BabyBear, KoalaBear):
            for w in (16, 24):
                default_poseidon2(f, w).upload(g)
        out.append(g)
    return out


@pytest.mark.parametrize("mode", ["dma", "staged", "fused"])
@pytest.mark.parametrize("f,log_h,w,world", [(KoalaBear, 12, 100, 2), (BabyBear, 13, 72, 4), (KoalaBear, 14, 328, 8), (KoalaBear, 15, 200, 2)])
def test_sharded_lde_scatters_row_blocks(f, log_h, w, world, mode, monkeypatch):
    """Every rank's column-block LDE lands in the right rows/columns of every rank's row block — both exchange variants:
    `staged` (column chunks into a staging buffer + coalesced push kernel on a second stream) and `fused` (the last pass of the
    transform stores its tiles straight into the owners' row blocks); `dma` (default) = staged with 2-D peer copies."""
    monkeypatch.setenv("P3GPU_SHARD_MODE", mode)
    gpus = _gpus(world)
    H = 2 << log_h
    groups = PeerGroup.simulate(gpus, H // world, w)
    full = O.random_matrix(f.id, 1 << log_h, w, seed=11)
    exp = O.coset_lde_batch(f.id, full, 1, f.generator, bitrev_out=True)
    for q, grp in enumerate(groups):
        c0, c1 = column_block(w, world, q, align=8)
        local = torch.from_numpy(np.ascontiguousarray(full[:, c0:c1]).view(np.int32)).cuda()
        grp.lde_sharded(f, local, 1, f.generator, c0)
        torch.cuda.synchronize()
    got = np.concatenate([host(grp.rows_tensor()) for grp in groups], axis=0)
    assert np.array_equal(got, exp)


# ---- the full sharded commit: one PROCESS per rank (exactly the production topology: CUDA IPC mappings, flag barrier, peer
# all-gather), all ranks on cuda:0 when the box has a single GPU (the driver's test box), one GPU per rank otherwise.  The
# bootstrap exchange of the IPC handles uses a gloo group (NCCL refuses two ranks on one device; the data path needs neither).
CASES = [("p2w24", 1, 12, 100, 3), ("p2w24", 1, 12, 100, 0), ("p2w16", 0, 13, 40, 1), ("keccak", 0, 12, 60, 3), ("p2w24", 1, 13, 164, 5)]


def _rank_main(rank, world, port, q):
    try:
        import os
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        import torch.distributed as dist
        ndev = torch.cuda.device_count()
        device = rank if ndev >= world else 0
        torch.cuda.set_device(device)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        from plonky3_b200.field import FIELDS
        gpu = Gpu(device)
        for fld in (BabyBear, KoalaBear):
            for wd in (16, 24):
                default_poseidon2(fld, wd).upload(gpu)
        ok, msg = True, ""
        for kind, fid, log_h, w, cap_height in CASES:
            f = FIELDS[fid]
            if (2 << log_h) // world < 1024:
                continue
            hash_kind = {"p2w16": _lib.HASH_POSEIDON2_W16, "p2w24": _lib.HASH_POSEIDON2_W24, "keccak": _lib.HASH_KECCAK}[kind]
            ohs = O.keccak_hasher() if kind == "keccak" else O.poseidon2_hasher(O.default_perm(f.id, 24 if kind == "p2w24" else 16), O.default_perm(f.id, 16))
            H = 2 << log_h
            grp = PeerGroup(gpu, H // world, w, timeout_s=60.0)
            full = O.random_matrix(f.id, 1 << log_h, w, seed=5)
            elde = O.coset_lde_batch(f.id, full, 1, f.generator, bitrev_out=True)
            olayers = O.merkle_tree(ohs, [elde])
            exp_cap = O.merkle_cap(olayers, cap_height)
            c0, c1 = column_block(w, world, rank, align=8)
            local = torch.from_numpy(np.ascontiguousarray(full[:, c0:c1]).view(np.int32)).cuda()   # may be EMPTY: more ranks than column units
            for _ in range(2):                               # twice: the epoch counter and the row blocks are reused
                cap, layers, ph = grp.commit(f, hash_kind, local, column_starts(w, world, align=8), 1, cap_height, phases=True)
            rows = H // world
            good = np.array_equal(cap, exp_cap) and len(ph) == 4
            good = good and np.array_equal(host(grp.row_block_dense()), elde[rank * rows:(rank + 1) * rows])
            for k, lay in enumerate(layers):                 # my sub-tree = slice `rank` of the global tree's lower layers
                n = max(rows >> k, 1)
                good = good and np.array_equal(host(lay)[:n], olayers[k][rank * n:(rank + 1) * n])
            if not good:
                ok, msg = False, f"mismatch in case {(kind, fid, log_h, w, cap_height)}"
            dist.barrier()
            grp.close()
        q.put((rank, ok, msg))
        dist.destroy_process_group()
    except Exception as e:                                   # noqa: BLE001 — surfaced by the parent
        q.put((rank, False, repr(e)))


@pytest.mark.parametrize("world", [2, 4, 8])
def test_sharded_commit_equals_single_commit(world):
    """cap of the sharded commit (on every rank) == cap of TwoAdicFriPcs::commit on the whole trace (oracle); every rank's row
    block == its rows of the full LDE; every rank's sub-tree == its slice of the oracle's tree."""
    import os
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29700 + (os.getpid() % 200) + world
    procs = [ctx.Process(target=_rank_main, args=(r, world, port, q)) for r in range(world)]
    for p in procs: p.start()
    res = [q.get(timeout=600) for _ in range(world)]
    for p in procs: p.join(timeout=60)
    assert all(ok for _, ok, _ in res), "; ".join(f"rank {r}: {m}" for r, ok, m in sorted(res) if not ok)
