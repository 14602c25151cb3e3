#!/usr/bin/env python3
"""bench.py — the driver's benchmark contract for the Plonky3 hot path on B200.

Primary workload = BASELINE.json configs[1]: coset_lde_batch, KoalaBear, 2^20 rows x 100 cols per GPU, blowup 2
(added_bits = 1, shift = GENERATOR), output in the committed (bit-reversed-row) layout.  metric = NTT Gelem/s of LDE
output.  A "step" is one LDE of one synthetic matrix (uniform field elements, seeded).

  value       device-resident throughput: input already in HBM, CUDA events on the launching stream, K steps.
              Input (419 MB) + output (839 MB) exceed the 126 MB L2, so no L2 flush is needed between iterations.
              N > 1 (torchrun): WEAK scaling of the same metric with the exchange in the timed region — the N ranks hold the N
              column blocks (100 columns each) of ONE 2^20 x 100N matrix; every step each rank runs the LDE of its block, whose
              last pass stores every tile into the ROW block of the rank that owns those rows (peer memory over NVLink: the
              all-to-all that re-shards column blocks into row blocks, SURVEY 8e), followed by the flag barrier that makes the
              step complete on all ranks.  value = N x 209,715,200 elements / max-over-ranks time.
  e2e         the same metric through the reference-facing C-ABI call p3gpu_coset_lde_batch with HOST (pinned, NUMA-local)
              buffers, ONE call at a time: H2D of the input and D2H of the result are inside the timed region.  The
              2-calls-in-flight figure (two contexts, full-duplex PCIe) is reported as a note.
  roofline    HBM roofline of the NTT pass kernel: algorithmic bytes of one LDE (read input once + write output once,
              SURVEY.md 8d: 1,258,291,200 B) / device time of the step (all launches of a step are the same kernel), plus the
              integer-issue floor the kernel is actually bound by.
  cpu_baseline the oracle port (OpenMP C restatement, oracle/p3_oracle.c) on the host cores, bounded sample.
  sharded_commit  (every N) STRONG scaling of ONE BASELINE config-5 trace commit (KoalaBear 2^20 x 1312, blowup 2, Poseidon2-24
              leaves, cap_height 3) column-sharded over the N ranks, per-phase device ms, in three modes: `peer` (the product:
              p3gpu_commit_sharded_dev — LDE with fused peer stores, flag barrier, row-sharded hashing, peer all-gather of the
              cap), `nccl` (baseline: LDE -> NCCL all_to_all -> hashing -> NCCL all_gather) and `column_blocks` (BASELINE's
              independent commitment per shard + one all-gather of roots).  Every rank asserts cap == the N=1 cap.
  others      (N=1 only) the remaining single-GPU BASELINE configs timed the same way.

--steps K times exactly K steps of the primary workload (`value`, `ms_per_step`, `roofline`); its warm-up is max(--warmup, 3)
steps.  The other legs use their own counts: e2e min(max(K, 4), 10) calls, --impl reference min(K, 5) steps, and the secondary
workloads and sharded_commit fixed counts sized to their run time.

--impl reference: times the reference's CPU algorithm (the oracle port — the reference is Rust and cannot be built in this
image) on the same metric with all physical cores; rank 0 only under torchrun.

--dump-outputs DIR: after the timed steps of the primary workload, writes what its last step computed (the LDE output, raw
Montgomery words as float64, which holds them exactly) for a fixed, seeded sample of DUMP_ROWS rows, as DIR/coset_lde.npy, and
the sampled row indices as DIR/coset_lde_rows.npy.  Inputs are seeded, so two builds run with the same arguments can be compared
file for file.  Under torchrun rank r writes DUMP_ROWS / N^2 rows of its own row block (each row 100N columns wide) as
coset_lde_rank<r>.npy, so the N ranks together write as many elements as one GPU does.
"""
import argparse
import json
import os
import pathlib
import subprocess
import sys
import threading
import time

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

LOG_H, W, ADDED_BITS = 20, 100, 1
ALG_BYTES = ((1 << LOG_H) * W + (1 << (LOG_H + ADDED_BITS)) * W) * 4       # 1,258,291,200
OUT_ELEMS = (1 << (LOG_H + ADDED_BITS)) * W                                   # 209,715,200
BUTTERFLIES = 3 * LOG_H * (1 << (LOG_H - 1)) * W                              # 3.146e9 (iDFT + two coset DFTs)
T_LOG_H, T_W, T_CAP = 20, 1312, 3                                             # config 5 trace
DUMP_ROWS = 1 << 16                   # 2^16 rows x 100 cols of float64 = 52 MB over all ranks, under the 64 MB a dump may take


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-others", action="store_true", help="skip the secondary workloads")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sharded", action="store_true", help="skip the config-5 sharded commit")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-pointer leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the primary workload's last output to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def dump_outputs(out_dir, rows, name, count):
    """Seeded sample of `count` rows of `rows` (a CUDA int32 tensor) as float64 .npy files; the sample depends only on the
    row counts, so runs with the same arguments sample the same rows."""
    import numpy as np
    import torch
    d = pathlib.Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    n = rows.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, count), replace=False))
    sample = rows.index_select(0, torch.from_numpy(idx).to(rows.device)).cpu().numpy()
    np.save(d / f"{name}.npy", sample.astype(np.float64))
    np.save(d / f"{name}_rows.npy", idx.astype(np.float64))


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock + throttle reasons DURING the timed region (NVML, ~1 kHz; falls back to nvidia-smi)."""

    def __init__(self, idx=0):
        self.idx, self.samples, self.reasons, self.stop = idx, [], set(), False
        self.max_mhz = None
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self.idx)
            self.max_mhz = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
            bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
            while not self.stop:
                self.samples.append(float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)))
                try:
                    r = N.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = N.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for n, b in bits.items():
                    if r & b:
                        self.reasons.add(n)
                time.sleep(0.001)
            return
        except Exception:
            pass
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0])); self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower() == "active":
                        self.reasons.add(n)
            except Exception:
                pass

    def __enter__(self): self.t.start(); time.sleep(0.05); self.samples.clear(); return self
    def __exit__(self, *a): self.stop = True; self.t.join(timeout=6)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------ host topology
def bind_to_gpu_numa(idx):
    """Pin this process to the CPUs that are NUMA-local to GPU idx, so that pinned host buffers allocated afterwards (first
    touch) and the threads that drive the copies sit on the socket the GPU hangs off.  Returns a description for the JSON."""
    try:
        import pynvml as N
        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(idx)
        n_cpu = os.cpu_count() or 1
        words = N.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = [64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1 and 64 * i + b < n_cpu]
        if cpus:
            os.sched_setaffinity(0, cpus)
            node = None
            try:
                bus = N.nvmlDeviceGetPciInfo(h).busId
                bus = bus.decode() if isinstance(bus, bytes) else bus
                node = int(pathlib.Path(f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node").read_text())
            except Exception:
                pass
            return {"cpus": len(cpus), "first_cpu": cpus[0], "numa_node": node}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}
    return {"cpus": 0}


# ------------------------------------------------------------------------------------------------ CPU (oracle) legs
def _omp_setup():
    """One OpenMP thread per PHYSICAL core, spread over the sockets, set UNCONDITIONALLY: torch.distributed.run exports
    OMP_NUM_THREADS=1 to its workers, which must not leak into the CPU reference (measured on the bench host, 2 x Xeon 8562Y+,
    64 cores / 128 threads: one thread per physical core is 2x faster than 128 threads)."""
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or os.cpu_count() or 1
    except Exception:
        phys = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(phys)
    os.environ["OMP_PROC_BIND"] = "spread"
    os.environ.pop("OMP_PLACES", None)
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))      # undo any inherited pinning: the reference may use every core
    except Exception:
        pass
    return phys


def _native_oracle():
    """The oracle compiled with -march=native for THIS host (the in-tree build may come from another CPU, and an illegal
    instruction would kill the bench), in a temporary directory: the bench writes nothing into the tree."""
    import tempfile
    from oracle import p3_oracle as O
    with tempfile.TemporaryDirectory() as d:
        O.lib(O.build(native=True, out=pathlib.Path(d) / "libp3oracle.so"))    # stays mapped after the directory is gone
    return O


def cpu_lde_throughput(budget_s=15.0):
    """Oracle port of coset_lde_batch on a bounded column sample of the same workload.  Returns (Gelem/s, cores, sample)."""
    cores = _omp_setup()
    O = _native_oracle()
    f = 1
    m = O.random_matrix(f, 1 << LOG_H, 4, seed=1)
    t0 = time.time(); O.coset_lde_batch(f, m, ADDED_BITS, O.generator(f)); t4 = time.time() - t0
    cols = int(max(4, min(W, 4 * budget_s / max(t4, 1e-3))))
    cols -= cols % 4
    m = O.random_matrix(f, 1 << LOG_H, cols, seed=1)
    t0 = time.time(); out = O.coset_lde_batch(f, m, ADDED_BITS, O.generator(f)); dt = time.time() - t0
    return out.size / dt / 1e9, cores, f"coset_lde_batch KoalaBear 2^{LOG_H} x {cols} of {W} cols, blowup 2, {dt:.1f} s, OpenMP {cores} threads"


def cpu_hash_legs():
    """CPU legs of the Merkle configs on bounded row samples (the oracle port): config 3 (Poseidon2-16 over 100 columns),
    config 4 leaves (Keccak over 300 columns) and config 5 leaves (Poseidon2-24 over 1312 columns)."""
    cores = _omp_setup()
    from oracle import p3_oracle as O
    out = {}
    for name, f, hs, rows, w, perms_per_row in [
            ("config3_poseidon2_w16_kb_x100", 1, O.poseidon2_hasher(O.default_perm(1, 16), O.default_perm(1, 16)), 1 << 16, 100, 13),
            ("config4_keccak_bb_x300", 0, O.keccak_hasher(), 1 << 16, 300, 9),
            ("config5_poseidon2_w24_kb_x1312", 1, O.poseidon2_hasher(O.default_perm(1, 24), O.default_perm(1, 16)), 1 << 14, 1312, 82)]:
        m = O.random_matrix(f, rows, w, seed=1)
        t0 = time.time(); O.merkle_tree(hs, [m]); dt = time.time() - t0
        out[name] = {"rows": rows, "s": dt, "Mperm_per_s": (rows * perms_per_row + rows - 1) / dt / 1e6, "cores": cores, "kind": "port"}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = _omp_setup()
    O = _native_oracle()
    f = 1
    cols = W if cores >= 16 else 16          # full workload on a many-core host, a 16-column sample on small hosts
    m = O.random_matrix(f, 1 << LOG_H, cols, seed=1)
    for _ in range(min(args.warmup, 1)):
        O.coset_lde_batch(f, m, ADDED_BITS, O.generator(f))
    steps = max(1, min(args.steps, 5))
    t0 = time.time()
    for _ in range(steps):
        out = O.coset_lde_batch(f, m, ADDED_BITS, O.generator(f))
    dt = (time.time() - t0) / steps
    v = out.size / dt / 1e9
    sample = f"coset_lde_batch KoalaBear 2^{LOG_H} x {cols} of {W} cols per step (bounded sample), OpenMP {cores} threads"
    print(json.dumps({
        "impl": "reference", "metric": "coset_lde_batch output Gelem/s (KoalaBear 2^20 x 100 per GPU, blowup 2)", "value": v, "unit": "Gelem/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": dt * 1e3 * (W / cols),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (31-bit Montgomery)", "data": "synthetic",
        "config": {"workload": "coset_lde_batch KoalaBear 2^20 x 100, added_bits 1, shift GENERATOR, bit-reversed rows (BASELINE configs[1])"},
        "cpu_baseline": {"value": v, "unit": "Gelem/s", "cores": cores, "kind": "port", "sample": sample, "omp_threads": int(os.environ["OMP_NUM_THREADS"])},
        "e2e": {"value": v, "unit": "Gelem/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference is Rust (no toolchain in this image): this is the OpenMP C restatement oracle/p3_oracle.c; ms_per_step is scaled to 100 columns; "
                "the CPU arm is one host's cores whatever --gpus is (one matrix per step)",
    }))


# ------------------------------------------------------------------------------------------------ GPU legs
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from plonky3_b200 import _lib
    from plonky3_b200.field import KoalaBear as KB, BabyBear as BB
    from plonky3_b200.gpu import Gpu
    from plonky3_b200.poseidon2 import default_poseidon2

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    numa = bind_to_gpu_numa(local)           # before any pinned allocation
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    gpu = Gpu(local)
    for f in (KB, BB):
        for w in (16, 24):
            default_poseidon2(f, w).upload(gpu)
    dev = f"cuda:{local}"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def timed(fn, steps, warmup):
        """W warm-up steps, then K timed steps bracketed by barrier+synchronize, CUDA events, max over ranks."""
        for _ in range(warmup):
            fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = gpu.launches
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        return max_over_ranks(a.elapsed_time(b)) / steps, (gpu.launches - l0)

    # ---- primary: coset LDE, device resident
    g = torch.Generator(device=dev); g.manual_seed(1 + rank)
    if world > 1:     # my column block of the 2^20 x 100N matrix: blocks are multiples of 8 columns (32-byte store segments stay sector-aligned)
        from plonky3_b200.distributed import column_block
        col0, col1 = column_block(W * world, world, rank, align=8)
    else:
        col0, col1 = 0, W
    x = torch.randint(0, KB.P, (1 << LOG_H, col1 - col0), device=dev, dtype=torch.int32, generator=g)
    gpu._use_torch_stream()
    warm = max(args.warmup, 3)
    if world == 1:
        out = torch.empty((1 << (LOG_H + ADDED_BITS), W), device=dev, dtype=torch.int32)

        def lde_step():
            _lib.check(gpu.L.p3gpu_coset_lde_batch_dev(gpu.h, KB.id, x.data_ptr(), 1 << LOG_H, W, ADDED_BITS, KB.generator, out.data_ptr(), 1))
        workload = "coset_lde_batch KoalaBear 2^20 x 100, added_bits 1, shift GENERATOR, bit-reversed rows (BASELINE configs[1])"
        grp = None
    else:
        from plonky3_b200.distributed import PeerGroup
        H = 1 << (LOG_H + ADDED_BITS)
        grp = PeerGroup(gpu, H // world, W * world)

        def lde_step():
            grp.lde_sharded(KB, x, ADDED_BITS, KB.generator, col0)            # last pass stores into every rank's row block
            grp.barrier()                                                     # ... and the step ends when all stores have landed
        workload = (f"coset_lde_batch KoalaBear 2^20 x {W * world} column-sharded over {world} GPUs (100 columns per GPU on average; blocks of 96/104 "
                    "columns = multiples of 8), row-sharded result through fused peer-memory stores + flag barrier (BASELINE configs[1] per GPU)")
    with ClockSampler(local) as clk:
        ms, launches = timed(lde_step, args.steps, warm)
    value = world * OUT_ELEMS / (ms * 1e-3) / 1e9
    if args.dump_outputs:
        if world == 1:
            dump_outputs(args.dump_outputs, out, "coset_lde", DUMP_ROWS)
        else:
            dump_outputs(args.dump_outputs, grp.rows_tensor(), f"coset_lde_rank{rank}", DUMP_ROWS // (world * world))

    line = {
        "metric": "coset_lde_batch output Gelem/s (KoalaBear 2^20 x 100 per GPU, blowup 2)", "value": value, "unit": "Gelem/s",
        "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32 (31-bit Montgomery)", "data": "synthetic",
        "config": {"workload": workload, "per_gpu_matrices": 1,
                   "l2_policy": "inputs+outputs (1.26 GB per GPU) exceed the 126 MB L2; no flush needed",
                   "collective": "none (N=1)" if world == 1 else "all-to-all fused into the LDE's last-pass stores (peer memory, NVLink) + flag barrier, inside the timed region"},
        "gpu_launches": launches, "clocks": clk.summary(), "host_numa_binding": numa,
    }
    if world > 1:      # what the exchange costs: the same LDE without it, and the bytes that cross NVLink per step
        wl = col1 - col0
        loc_out = torch.empty((1 << (LOG_H + ADDED_BITS), wl), device=dev, dtype=torch.int32)
        ms_local, _ = timed(lambda: _lib.check(gpu.L.p3gpu_coset_lde_batch_dev(gpu.h, KB.id, x.data_ptr(), 1 << LOG_H, wl, ADDED_BITS, KB.generator,
                                                                              loc_out.data_ptr(), 1)), max(3, args.steps // 2), 2)
        sent = (1 << (LOG_H + ADDED_BITS)) * wl * 4 * (world - 1) // world
        line["exchange"] = {"ms_per_step_without_exchange": ms_local, "nvlink_bytes_sent_per_gpu_per_step": sent,
                            "nvlink_GBps_per_gpu": sent / (ms * 1e-3) / 1e9, "nvlink_peer_copy_peak_GBps": 770.0}
        del loc_out

    # ---- e2e: host-pointer C-ABI call, pinned host buffers, copies inside the timed region, ONE call at a time
    if not args.no_e2e:
        import threading as _th
        xe = x if x.shape[1] == W else torch.randint(0, KB.P, (1 << LOG_H, W), device=dev, dtype=torch.int32, generator=g)
        lanes = []
        for _ in range(2):
            lg = Gpu(local)
            hx = torch.empty((1 << LOG_H, W), dtype=torch.int32).pin_memory(); hx.copy_(xe.cpu())
            hout = torch.empty((1 << (LOG_H + ADDED_BITS), W), dtype=torch.int32).pin_memory()
            lanes.append((lg, hx, hout))

        def e2e_call(lane):
            lg, hx, hout = lane
            _lib.check(lg.L.p3gpu_coset_lde_batch(lg.h, KB.id, hx.data_ptr(), 1 << LOG_H, W, ADDED_BITS, KB.generator, hout.data_ptr(), 1))

        def e2e_run(n_steps, inflight):
            def worker(lane, n):
                for _ in range(n):
                    e2e_call(lane)
            ths = [_th.Thread(target=worker, args=(lanes[i], n_steps // inflight + (1 if i < n_steps % inflight else 0))) for i in range(inflight)]
            barrier()
            t0 = time.perf_counter()
            for t_ in ths: t_.start()
            for t_ in ths: t_.join()
            torch.cuda.synchronize()
            return max_over_ranks((time.perf_counter() - t0) * 1e3) / n_steps

        e2e_steps = max(4, min(args.steps, 10))
        for lane in lanes:
            for _ in range(3):
                e2e_call(lane)                               # warm-up (allocations, twiddle tables, pinned pages)
        single_ms = e2e_run(e2e_steps, 1)
        two_ms = e2e_run(e2e_steps, 2)
        ref_out = torch.empty((1 << (LOG_H + ADDED_BITS), W), device=dev, dtype=torch.int32)
        gpu._use_torch_stream()
        _lib.check(gpu.L.p3gpu_coset_lde_batch_dev(gpu.h, KB.id, xe.data_ptr(), 1 << LOG_H, W, ADDED_BITS, KB.generator, ref_out.data_ptr(), 1))
        for lane in lanes:
            assert torch.equal(lane[2].to(dev), ref_out), "e2e result differs from device-resident result"
        del ref_out
        line["e2e"] = {"value": world * OUT_ELEMS / (single_ms * 1e-3) / 1e9, "unit": "Gelem/s", "ms_per_step": single_ms,
                       "h2d_bytes_per_step": lanes[0][1].numel() * 4, "d2h_bytes_per_step": lanes[0][2].numel() * 4,
                       "api": "p3gpu_coset_lde_batch (host pointers, pinned, NUMA-local), ONE call at a time (strictly serial H2D -> LDE -> D2H with contiguous copies; "
                              f"P3GPU_E2E_CHUNKS={os.environ.get('P3GPU_E2E_CHUNKS', '1')}: the chunk-pipelined variant is slower on this PCIe, profiles/r02_pcie_probe.txt)",
                       "two_calls_in_flight_ms": two_ms, "two_calls_in_flight_value": world * OUT_ELEMS / (two_ms * 1e-3) / 1e9,
                       "d2h_floor_ms_at_55GBps": lanes[0][2].numel() * 4 / 55e9 * 1e3,
                       "timer": "host wall clock around the calls (device work is synchronous inside the call), max over ranks"}
        del lanes

    # ---- roofline of the dominant kernel (ntt_pass_pipe_kernel): every launch of the step is this kernel
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak, peak_src = json.loads(peaks_path.read_text())["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    achieved = ALG_BYTES / (ms * 1e-3) / 1e9
    traffic, traffic_src = None, None      # dram__bytes_read.sum + dram__bytes_write.sum over the launches of one LDE step (ncu --set full)
    tp = ROOT / "profiles" / "ncu_traffic.json"
    if tp.exists():
        tj = json.loads(tp.read_text())
        traffic, traffic_src = tj.get("lde_step_dram_bytes"), tj.get("source")
    sm_hz = (line["clocks"]["sm_mhz"] or 1965.0) * 1e6
    int_floor_ms = BUTTERFLIES / (12.85 * 148 * sm_hz) * 1e3
    line["roofline"] = {"bound": "hbm", "kernel": "ntt_pass_pipe_kernel (all launches of an LDE step)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                        "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                        "algorithmic_bytes_per_step": ALG_BYTES, "launches_per_step": launches / args.steps,
                        "int_floor_ms": int_floor_ms, "int_floor_frac": int_floor_ms / ms,
                        "note": "integer-issue bound, not HBM bound: 3.146e9 butterflies x (IMAD.HI + 2 IMAD + 4 ALU); the register-only butterfly loop "
                                "(tools/ubench) peaks at 12.85 butterflies/clk/SM = int_floor_ms at the sampled SM clock (DESIGN.md 4.1)"}

    # ---- config-5 trace commit, column-sharded over the ranks: strong scaling, per-phase, three modes
    if not args.no_sharded:
        line["sharded_commit"] = sharded_commit(gpu, world, rank, dev, barrier, max_over_ranks, KB, _lib, torch, dist, np)

    # ---- secondary workloads (single GPU only)
    if world == 1 and not args.no_others:
        line["others"] = others(gpu, timed, g, dev, peak, KB, BB, _lib, torch, np)

    # ---- CPU baseline (rank 0, N=1)
    if world == 1 and rank == 0 and not args.no_cpu:
        try:
            v, cores, sample = cpu_lde_throughput()
            line["cpu_baseline"] = {"value": v, "unit": "Gelem/s", "cores": cores, "kind": "port", "sample": sample}
            if not args.no_others:
                line["others"]["cpu_hash_legs"] = cpu_hash_legs()
        except Exception as e:  # the oracle is test infrastructure; never let it break the GPU numbers
            line["cpu_baseline"] = {"value": None, "unit": "Gelem/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}

    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        if grp is not None:
            grp.close()
        dist.destroy_process_group()


def sharded_commit(gpu, world, rank, dev, barrier, max_over_ranks, KB, _lib, torch, dist, np):
    """One config-5 trace (2^20 x 1312, every rank derives the same synthetic trace from the same seed and keeps its column
    block), committed across the ranks.  Returns per-mode ms (max over ranks, CUDA events), phases and the cap check."""
    from plonky3_b200.distributed import GpuBackend, PeerGroup, column_block, column_starts, commit_bit_exact, commit_column_blocks
    h, H = 1 << T_LOG_H, 2 << T_LOG_H
    gt = torch.Generator(device=dev); gt.manual_seed(12345)
    full = torch.randint(0, KB.P, (h, T_W), device=dev, dtype=torch.int32, generator=gt)
    # the N=1 commitment of the whole trace (untimed here unless N == 1): what every sharded mode must reproduce
    lde1, layers1 = gpu.pcs_commit(KB.id, _lib.HASH_POSEIDON2_W24, full, 1)
    cap_ref = layers1[len(layers1) - 1 - T_CAP][: 1 << T_CAP].cpu().numpy().view(np.uint32).copy()
    res = {"workload": f"TwoAdicFriPcs::commit KoalaBear 2^{T_LOG_H} x {T_W}, blowup 2, Poseidon2-24 leaves / Poseidon2-16 nodes, cap_height {T_CAP} "
                       "(BASELINE configs[4] trace commit), ONE trace column-sharded over the ranks", "scaling": "strong",
           "lde_out_elems": H * T_W}
    reps = 3

    def ev_time(fn, n=reps):
        fn(); barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record(); barrier()
        return max_over_ranks(a.elapsed_time(b)) / n

    if world == 1:
        t = ev_time(lambda: gpu.pcs_commit(KB.id, _lib.HASH_POSEIDON2_W24, full, 1))
        res["single_gpu"] = {"ms": t, "lde_out_Gelem_per_s": H * T_W / t / 1e6}
    del lde1, layers1
    torch.cuda.empty_cache()
    c0, c1 = column_block(T_W, world, rank, align=8)
    local = full[:, c0:c1].contiguous()
    widths = [column_block(T_W, world, q, align=8)[1] - column_block(T_W, world, q, align=8)[0] for q in range(world)]
    del full
    torch.cuda.empty_cache()
    ok = True

    # mode `peer`: the product path
    grp = PeerGroup(gpu, H // world, T_W)
    phases = np.zeros(4)
    cap, _, _ = grp.commit(KB, _lib.HASH_POSEIDON2_W24, local, column_starts(T_W, world, align=8), 1, T_CAP)
    ok_peer = bool(np.array_equal(cap, cap_ref))

    def peer_step():
        nonlocal phases
        _, _, ph = grp.commit(KB, _lib.HASH_POSEIDON2_W24, local, column_starts(T_W, world, align=8), 1, T_CAP, phases=True)
        phases = phases + np.array(ph)
    phases[:] = 0
    t_peer = ev_time(peer_step)
    ph = phases / (reps + 1)
    if world > 1:
        tt = torch.tensor(ph, device=dev); dist.all_reduce(tt, op=dist.ReduceOp.MAX); ph = tt.cpu().numpy()
    sent = (H // world) * (c1 - c0) * 4 * (world - 1)
    res["peer"] = {"ms": t_peer, "lde_out_Gelem_per_s": H * T_W / t_peer / 1e6, "cap_equals_single_gpu_cap": ok_peer,
                   "phase_ms_max_over_ranks": {"lde_with_fused_peer_stores": float(ph[0]), "barrier_wait": float(ph[1]), "row_sharded_hashing": float(ph[2]),
                                                "cap_exchange_and_barrier": float(ph[3])},
                   "nvlink_bytes_sent_by_this_gpu": sent, "api": "p3gpu_commit_sharded_dev (CUDA IPC peer memory, no collective library on the data path)"}
    ok &= ok_peer
    grp.close()
    del grp
    torch.cuda.empty_cache()

    if world > 1:
        be = GpuBackend(gpu, KB, _lib.HASH_POSEIDON2_W24, 1)
        # mode `nccl`: LDE -> all_to_all -> hashing -> all_gather, timed phase by phase with events on the same stream
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        acc = np.zeros(4)

        def nccl_step(record=False):
            nonlocal acc
            rows = H // world
            evs[0].record()
            lde = be.lde(local)
            evs[1].record()
            send = [lde[k * rows:(k + 1) * rows] for k in range(world)]
            recv = [torch.empty((rows, widths[q]), dtype=lde.dtype, device=lde.device) for q in range(world)]
            dist.all_to_all(recv, send)
            evs[2].record()
            layers = be.commit_rows(recv)
            evs[3].record()
            roots = torch.empty((world, 8), dtype=lde.dtype, device=lde.device)
            dist.all_gather_into_tensor(roots, layers[-1][0].contiguous())
            top = be.tree_from_digests(roots)
            evs[4].record()
            if record:
                torch.cuda.synchronize()
                acc = acc + np.array([evs[k].elapsed_time(evs[k + 1]) for k in range(4)])
            return top
        cap_n, _, _ = commit_bit_exact(be, local, widths, T_CAP)
        ok_nccl = bool(np.array_equal(cap_n.cpu().numpy().view(np.uint32), cap_ref))
        t_nccl = ev_time(nccl_step)
        for _ in range(reps):
            nccl_step(record=True)
        pn = acc / reps
        tt = torch.tensor(pn, device=dev); dist.all_reduce(tt, op=dist.ReduceOp.MAX); pn = tt.cpu().numpy()
        res["nccl"] = {"ms": t_nccl, "lde_out_Gelem_per_s": H * T_W / t_nccl / 1e6, "cap_equals_single_gpu_cap": ok_nccl,
                       "phase_ms_max_over_ranks": {"lde": float(pn[0]), "all_to_all": float(pn[1]), "row_sharded_hashing": float(pn[2]), "all_gather_and_top": float(pn[3])},
                       "api": "plonky3_b200.distributed.commit_bit_exact (torch.distributed / NCCL all_to_all + all_gather): the baseline the peer mode replaces"}
        ok &= ok_nccl
        t_cb = ev_time(lambda: commit_column_blocks(be, local))
        res["column_blocks"] = {"ms": t_cb, "lde_out_Gelem_per_s": H * T_W / t_cb / 1e6,
                                "note": "BASELINE's independent NTT + Merkle per column block + ONE all-gather of roots: G commitments, not the reference's single commitment"}
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok = bool(flag.item())
    res["cap_equal_on_every_rank"] = ok
    assert ok, "sharded commit: cap differs from the single-GPU commitment"
    return res


def others(gpu, timed, g, dev, peak, KB, BB, _lib, torch, np):
    from plonky3_b200.dft import Radix2DitParallel
    from plonky3_b200.fri import FriParameters, TwoAdicFriFolding, commit_phase
    from plonky3_b200.merkle_tree import MerkleTreeMmcs
    from plonky3_b200.poseidon2 import default_poseidon2
    o = {}
    k = 3
    # config 1: Radix2DitParallel forward NTT, BabyBear, 2^16 x 1 (parity case; device time of the single-column transform)
    x1 = torch.randint(0, BB.P, (1 << 16, 1), device=dev, dtype=torch.int32, generator=g)
    t, nl = timed(lambda: gpu.dft_batch(BB.id, _lib.DFT, x1), 20, 3)
    o["config1_dft_bb_2^16x1"] = {"us": t * 1e3, "launches": nl / 20}
    # config 3: MerkleTreeMmcs commit 2^22 x 100 KoalaBear, Poseidon2-16 sponge, cap 0
    xm = torch.randint(0, KB.P, (1 << 22, 100), device=dev, dtype=torch.int32, generator=g)
    t, nl = timed(lambda: gpu.merkle_commit(KB.id, _lib.HASH_POSEIDON2_W16, [xm]), k, 1)
    o["config3_merkle_commit_poseidon2_w16_kb_2^22x100"] = {"ms": t, "Mleaf_per_s": (1 << 22) / t / 1e3, "Mperm_per_s": 58720255 / t / 1e3,
                                                            "alg_GBps": 1.946e9 / (t * 1e-3) / 1e9, "hbm_frac": 1.946e9 / (t * 1e-3) / 1e9 / peak, "launches": nl / k}
    del xm
    # Keccak tree at the config-3 shape (the config-4 hash)
    xk = torch.randint(0, BB.P, (1 << 22, 100), device=dev, dtype=torch.int32, generator=g)
    t, nl = timed(lambda: gpu.merkle_commit(BB.id, _lib.HASH_KECCAK, [xk]), k, 1)
    o["merkle_commit_keccak_bb_2^22x100"] = {"ms": t, "Mperm_per_s": ((1 << 22) * 3 + (1 << 22) - 1) / t / 1e3}
    del xk

    class Betas:           # transcript stand-in: forces the per-round cap D2H + host round trip of the real Fiat-Shamir flow
        def __init__(self, b): self.b = [np.array(v, dtype=np.uint32) for v in b]; self.i = 0
        def observe_cap(self, cap): self.last = np.array(cap)
        def grind(self, bits): return 0
        def sample_algebra_element(self): v = self.b[self.i % len(self.b)]; self.i += 1; return v
        def observe_algebra_slice(self, v): pass

    # config 4 (full size): BabyBear 2^22 x 300, TwoAdicFriPcs::commit = LDE blowup 2 + Keccak Merkle (cap 3), then the FRI commit
    # phase on a 2^23 EF4 codeword, round by round (cap to the host, beta back) with arities [3]*7+[1]
    betas = np.random.default_rng(2).integers(0, BB.P, size=(10, 4), dtype=np.uint32)
    xb = torch.randint(0, BB.P, (1 << 22, 300), device=dev, dtype=torch.int32, generator=g)
    t, nl = timed(lambda: gpu.pcs_commit(BB.id, _lib.HASH_KECCAK, xb, 1), 2, 1)
    tl4, _ = timed(lambda: gpu.coset_lde_batch(BB.id, xb, 1, BB.generator), 2, 1)
    o["config4_pcs_commit_keccak_bb_2^22x300"] = {"ms": t, "of_which_lde_ms": tl4, "launches": nl / 2, "lde_out_Gelem_per_s": (1 << 23) * 300 / tl4 / 1e6,
                                                  "Mperm_per_s_hash_part": 83886079 / (t - tl4) / 1e3}
    del xb
    mm4 = MerkleTreeMmcs.keccak(BB, 3, gpu)
    p4 = FriParameters.new_benchmark_high_arity(mm4)
    v0 = torch.randint(0, BB.P, (1 << 23, 4), device=dev, dtype=torch.int32, generator=g)
    t, nl = timed(lambda: commit_phase(TwoAdicFriFolding(BB, gpu), p4, [v0], Betas(betas), Radix2DitParallel(BB, gpu)), k, 1)
    t_pre, _ = timed(lambda: gpu.fri_commit_phase(BB.id, _lib.HASH_KECCAK, v0.clone(), 1, 0, 3, 3, betas), k, 1)
    o["config4_fri_commit_phase_keccak_bb_2^23"] = {"ms": t, "launches": nl / k, "api": "per-round: p3gpu_merkle_commit_dev -> cap D2H -> host -> p3gpu_fri_fold_dev",
                                                    "presupplied_betas_single_call_ms": t_pre}
    del v0
    # config 5 hot path: KoalaBear, trace 2^20 x 1312, blowup 2, Poseidon2-24 sponge + Poseidon2-16 compression, cap 3
    xt = torch.randint(0, KB.P, (1 << 20, 1312), device=dev, dtype=torch.int32, generator=g)
    t_trace, nl = timed(lambda: gpu.pcs_commit(KB.id, _lib.HASH_POSEIDON2_W24, xt, 1), 2, 1)
    tl, _ = timed(lambda: gpu.coset_lde_batch(KB.id, xt, 1, KB.generator), 2, 1)
    # Pcs::commit with the trace in (pinned) HOST memory: p3gpu_pcs_commit, H2D chunks overlapped with the LDE, cap back
    hx = torch.empty((1 << 20, 1312), dtype=torch.int32).pin_memory(); hx.copy_(xt.cpu())
    gpu.pcs_commit_host(KB.id, _lib.HASH_POSEIDON2_W24, hx, 1, 3)
    t0 = time.perf_counter()
    for _ in range(2):
        cap_h, _, _ = gpu.pcs_commit_host(KB.id, _lib.HASH_POSEIDON2_W24, hx, 1, 3)
    t_host = (time.perf_counter() - t0) * 1e3 / 2
    _, lay = gpu.pcs_commit(KB.id, _lib.HASH_POSEIDON2_W24, xt, 1)
    assert np.array_equal(cap_h, lay[len(lay) - 4][:8].cpu().numpy().view(np.uint32)), "host-memory commit differs from the device-resident commit"
    del hx, lay
    o["config5_pcs_commit_from_host_memory"] = {"ms": t_host, "h2d_bytes": (1 << 20) * 1312 * 4, "d2h_bytes": 256,
                                                "api": "p3gpu_pcs_commit (pinned host trace in, cap out, LDE + digest layers resident)",
                                                "h2d_floor_ms_at_55GBps": (1 << 20) * 1312 * 4 / 55e9 * 1e3}
    lde_t = gpu.coset_lde_batch(KB.id, xt, 1, KB.generator)
    del xt
    from plonky3_b200 import extension as X
    zs = [np.array([11, 22, 33, 44], dtype=np.uint32), np.array([55, 66, 77, 88], dtype=np.uint32)]
    al = np.array([5, 6, 7, 8], dtype=np.uint32)
    zinv0 = X.ef_inv(KB, zs[0])
    t_inv, _ = timed(lambda: gpu.open_inv_denoms(KB.id, 21, zs[0], zinv0), k, 1)
    invd, adj = gpu.open_inv_denoms(KB.id, 21, zs[0], zinv0)
    low = lde_t[: 1 << 20]
    t_col, _ = timed(lambda: gpu.columnwise_dot(KB.id, low, adj), k, 1)
    t_row, _ = timed(lambda: gpu.rowwise_dot(KB.id, lde_t, al), k, 1)
    rr = gpu.rowwise_dot(KB.id, lde_t, al); ro = torch.zeros((1 << 21, 4), dtype=torch.int32, device=dev)
    t_red, _ = timed(lambda: gpu.open_reduce(KB.id, ro, rr, invd, al, al), k, 1)
    col_bytes, row_bytes = (1 << 20) * 1312 * 4 + (1 << 20) * 16, (1 << 21) * 1312 * 4 + (1 << 21) * 16
    open_ms = 2 * (t_inv + t_col + t_red) + t_row
    o["config5_open_pre_fri_kb_2^21x1312"] = {
        "inv_denoms_ms": t_inv, "columnwise_dot_ms": t_col, "columnwise_dot_GBps": col_bytes / t_col / 1e6, "columnwise_dot_hbm_frac": col_bytes / t_col / 1e6 / peak,
        "rowwise_dot_ms": t_row, "rowwise_dot_GBps": row_bytes / t_row / 1e6, "rowwise_dot_hbm_frac": row_bytes / t_row / 1e6 / peak, "reduce_ms": t_red,
        "open_two_points_ms": open_ms, "hbm_peak_GBps": peak,
        "note": "barycentric evaluation at 2 points + alpha compression + quotient accumulation over the resident trace LDE; HBM-bound streaming reductions"}
    del lde_t, invd, adj, rr, ro, low
    xq = torch.randint(0, KB.P, (1 << 20, 4), device=dev, dtype=torch.int32, generator=g)

    def quot():
        a_ = gpu.coset_lde_batch(KB.id, xq, 1, KB.generator); b_ = gpu.coset_lde_batch(KB.id, xq, 1, KB.generator)
        gpu.merkle_commit(KB.id, _lib.HASH_POSEIDON2_W24, [a_, b_])
    t_quot, _ = timed(quot, k, 1)
    v1 = torch.randint(0, KB.P, (1 << 21, 4), device=dev, dtype=torch.int32, generator=g)
    kbetas = np.random.default_rng(3).integers(0, KB.P, size=(10, 4), dtype=np.uint32)
    mm5 = MerkleTreeMmcs.poseidon2(default_poseidon2(KB, 16), default_poseidon2(KB, 24), 3, gpu)
    p5 = FriParameters.new_benchmark_high_arity(mm5)
    t_fri, _ = timed(lambda: commit_phase(TwoAdicFriFolding(KB, gpu), p5, [v1], Betas(kbetas), Radix2DitParallel(KB, gpu)), k, 1)
    o["config5_hot_path_kb_2^20x1312"] = {
        "commit_trace_ms": t_trace, "of_which_lde_ms": tl, "lde_out_Gelem_per_s": (1 << 21) * 1312 / tl / 1e6,
        "Mperm_per_s_hash_part": (171966464 + 2097151) / (t_trace - tl) / 1e3, "commit_quotient_ms": t_quot, "fri_commit_phase_ms": t_fri,
        "hot_path_total_ms": t_trace + t_quot + t_fri + open_ms, "of_which_open_ms": open_ms,
        "note": "device-resident LDE + Merkle + open + FRI commit phase (per-round transcript round trip) of prove_prime_field_31 -f koala-bear "
                "-o poseidon-2-permutations -l 20"}
    del v1, xq
    # config 5 end to end (BASELINE's lead metric): prove_prime_field_31 -f koala-bear -o poseidon-2-permutations -l 20 -d radix-2-dit-parallel
    # -m poseidon-2 = uni-stark prove of 2^23 Poseidon2 permutations (8 per row), every data-parallel step on the device
    from plonky3_b200.fri import TwoAdicFriPcs
    from plonky3_b200.uni_stark import RoundConstants, StarkConfig, VectorizedPoseidon2Air, prove
    torch.cuda.empty_cache()
    rs = np.random.default_rng(7)
    rc = RoundConstants(rs.integers(0, KB.P, (4, 16), dtype=np.uint32), rs.integers(0, KB.P, 20, dtype=np.uint32), rs.integers(0, KB.P, (4, 16), dtype=np.uint32))
    air = VectorizedPoseidon2Air(KB, rc, gpu)
    cfg = StarkConfig(TwoAdicFriPcs(Radix2DitParallel(KB, gpu), mm5, p5), default_poseidon2(KB, 24), 16)
    perm_inputs = torch.randint(0, KB.P, (1 << 23, 16), device=dev, dtype=torch.int32, generator=g)
    t_gen, _ = timed(lambda: air.generate_trace_rows(perm_inputs), 2, 1)
    trace = air.generate_trace_rows(perm_inputs)
    del perm_inputs
    prove(cfg, air, trace)                                   # warm-up (twiddles, allocator)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    reps = 2
    for _ in range(reps):
        proof = prove(cfg, air, trace)
    torch.cuda.synchronize()
    t_prove = (time.perf_counter() - t0) * 1e3 / reps
    t0 = time.perf_counter()
    wire = proof.to_postcard()                               # the reference's wire form (postcard, pruned multiproofs); host re-encoding
    t_wire = (time.perf_counter() - t0) * 1e3
    o["config5_prove_kb_2^20x1312"] = {
        "prove_ms": t_prove, "proof_bytes": len(wire), "serialise_ms": t_wire, "trace_generation_ms": t_gen, "spans_ms": proof.timings_ms, "permutations_proved": 1 << 23,
        "fri": {"log_blowup": 1, "max_log_arity": 3, "num_queries": 100, "query_pow_bits": 16, "cap_height": 3},
        "timer": "host wall clock around prove() with the trace resident on the device (synchronised before and after)",
        "note": "uni-stark prove (uni-stark/src/prover.rs:87-442) with trace commit, quotient, quotient commit, opening, FRI commit phase, "
                "proof-of-work and the 100 query openings all on the device; the transcript sponge is device resident (csrc/challenger.cu)"}
    del trace, proof
    return o


if __name__ == "__main__":
    main()
