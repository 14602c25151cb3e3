"""CPU-side checks of the drop-in boundary: the C-ABI library loads and exports every symbol include/p3gpu.h declares,
host logic (arity schedule, field helpers, height ladder) matches the reference's definitions, and the product path
fails loudly without a CUDA device.  No compute calls here."""
import pathlib
import re

import numpy as np
import pytest
import torch

import plonky3_b200 as P
from plonky3_b200 import _lib
from plonky3_b200.field import BabyBear, KoalaBear
from plonky3_b200.fri import compute_log_arity_for_round, FriParameters

ROOT = pathlib.Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol():
    hdr = (ROOT / "include" / "p3gpu.h").read_text()
    declared = sorted(set(re.findall(r"\b(p3gpu_[a-z0-9_]+)\s*\(", hdr)))
    assert declared, "no declarations found"
    L = _lib.load()
    missing = [n for n in declared if not hasattr(L, n)]
    assert not missing, missing
    assert sorted(_lib.EXPORTS) == declared


def test_rust_ffi_declares_every_header_symbol():
    """bindings/rust/p3-gpu/src/ffi.rs (source only: no Rust toolchain in this image) must stay in step with include/p3gpu.h."""
    import re
    header = (ROOT / "include" / "p3gpu.h").read_text()
    ffi = (ROOT / "bindings" / "rust" / "p3-gpu" / "src" / "ffi.rs").read_text()
    declared = set(re.findall(r"\b(p3gpu_[a-z0-9_]+)\s*\(", header))
    bound = set(re.findall(r"fn (p3gpu_[a-z0-9_]+)", ffi))
    assert declared == bound, (sorted(declared - bound), sorted(bound - declared))


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("device present")
    from plonky3_b200.gpu import Gpu
    with pytest.raises(P.P3GpuError, match="no CPU fallback"):
        Gpu(0)


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under plonky3_b200/ may import, link or load it."""
    pat = re.compile(r"p3_oracle|libp3oracle|^\s*(from|import)\s+oracle|oracle/", re.M)
    for f in (ROOT / "plonky3_b200").rglob("*"):
        if f.suffix in (".py", ".cu", ".cuh", ".h", ".sh"):
            assert not pat.search(f.read_text()), f


def test_library_has_no_variant_switches():
    """The NTT pass kernels and the sharded LDE's exchange have one code path each: no environment variable picks a kernel
    variant, tile shape, pass depth or exchange mode.  In particular every rank derives the same exchange chunks (and with them
    the chunk-major row-block layout of the sharded commit) whatever its environment."""
    removed = ["P3GPU_SHARD_MODE", "P3GPU_SHARD_CHUNK", "P3GPU_NTT_THREADS", "P3GPU_NTT_CT", "P3GPU_NTT_LOGCT", "P3GPU_NTT_MAXR",
               "P3GPU_NTT_GENERIC", "P3GPU_NTT_TILED", "P3GPU_NTT_NOBFLY", "P3GPU_NTT_NOLOAD", "P3GPU_NTT_NOSTORE"]
    for f in (ROOT / "plonky3_b200" / "csrc").iterdir():
        if f.suffix in (".cu", ".cuh", ".h"):
            found = [n for n in removed if re.search(rf"\b{n}\b", f.read_text())]
            assert not found, (f.name, found)


def test_field_helpers_match_reference_constants():
    # SURVEY Appendix A (baby_bear.rs:17-68, koala_bear.rs:20-94)
    assert BabyBear.ONE == 0x0FFFFFFE and KoalaBear.ONE == 0x01FFFFFE
    assert BabyBear.from_monty(BabyBear.two_adic_generator(27)) == 0x1A427A41
    assert KoalaBear.from_monty(KoalaBear.two_adic_generator(24)) == 0x6AC49F88
    assert KoalaBear.from_monty(KoalaBear.two_adic_generator(1)) == KoalaBear.P - 1
    a = np.array([0, 1, 5, KoalaBear.P - 1], dtype=np.uint32)
    assert np.array_equal(KoalaBear.from_monty_array(KoalaBear.to_monty_array(a)), a)
    with pytest.raises(ValueError):
        KoalaBear.two_adic_generator(25)


def test_arity_schedule():
    # fri/src/config.rs:180-207 and SURVEY §8 a17: cfg5 2^21 -> [3,3,3,3,3,3,2], cfg4 2^23 -> [3]*7+[1]
    def sched(log_len, log_final, mx):
        out = []
        while log_len > log_final:
            a = compute_log_arity_for_round(log_len, None, log_final, mx); out.append(a); log_len -= a
        return out
    assert sched(21, 1, 3) == [3, 3, 3, 3, 3, 3, 2]
    assert sched(23, 1, 3) == [3] * 7 + [1]
    assert compute_log_arity_for_round(10, 8, 1, 3) == 2
    with pytest.raises(ValueError):
        compute_log_arity_for_round(5, None, 1, 0)
    p = FriParameters.new_benchmark_high_arity(None)
    assert (p.log_blowup, p.max_log_arity, p.num_queries, p.query_proof_of_work_bits) == (1, 3, 100, 16)


def test_cpp_host_mirror_compiles_and_fails_loudly_without_gpu(tmp_path):
    """include/p3gpu.hpp (C++ mirror of the trait surfaces) compiles against the header and links libp3gpu.so."""
    import subprocess
    exe = tmp_path / "host_mirror_check"
    lib_dir = ROOT / "plonky3_b200"
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-I", str(ROOT / "include"), str(ROOT / "tests" / "cpp" / "host_mirror_check.cpp"),
                    "-o", str(exe), f"-L{lib_dir}", "-l:libp3gpu.so", f"-Wl,-rpath,{lib_dir}"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    if torch.cuda.is_available():
        assert r.returncode == 0, r.stdout + r.stderr
    else:
        assert r.returncode == 3 and "no CPU fallback" in r.stdout, r.stdout + r.stderr


def test_cpp_prune_paths_matches_python(tmp_path):
    """p3gpu::prune_paths (include/p3gpu.hpp, host-only) against plonky3_b200.merkle_tree.prune_paths, which the reference's
    committed proof pins (tests/test_oracle.py)."""
    import subprocess
    from plonky3_b200.merkle_tree import prune_paths
    exe = tmp_path / "prune_check"
    lib_dir = ROOT / "plonky3_b200"
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-I", str(ROOT / "include"), str(ROOT / "tests" / "cpp" / "prune_check.cpp"),
                    "-o", str(exe), f"-L{lib_dir}", "-l:libp3gpu.so", f"-Wl,-rpath,{lib_dir}"], check=True)
    rng = np.random.default_rng(5)
    for levels, n in [(1, 1), (3, 2), (5, 7), (10, 100), (6, 150), (4, 0)]:
        idx = [int(v) for v in rng.integers(0, 1 << levels, n)]
        layers = [rng.integers(0, 1 << 32, ((1 << levels) >> l, 8), dtype=np.uint32) for l in range(levels)]
        paths = np.array([[layers[l][(i >> l) ^ 1] for l in range(levels)] for i in idx], dtype=np.uint32).reshape(n, levels, 8)
        text = f"{levels} {n}\n" + "".join(f"{i} " + " ".join(f"{w:x}" for w in paths[q].ravel()) + "\n" for q, i in enumerate(idx))
        r = subprocess.run([str(exe)], input=text, capture_output=True, text=True, check=True)
        got = np.array([int(w, 16) for w in r.stdout.split()], dtype=np.uint32).reshape(-1, 8)
        assert np.array_equal(got, prune_paths(idx, paths)), (levels, n)


def test_device_arithmetic_source_on_the_host(tmp_path):
    """csrc/field.cuh (the arithmetic every kernel is built from) compiled as plain C++ and run on the host: Montgomery and Shoup
    multiplies, the lazy [0, 2p) butterfly contract for any 32-bit input, EF4 products and the two-adic generators, for both
    fields, against 64-bit reference arithmetic (tests/cpp/device_math_check.cpp)."""
    import os
    import subprocess
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    exe = tmp_path / "device_math_check"
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O2", "-w", "-I", cuda_inc, str(ROOT / "tests" / "cpp" / "device_math_check.cpp"), "-o", str(exe)],
                   check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.count("ok ") == 2, r.stdout + r.stderr


def test_device_permutation_source_on_the_host(tmp_path):
    """csrc/hash_core.cuh — the Poseidon2 (looped rounds, lazy S-box, shift-based diagonal) and Keccak-f (32-bit halves) device
    functions the hash kernels are built from — compiled as plain C++ (tests/cpp/hash_core_host.cpp) and checked on the host:
    the reference's Poseidon2 known-answer vectors, random states against the oracle, Keccak-f against the oracle (itself pinned
    to FIPS-202)."""
    import json
    import os
    import subprocess
    import numpy as np
    from oracle import p3_oracle as O
    from plonky3_b200.field import BabyBear, KoalaBear
    from plonky3_b200.poseidon2 import default_poseidon2
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    exe = tmp_path / "hash_core_host"
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O2", "-w", "-I", cuda_inc, str(ROOT / "tests" / "cpp" / "hash_core_host.cpp"), "-o", str(exe)], check=True)
    kats = json.loads((ROOT / "tests" / "golden" / "poseidon2_kat.json").read_text())
    jobs, expect = [], []
    for f in (BabyBear, KoalaBear):
        for w in (16, 24):
            cfg = default_poseidon2(f, w)
            kat = kats[f"{f.name}_{w}"]
            states = np.vstack([O.to_monty_arr(f.id, kat["input"])[None, :], O.random_matrix(f.id, 40, w, seed=w + f.id)])
            pm = O.default_perm(f.id, w)
            want = np.vstack([O.poseidon2_permute(pm, s) for s in states])
            assert O.from_monty_arr(f.id, want[0]).tolist() == kat["expected"]      # the oracle on the reference's vector
            rc_ext = np.concatenate([cfg.rc_initial.ravel(), cfg.rc_terminal.ravel()])
            jobs.append(" ".join(map(str, ["p2", f.id, w, len(cfg.rc_internal), *rc_ext.tolist(), *cfg.rc_internal.tolist(), len(states),
                                           *states.ravel().tolist()])))
            expect.append(want.ravel().astype(np.uint64))
    kst = np.random.default_rng(5).integers(0, 1 << 63, size=(20, 25), dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    kst[0] = 0
    jobs.append("keccak %d %s" % (len(kst), " ".join(map(str, kst.ravel().tolist()))))
    expect.append(np.vstack([O.keccak_f(s) for s in kst]).ravel())
    r = subprocess.run([str(exe)], input="\n".join(jobs) + "\n", capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = np.array(r.stdout.split(), dtype=np.uint64)
    assert np.array_equal(got, np.concatenate(expect))
