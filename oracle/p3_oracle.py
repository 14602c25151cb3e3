"""ctypes front-end of the CPU parity oracle (oracle/p3_oracle.c) — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module.  The product package plonky3_b200 never does.

All arrays are numpy uint32 in Montgomery form (MontyField31.value, monty-31/src/monty_31.rs:34-44).
Field ids: 0 = BabyBear, 1 = KoalaBear.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import pathlib
import subprocess

import numpy as np

_HERE = pathlib.Path(__file__).resolve().parent
BABY_BEAR, KOALA_BEAR = 0, 1
P2_MAXW = 24


def build(native: bool = False, out=None) -> pathlib.Path:
    """Compile the oracle with the system gcc (oracle/Makefile), into oracle/_build or to the path `out`."""
    so = pathlib.Path(out).resolve() if out else _HERE / "_build" / "libp3oracle.so"
    src = _HERE / "p3_oracle.c"
    if native or not so.exists() or so.stat().st_mtime < src.stat().st_mtime:
        subprocess.run(["make", "-C", str(_HERE), "-B" if native else "-s", f"OUT={so}"], check=True,
                       stdout=subprocess.DEVNULL)
    return so


class Perm(C.Structure):
    _fields_ = [("field", C.c_int), ("width", C.c_int), ("rounds_p", C.c_int),
                ("rc_init", C.c_uint32 * (4 * P2_MAXW)), ("rc_term", C.c_uint32 * (4 * P2_MAXW)),
                ("rc_int", C.c_uint32 * 32)]


class Air(C.Structure):
    """p3o_air: VectorizedPoseidon2Air round constants (width 16, degree-3 S-box: the KoalaBear instance)."""
    _fields_ = [("field", C.c_int), ("rounds_p", C.c_int), ("beg", C.c_uint32 * 64), ("part", C.c_uint32 * 32), ("end", C.c_uint32 * 64)]


class Hasher(C.Structure):
    _fields_ = [("kind", C.c_int), ("leaf_rate", C.c_int), ("leaf", Perm), ("comp", Perm)]


_lib = None


def lib(so=None):
    """The loaded oracle; the first call loads `so` if given, else the in-tree build."""
    global _lib
    if _lib is None:
        L = C.CDLL(str(so or build()))
        u32, u64, sz, p32 = C.c_uint32, C.c_uint64, C.c_size_t, C.POINTER(C.c_uint32)
        for name, res, args in [
            ("p3o_prime", u32, [C.c_int]), ("p3o_add", u32, [C.c_int, u32, u32]), ("p3o_sub", u32, [C.c_int, u32, u32]),
            ("p3o_mul", u32, [C.c_int, u32, u32]), ("p3o_pow", u32, [C.c_int, u32, u64]), ("p3o_inv", u32, [C.c_int, u32]),
            ("p3o_halve", u32, [C.c_int, u32]), ("p3o_to_monty", u32, [C.c_int, u32]), ("p3o_from_monty", u32, [C.c_int, u32]),
            ("p3o_two_adic_generator", u32, [C.c_int, u32]), ("p3o_generator", u32, [C.c_int]),
            ("p3o_to_monty_vec", None, [C.c_int, C.c_void_p, sz]), ("p3o_from_monty_vec", None, [C.c_int, C.c_void_p, sz]),
            ("p3o_reverse_matrix_index_bits", None, [C.c_void_p, sz, sz]),
            ("p3o_naive_dft", None, [C.c_int, C.c_void_p, sz, sz, C.c_void_p]),
            ("p3o_dft_batch", None, [C.c_int, C.c_void_p, sz, sz]), ("p3o_idft_batch", None, [C.c_int, C.c_void_p, sz, sz]),
            ("p3o_coset_dft_batch", None, [C.c_int, C.c_void_p, sz, sz, u32]),
            ("p3o_coset_idft_batch", None, [C.c_int, C.c_void_p, sz, sz, u32]),
            ("p3o_coset_lde_batch", None, [C.c_int, C.c_void_p, sz, sz, C.c_uint, u32, C.c_void_p, C.c_int]),
            ("p3o_poseidon2_diag", None, [C.c_int, C.c_int, C.c_void_p]),
            ("p3o_poseidon2_permute", None, [C.POINTER(Perm), C.c_void_p]),
            ("p3o_keccak_f", None, [C.c_void_p]),
            ("p3o_hash_row", None, [C.POINTER(Hasher), C.c_void_p, sz, C.c_void_p]),
            ("p3o_compress", None, [C.POINTER(Hasher), C.c_void_p, C.c_void_p, C.c_void_p]),
            ("p3o_validate_heights", C.c_int, [C.c_void_p, sz]),
            ("p3o_merkle_tree", sz, [C.POINTER(Hasher), sz, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
            ("p3o_merkle_total_digests", sz, [sz]),
            ("p3o_ef_mul", None, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
            ("p3o_fold_matrix", None, [C.c_int, C.c_void_p, sz, C.c_uint, C.c_void_p, C.c_void_p]),
            ("p3o_ef_inv", None, [C.c_int, C.c_void_p, C.c_void_p]),
            ("p3o_open_inv_denoms", None, [C.c_int, C.c_uint, C.c_void_p, C.c_void_p]),
            ("p3o_columnwise_dot", None, [C.c_int, C.c_void_p, sz, sz, C.c_void_p, C.c_void_p]),
            ("p3o_rowwise_dot", None, [C.c_int, C.c_void_p, sz, sz, C.c_void_p, C.c_void_p]),
            ("p3o_open_reduce", None, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, sz, C.c_void_p, C.c_void_p]),
            ("p3o_p2air_cols", sz, [C.POINTER(Air)]), ("p3o_p2air_constraints", sz, [C.POINTER(Air)]),
            ("p3o_p2air_generate", None, [C.POINTER(Air), C.c_void_p, sz, C.c_void_p]),
            ("p3o_p2air_check", sz, [C.POINTER(Air), C.c_int, C.c_void_p, sz]),
            ("p3o_p2air_quotient", None, [C.POINTER(Air), C.c_int, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p]),
            ("p3o_smallrng_seed", None, [u64, C.c_void_p]), ("p3o_smallrng_field", None, [C.c_int, C.c_void_p, C.c_void_p, sz]),
        ]:
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def _u32(a):
    a = np.ascontiguousarray(a, dtype=np.uint32)
    return a


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


# ---------------------------------------------------------------- field helpers
def prime(f): return lib().p3o_prime(f)
def add(f, a, b): return lib().p3o_add(f, a, b)
def sub(f, a, b): return lib().p3o_sub(f, a, b)
def mul(f, a, b): return lib().p3o_mul(f, a, b)
def fpow(f, a, e): return lib().p3o_pow(f, a, e)
def inv(f, a): return lib().p3o_inv(f, a)
def halve(f, a): return lib().p3o_halve(f, a)
def to_monty(f, x): return lib().p3o_to_monty(f, x % prime(f))
def from_monty(f, x): return lib().p3o_from_monty(f, x)
def two_adic_generator(f, bits): return lib().p3o_two_adic_generator(f, bits)
def generator(f): return lib().p3o_generator(f)


def to_monty_arr(f, a):
    a = _u32(np.array(a, dtype=np.uint64) % prime(f)).copy()
    lib().p3o_to_monty_vec(f, _ptr(a), a.size)
    return a


def from_monty_arr(f, a):
    a = _u32(a).copy()
    lib().p3o_from_monty_vec(f, _ptr(a), a.size)
    return a


def random_matrix(f, h, w, seed=1):
    """Uniform field elements (Montgomery representation is itself uniform), deterministic."""
    rng = np.random.default_rng(seed)
    return rng.integers(0, prime(f), size=(h, w), dtype=np.uint32)


# ---------------------------------------------------------------- DFT family
def reverse_matrix_index_bits(m):
    m = _u32(m).copy()
    lib().p3o_reverse_matrix_index_bits(_ptr(m), m.shape[0], m.shape[1])
    return m


def naive_dft(f, m):
    m = _u32(m); out = np.empty_like(m)
    lib().p3o_naive_dft(f, _ptr(m), m.shape[0], m.shape[1], _ptr(out))
    return out


def dft_batch(f, m):
    m = _u32(m).copy(); lib().p3o_dft_batch(f, _ptr(m), m.shape[0], m.shape[1]); return m


def idft_batch(f, m):
    m = _u32(m).copy(); lib().p3o_idft_batch(f, _ptr(m), m.shape[0], m.shape[1]); return m


def coset_dft_batch(f, m, shift):
    m = _u32(m).copy(); lib().p3o_coset_dft_batch(f, _ptr(m), m.shape[0], m.shape[1], shift); return m


def coset_idft_batch(f, m, shift):
    m = _u32(m).copy(); lib().p3o_coset_idft_batch(f, _ptr(m), m.shape[0], m.shape[1], shift); return m


def coset_lde_batch(f, m, added_bits, shift, bitrev_out=True):
    m = _u32(m)
    out = np.empty((m.shape[0] << added_bits, m.shape[1]), dtype=np.uint32)
    lib().p3o_coset_lde_batch(f, _ptr(m), m.shape[0], m.shape[1], added_bits, shift, _ptr(out), int(bitrev_out))
    return out


# ---------------------------------------------------------------- Poseidon2 / Keccak / hashers
_CONSTS = None


def default_constants():
    """Canonical-form default round constants extracted by tools/gen_constants.py."""
    global _CONSTS
    if _CONSTS is None:
        _CONSTS = json.loads((_HERE.parent / "plonky3_b200" / "p2_constants.json").read_text())
    return _CONSTS


def make_perm(f, width, rc_init, rc_term, rc_int, monty=False) -> Perm:
    """rc_* canonical (monty=False) or Montgomery (monty=True) integer lists."""
    pm = Perm()
    pm.field, pm.width, pm.rounds_p = f, width, len(rc_int)
    conv = (lambda x: _u32(x)) if monty else (lambda x: to_monty_arr(f, x))
    a, b, c = conv(rc_init).ravel(), conv(rc_term).ravel(), conv(rc_int).ravel()
    assert a.size == 4 * width and b.size == 4 * width and c.size <= 32
    for i, v in enumerate(a): pm.rc_init[i] = int(v)
    for i, v in enumerate(b): pm.rc_term[i] = int(v)
    for i, v in enumerate(c): pm.rc_int[i] = int(v)
    return pm


def default_perm(f, width) -> Perm:
    name = ("baby_bear", "koala_bear")[f]
    k = default_constants()[f"{name}_{width}"]
    return make_perm(f, width, k["external_initial"], k["external_final"], k["internal"])


def poseidon2_permute(pm: Perm, state):
    s = _u32(state).copy()
    lib().p3o_poseidon2_permute(C.byref(pm), _ptr(s))
    return s


def poseidon2_diag(f, width):
    out = np.empty(width, dtype=np.uint32)
    lib().p3o_poseidon2_diag(f, width, _ptr(out))
    return out


def keccak_f(state25):
    s = np.ascontiguousarray(state25, dtype=np.uint64).copy()
    lib().p3o_keccak_f(_ptr(s))
    return s


def poseidon2_hasher(leaf: Perm, comp: Perm) -> Hasher:
    """leaf: PaddingFreeSponge<leaf,W,W-8,8>; node: TruncatedPermutation<comp,2,8,16>."""
    h = Hasher()
    h.kind, h.leaf_rate, h.leaf, h.comp = 0, leaf.width - 8, leaf, comp
    return h


def keccak_hasher() -> Hasher:
    h = Hasher()
    h.kind, h.leaf_rate = 1, 17
    return h


def hash_row(hs: Hasher, row):
    row = _u32(row); d = np.empty(8, dtype=np.uint32)
    lib().p3o_hash_row(C.byref(hs), _ptr(row), row.size, _ptr(d))
    return d


def compress(hs: Hasher, left, right):
    l, r = _u32(left), _u32(right); d = np.empty(8, dtype=np.uint32)
    lib().p3o_compress(C.byref(hs), _ptr(l), _ptr(r), _ptr(d))
    return d


def validate_heights(heights):
    a = np.ascontiguousarray(heights, dtype=np.uintp)
    return lib().p3o_validate_heights(_ptr(a), a.size)


def merkle_tree(hs: Hasher, mats):
    """MerkleTree::new (arity 2).  Returns list of digest layers, each (len, 8) uint32."""
    mats = [_u32(m) for m in mats]
    n = len(mats)
    hts = np.array([m.shape[0] for m in mats], dtype=np.uintp)
    wds = np.array([m.shape[1] for m in mats], dtype=np.uintp)
    if validate_heights(hts) != 0:
        raise ValueError("incompatible matrix heights")
    ptrs = (C.c_void_p * n)(*[m.ctypes.data for m in mats])
    tot = lib().p3o_merkle_total_digests(int(hts.max()))
    out = np.zeros((tot, 8), dtype=np.uint32)
    lens = np.zeros(80, dtype=np.uintp)
    nl = lib().p3o_merkle_tree(C.byref(hs), n, ptrs, _ptr(hts), _ptr(wds), _ptr(out), _ptr(lens))
    layers, off = [], 0
    for k in range(nl):
        layers.append(out[off:off + int(lens[k])].copy()); off += int(lens[k])
    return layers


def merkle_cap(layers, cap_height):
    """MerkleTree::cap + the clamp in MerkleTreeMmcs::commit (merkle_tree.rs:198-217, mmcs/batch.rs:56-62)."""
    nl = len(layers)
    eff = min(cap_height, max(nl - 1, 0))
    layer = layers[nl - 1 - eff]
    return layer[: min(1 << eff, len(layer))].copy()


# ---------------------------------------------------------------- EF4 / FRI
def ef_mul(f, a, b):
    a, b = _u32(a), _u32(b); o = np.empty(4, dtype=np.uint32)
    lib().p3o_ef_mul(f, _ptr(a), _ptr(b), _ptr(o))
    return o


def ef_inv(f, a):
    a = _u32(a); o = np.empty(4, dtype=np.uint32)
    lib().p3o_ef_inv(f, _ptr(a), _ptr(o))
    return o


def ef_add(f, a, b): return np.array([add(f, int(x), int(y)) for x, y in zip(a, b)], dtype=np.uint32)
def ef_sub(f, a, b): return np.array([sub(f, int(x), int(y)) for x, y in zip(a, b)], dtype=np.uint32)
def ef_from_base(f, x): return np.array([x, 0, 0, 0], dtype=np.uint32)


def ef_pow(f, a, e):
    r = ef_from_base(f, to_monty(f, 1)); a = _u32(a)
    while e:
        if e & 1: r = ef_mul(f, r, a)
        a = ef_mul(f, a, a); e >>= 1
    return r


def open_inv_denoms(f, log_h, z):
    z = _u32(z); out = np.empty((1 << log_h, 4), dtype=np.uint32)
    lib().p3o_open_inv_denoms(f, log_h, _ptr(z), _ptr(out))
    return out


def columnwise_dot(f, mat, v):
    mat, v = _u32(mat), _u32(v); out = np.empty((mat.shape[1], 4), dtype=np.uint32)
    lib().p3o_columnwise_dot(f, _ptr(mat), mat.shape[0], mat.shape[1], _ptr(v), _ptr(out))
    return out


def rowwise_dot(f, mat, alpha):
    mat, alpha = _u32(mat), _u32(alpha); out = np.empty((mat.shape[0], 4), dtype=np.uint32)
    lib().p3o_rowwise_dot(f, _ptr(mat), mat.shape[0], mat.shape[1], _ptr(alpha), _ptr(out))
    return out


def open_reduce(f, ro, r, inv_denoms, coeff, yred):
    ro = _u32(ro).copy(); r, inv_denoms, coeff, yred = _u32(r), _u32(inv_denoms), _u32(coeff), _u32(yred)
    lib().p3o_open_reduce(f, _ptr(ro), _ptr(r), _ptr(inv_denoms), ro.shape[0], _ptr(coeff), _ptr(yred))
    return ro


def interpolate_coset(f, low_coset_bitrev, z, inv_denoms):
    """interpolate_coset_with_precomputation (matrix/src/interpolation.rs:161-193) on the first h rows of a committed
    (bit-reversed) LDE: f(z) = z (z^N - g^N) / (N g^N) * sum_i adjusted_i f(x_i), adjusted_i = 1/(z - x_i) - 1/z."""
    m = _u32(low_coset_bitrev)
    h = m.shape[0]; log_h = int(np.log2(h))
    zinv = ef_inv(f, z)
    adj = np.array([ef_sub(f, inv_denoms[i], zinv) for i in range(h)], dtype=np.uint32) if h <= 4096 else None
    if adj is None:
        adj = _u32(inv_denoms[:h]).copy()
        for k in range(4):
            col = adj[:, k].astype(np.int64) - int(zinv[k])
            adj[:, k] = np.where(col < 0, col + prime(f), col).astype(np.uint32)
    sums = columnwise_dot(f, m, adj)
    g = generator(f)
    z_pow_n = ef_pow(f, z, h)
    g_pow_n = fpow(f, g, h)
    denom_inv = inv(f, mul(f, g_pow_n, to_monty(f, h)))
    scal = ef_mul(f, z, ef_sub(f, z_pow_n, ef_from_base(f, g_pow_n)))
    scal = np.array([mul(f, int(c), denom_inv) for c in scal], dtype=np.uint32)
    return np.array([ef_mul(f, scal, s_) for s_ in sums], dtype=np.uint32)


def fold_matrix(f, vec_ef, log_arity, beta):
    """vec_ef: (len, 4) EF4 values in bit-reversed order; returns (len >> log_arity, 4)."""
    v = _u32(vec_ef); b = _u32(beta)
    rows = v.shape[0] >> log_arity
    out = np.empty((rows, 4), dtype=np.uint32)
    lib().p3o_fold_matrix(f, _ptr(v), rows, log_arity, _ptr(b), _ptr(out))
    return out


def compute_log_arity_for_round(log_cur, next_input_log, log_final, max_log_arity):
    """fri/src/config.rs:180-207."""
    m = log_cur - log_final
    if next_input_log is not None:
        m = min(m, log_cur - next_input_log)
    return min(m, max_log_arity)


def commit_phase(f, hs: Hasher, cap_height, inputs, log_blowup, log_final_poly_len, max_log_arity, betas):
    """FRI commit phase with externally supplied betas (fri/src/prover.rs:192-286; no proof-of-work:
    commit_proof_of_work_bits = 0 as in the benchmark parameters).  `inputs`: one (len,4) EF4 vector or a list of them in
    descending length (shorter inputs are rolled in with beta^arity, prover.rs:258-265).  Returns
    (list of caps, list of log_arities, final folded vector before the final-poly iDFT)."""
    if isinstance(inputs, np.ndarray):
        inputs = [inputs]
    inputs = [_u32(v) for v in inputs]
    folded = inputs.pop(0)
    caps, arities = [], []
    log_final = log_blowup + log_final_poly_len
    k = 0
    while folded.shape[0] > (1 << log_final):
        log_cur = int(np.log2(folded.shape[0]))
        nxt = int(np.log2(inputs[0].shape[0])) if inputs else None
        la = compute_log_arity_for_round(log_cur, nxt, log_final, max_log_arity)
        arities.append(la)
        leaves = folded.reshape(folded.shape[0] >> la, (1 << la) * 4)   # ExtensionMmcs flattening
        layers = merkle_tree(hs, [leaves])
        caps.append(merkle_cap(layers, cap_height))
        beta = _u32(betas[k]); k += 1
        folded = fold_matrix(f, folded, la, beta)
        if inputs and inputs[0].shape[0] == folded.shape[0]:
            bp = beta
            for _ in range(la):
                bp = ef_mul(f, bp, bp)
            x = inputs.pop(0)
            for i in range(folded.shape[0]):
                t = ef_mul(f, bp, x[i])
                folded[i] = [add(f, int(a), int(b)) for a, b in zip(folded[i], t)]
    return caps, arities, folded


# ---------------------------------------------------------------- Poseidon2 AIR (SURVEY 8f ranks 2-3) + SmallRng
class SmallRng:
    """rand 0.10 SmallRng (xoshiro256++ via SplitMix64) drawing MontyField31 samples (values ARE Montgomery representations)."""

    def __init__(self, seed: int):
        self.state = np.zeros(4, dtype=np.uint64)
        lib().p3o_smallrng_seed(seed, _ptr(self.state))

    def field(self, f, n):
        out = np.empty(int(n), dtype=np.uint32)
        lib().p3o_smallrng_field(f, _ptr(self.state), _ptr(out), int(n))
        return out


def make_air(f, beg, part, end) -> Air:
    """RoundConstants::new (poseidon2-air/src/constants.rs:47-57); constants in Montgomery form."""
    a = Air()
    a.field = f
    part = _u32(part).ravel()
    a.rounds_p = part.size
    for i, v in enumerate(_u32(beg).ravel()): a.beg[i] = int(v)
    for i, v in enumerate(part): a.part[i] = int(v)
    for i, v in enumerate(_u32(end).ravel()): a.end[i] = int(v)
    return a


def air_from_rng(f, rng: SmallRng, rounds_p=20) -> Air:
    """RoundConstants::from_rng (constants.rs:59-68): beginning full rounds, partial rounds, ending full rounds, in that order."""
    beg = rng.field(f, 64); part = rng.field(f, rounds_p); end = rng.field(f, 64)
    return make_air(f, beg, part, end)


def perm_from_rng(f, width, rng: SmallRng) -> Perm:
    """Poseidon2::new_from_rng_128 (poseidon2/src/lib.rs:92-107): 4 x width initial, 4 x width terminal, then R_P internal."""
    rp = {(0, 16): 13, (0, 24): 21, (1, 16): 20, (1, 24): 23}[(f, width)]
    init = rng.field(f, 4 * width); term = rng.field(f, 4 * width); internal = rng.field(f, rp)
    return make_perm(f, width, init, term, internal, monty=True)


def p2air_cols(a: Air): return int(lib().p3o_p2air_cols(C.byref(a)))
def p2air_constraints(a: Air): return int(lib().p3o_p2air_constraints(C.byref(a)))


def p2air_generate(a: Air, inputs, vec_len=8):
    """generate_vectorized_trace_rows (generation.rs:14-70): inputs (n_perms, 16) -> trace (n_perms / vec_len, vec_len * cols)."""
    x = _u32(inputs); n = x.shape[0]
    cols = p2air_cols(a)
    out = np.empty((n, cols), dtype=np.uint32)
    lib().p3o_p2air_generate(C.byref(a), _ptr(x), n, _ptr(out))
    return out.reshape(n // vec_len, vec_len * cols)


def p2air_check(a: Air, trace, vec_len=8):
    t = _u32(trace)
    return int(lib().p3o_p2air_check(C.byref(a), vec_len, _ptr(t), t.shape[0]))


def p2air_quotient(a: Air, lde_bitrev, log_n, alpha, vec_len=8):
    """quotient_values over the quotient domain GENERATOR * K, |K| = LDE height; natural order, (H, 4)."""
    m = _u32(lde_bitrev); al = _u32(alpha)
    log_h = int(np.log2(m.shape[0]))
    q = np.empty((m.shape[0], 4), dtype=np.uint32)
    lib().p3o_p2air_quotient(C.byref(a), vec_len, _ptr(m), log_h, log_n, _ptr(al), _ptr(q))
    return q
