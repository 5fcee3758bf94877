"""
The arithmetic of the end-of-step reductions (genesis_forge_b200/csrc/tail_math.cuh), compiled on the host
from the same header the kernels include, against exact references:

  * the exact sums behind the logged episode means (reward_manager.py:205-216): each fp32 quotient is added
    as an integer, so the sum is exact over the whole fp32 range, whatever the order.  Checked against
    `fractions.Fraction` / `math.fsum` and against torch-CPU's fp32 mean, within torch's own summation bound.
  * compact_kernel's launch geometry, swept over every mask-word count up to 4 * 2^20 envs.

A pure-Python model of the previous accumulator (64-bit fixed point with 32 fractional bits) documents what
it got wrong: a launch-wide sum past 2^31 wrapped, one quotient of 2^20 or more logged +-Inf, and quotients
were rounded to 2^-32 (denormals logged 0).  tests/test_gpu_logging_reductions.py checks the kernels.
"""
import ctypes as C
import math
import os
import shutil
import subprocess
from fractions import Fraction

import numpy as np
import pytest
import torch

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "genesis_forge_b200", "csrc")
NVCC = shutil.which("nvcc") or ("/usr/local/cuda/bin/nvcc" if os.path.exists("/usr/local/cuda/bin/nvcc") else None)
XS_WORDS = 10
FLT_MAX = float(np.finfo(np.float32).max)
FLT_MIN = float(np.finfo(np.float32).tiny)
DENORM_MIN = 2.0 ** -149

SHIM = r"""
#include "tail_math.cuh"
extern "C" {
// as the post kernel: slabs of up to 256 values sum 16-bit pieces in 32-bit counters, then add their
// nonzero words to the launch's words (whose atomics wrap modulo 2^64 too)
void xs_accumulate(const float* q, long long n, unsigned long long* words, unsigned* flags) {
  for (long long s0 = 0; s0 < n; s0 += 256) {
    int c[gfb::XS_WORDS * 2] = {0};
    for (long long i = s0; i < n && i < s0 + 256; ++i) {
      long long lo, hi;
      const int k = gfb::xs_split(q[i], lo, hi, *flags);
      if (k < 0) continue;
      int p0, p1, p2, p3;
      gfb::xs_pieces(lo, p0, p1);
      gfb::xs_pieces(hi, p2, p3);
      c[2 * k] += p0;
      c[2 * k + 1] += p1;
      c[2 * k + 2] += p2;
      c[2 * k + 3] += p3;
    }
    for (int w = 0; w < gfb::XS_WORDS; ++w) words[w] += (unsigned long long)gfb::xs_join(c[2 * w], c[2 * w + 1]);
  }
}
long long xs_pieces_roundtrip(long long v, int times) {  // times * v through the 32-bit counters
  int p0, p1;
  gfb::xs_pieces(v, p0, p1);
  return gfb::xs_join(p0 * times, p1 * times);
}
int xs_split_one(float q, long long* lo, long long* hi, unsigned* flags) { return gfb::xs_split(q, *lo, *hi, *flags); }
double xs_value(const long long* words, unsigned flags) { return gfb::xs_to_double(words, flags); }
float xs_mean_of(double sum, double n) { return gfb::xs_mean(sum, n); }
void compact_geometry_many(const int* n_words, int n, int* n_blocks, int* words_per_block) {
  for (int i = 0; i < n; ++i) {
    const gfb::CompactGeometry g = gfb::compact_geometry(n_words[i]);
    n_blocks[i] = g.n_blocks;
    words_per_block[i] = g.words_per_block;
  }
}
}
"""


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    if NVCC is None:
        pytest.skip("nvcc not available")
    d = tmp_path_factory.mktemp("tail_math")
    src, out = d / "shim.cu", d / "libtail_math.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-x", "cu", "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "-Xcompiler",
           "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(out)]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    assert proc.returncode == 0, proc.stderr
    lib = C.CDLL(str(out))
    lib.xs_accumulate.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.POINTER(C.c_uint)]
    lib.xs_split_one.argtypes = [C.c_float, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), C.POINTER(C.c_uint)]
    lib.xs_split_one.restype = C.c_int
    lib.xs_pieces_roundtrip.argtypes = [C.c_longlong, C.c_int]
    lib.xs_pieces_roundtrip.restype = C.c_longlong
    lib.xs_value.argtypes = [C.c_void_p, C.c_uint]
    lib.xs_value.restype = C.c_double
    lib.xs_mean_of.argtypes = [C.c_double, C.c_double]
    lib.xs_mean_of.restype = C.c_float
    lib.compact_geometry_many.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return lib


class Acc:
    """One term's accumulator, filled in chunks (the order of the chunks does not matter)."""

    def __init__(self, lib):
        self.lib, self.words, self.flags = lib, np.zeros(XS_WORDS, dtype=np.uint64), C.c_uint(0)

    def add(self, q):
        q = np.ascontiguousarray(q, dtype=np.float32)
        self.lib.xs_accumulate(q.ctypes.data, len(q), self.words.ctypes.data, C.byref(self.flags))
        return self

    def value(self) -> float:
        return self.lib.xs_value(self.words.ctypes.data, self.flags.value)

    def mean(self, n: int) -> np.float32:
        return np.float32(self.lib.xs_mean_of(self.value(), float(n)))


def exact_sum(q) -> Fraction:
    return sum((Fraction(float(v)) for v in np.asarray(q, dtype=np.float32)), Fraction(0))


def contract_mean(q) -> np.float32 | None:
    """The contract's value, or None when any value within 1 fp32 ulp of S / n is right (finite case)."""
    q = np.asarray(q, dtype=np.float32)
    if np.isnan(q).any() or (np.isposinf(q).any() and np.isneginf(q).any()):
        return np.float32("nan")
    if np.isinf(q).any():
        return q[np.isinf(q)][0]
    s = exact_sum(q)
    if abs(s) >= Fraction(2 ** 128 - 2 ** 103):  # fp32 rounding of S overflows
        return np.float32(math.copysign(math.inf, s))
    return np.float32(0.0) if s == 0 else None


def check_mean(got: np.float32, q):
    """The contract of a logged mean (tail.cuh) for the values q, whose exact sum is S."""
    q = np.asarray(q, dtype=np.float32)
    want = contract_mean(q)
    if want is not None:
        assert np.array_equal(np.array([got]).view(np.int32), np.array([want]).view(np.int32)) or (
            np.isnan(got) and np.isnan(want)), (got, want)
        return
    exact = exact_sum(q) / len(q)
    ulp = np.spacing(np.float32(abs(float(exact))))
    assert abs(Fraction(float(got)) - exact) <= Fraction(float(ulp)), (got, float(exact), float(ulp))


def torch_bound(q) -> float:
    """torch-CPU's fp32 mean is itself within (n-1) 2^-24 sum|q| / n of S / n; + 1 ulp of the result."""
    q = np.asarray(q, dtype=np.float64)
    return (len(q) - 1) * 2.0 ** -24 * float(np.abs(q).sum()) / len(q)


def check_vs_torch(got: np.float32, q):
    q = np.asarray(q, dtype=np.float32)
    cpu = np.float32(torch.from_numpy(q).mean().item())
    if np.isfinite(q).all() and np.abs(q.astype(np.float64)).sum() > FLT_MAX and (q > 0).any() and (q < 0).any():
        return  # unspecified (DESIGN.md section 4): torch's own partial sums may overflow
    if not (np.isfinite(got) and np.isfinite(cpu)):
        assert (np.isnan(got) and np.isnan(cpu)) or got == cpu, (got, cpu)
        return
    bound = torch_bound(q) + float(np.spacing(np.float32(abs(cpu))))
    assert abs(float(got) - float(cpu)) <= bound, (got, cpu, bound)


def logged(lib, q, chunks=1):
    acc = Acc(lib)
    for part in np.array_split(np.asarray(q, dtype=np.float32), chunks):
        acc.add(part)
    return acc


# ------------------------------------------------------------------------------------------------
# the split of one value
# ------------------------------------------------------------------------------------------------
def test_split_is_exact_for_every_exponent(lib):
    rng = np.random.default_rng(0)
    for ef in range(0, 255):
        for sign in (0, 1):
            mant = rng.integers(0, 1 << 23, size=4)
            mant[0] = 0 if ef else 1
            mant[1] = (1 << 23) - 1
            for m in mant:
                bits = np.array([(sign << 31) | (ef << 23) | int(m)], dtype=np.uint32)
                q = float(bits.view(np.float32)[0])
                lo, hi, fl = C.c_longlong(), C.c_longlong(), C.c_uint(0)
                k = lib.xs_split_one(q, C.byref(lo), C.byref(hi), C.byref(fl))
                if q == 0.0:
                    assert k == -1 and lo.value == hi.value == 0
                    continue
                assert 0 <= k <= XS_WORDS - 2 and fl.value == 0
                assert abs(lo.value) < 2 ** 32 and abs(hi.value) < 2 ** 32
                value = Fraction(lo.value * 2 ** (32 * k) + hi.value * 2 ** (32 * k + 32)) * Fraction(2) ** -149
                assert value == Fraction(q), (ef, sign, m)


def test_slab_pieces_hold_a_full_slab_of_the_largest_increments(lib):
    """A slab's 32-bit counters hold 256 (and up to 2^15) increments of any magnitude below 2^32, exactly."""
    rng = np.random.default_rng(1)
    for v in [0, 1, -1, 0xFFFF, 0x10000, 2 ** 32 - 1, -(2 ** 32 - 1), *rng.integers(-(2 ** 32) + 1, 2 ** 32, 64)]:
        for times in (1, 256, 2 ** 15):
            assert lib.xs_pieces_roundtrip(int(v), times) == int(v) * times, (v, times)


@pytest.mark.parametrize("q,flags", [(math.nan, 1), (math.inf, 2), (-math.inf, 4), (0.0, 0), (-0.0, 0)])
def test_split_of_special_values(lib, q, flags):
    lo, hi, fl = C.c_longlong(), C.c_longlong(), C.c_uint(0)
    assert lib.xs_split_one(q, C.byref(lo), C.byref(hi), C.byref(fl)) == -1
    assert fl.value == flags and lo.value == hi.value == 0


# ------------------------------------------------------------------------------------------------
# sums and means against the exact references
# ------------------------------------------------------------------------------------------------
def _random_full_range(rng, n, denormals=True):
    ef = rng.integers(0 if denormals else 1, 255, size=n, dtype=np.uint32)
    bits = (rng.integers(0, 2, size=n, dtype=np.uint32) << 31) | (ef << 23) | rng.integers(0, 1 << 23, size=n,
                                                                                          dtype=np.uint32)
    return bits.view(np.float32)


@pytest.mark.parametrize("seed", range(6))
def test_random_exponents_over_the_full_range(lib, seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 3000))
    q = _random_full_range(rng, n)
    if seed % 2:  # only small exponents: the mean is far below 1 and the denormals matter
        q = (q.view(np.uint32) & np.uint32(0x87FFFFFF)).view(np.float32)
    acc = logged(lib, q, chunks=3)
    ref = math.fsum(q.astype(np.float64))  # (the exact sum rounded to double)
    assert abs(acc.value() - ref) <= 2 * math.ulp(ref), (acc.value(), ref)
    check_mean(acc.mean(n), q)
    check_vs_torch(acc.mean(n), q)
    # order-independent: the words are the same in any order and any chunking
    other = logged(lib, rng.permutation(q), chunks=7)
    assert np.array_equal(other.words, acc.words)


CASES = {
    "flt_max_min": [FLT_MAX, -FLT_MAX, FLT_MIN, -FLT_MIN, DENORM_MIN],
    "denormals": [DENORM_MIN, 3 * DENORM_MIN, 2.0 ** -127, -(2.0 ** -140)],
    "one_denormal": [DENORM_MIN],
    "tiny": [1e-9, 1e-9, 1e-9],
    "tiny_30": [1e-30] * 5,
    "cancel_2p100": [2.0 ** 100, -(2.0 ** 100), 1e-30],
    "cancel_flt_max": [FLT_MAX, DENORM_MIN, -FLT_MAX],
    "cancel_to_zero": [1.0, -0.5, -0.5],
    "below_2p20": [2.0 ** 20 - 2.0 ** -4] * 3,
    "at_2p20": [2.0 ** 20, 1.0],
    "large": [1e10, 1e30, -1e10],
    "minus_zero": [-0.0] * 4,
    "normal": [10.0, -3.25, 7.5, -10.0],
    "nan": [1.0, math.nan, 2.0],
    "pos_inf": [1.0, math.inf, -5.0],
    "neg_inf": [-math.inf, 3.0],
    "both_inf": [math.inf, -math.inf],
    "sum_overflows": [3e38] * 1000,
    "sum_overflows_negative": [-3e38] * 3,
    "sum_at_flt_max": [FLT_MAX / 2, FLT_MAX / 2],
}


@pytest.mark.parametrize("case", list(CASES))
def test_edge_cases_meet_the_contract(lib, case):
    q = np.asarray(CASES[case], dtype=np.float32)
    acc = logged(lib, q)
    got = acc.mean(len(q))
    check_mean(got, q)
    check_vs_torch(got, q)
    if np.isfinite(q).all():
        ref = math.fsum(q.astype(np.float64))
        assert abs(acc.value() - ref) <= 2 * math.ulp(ref)
    if case == "minus_zero":
        assert not np.signbit(got) and not np.signbit(torch.tensor(q).mean().item())


def test_repeated_large_quotient_sums_past_two_to_the_31(lib):
    """40000 on 2^17 envs: the sum (5.2e9) passes 2^31; the mean is exactly 40000."""
    q = np.full(1 << 17, 40000.0, dtype=np.float32)
    acc = logged(lib, q, chunks=16)
    assert acc.value() == 40000.0 * 2 ** 17 and acc.mean(len(q)) == np.float32(40000.0)
    check_vs_torch(acc.mean(len(q)), q)


def test_small_quotients_within_torchs_own_bound(lib):
    """torch-CPU's mean of 100,000 copies of 3.7e-6 is itself a few ulp off; ours is within 1 ulp."""
    q = np.full(100_000, 3.7e-6, dtype=np.float32)
    got = logged(lib, q, chunks=4).mean(len(q))
    assert got == np.float32(3.7e-6)
    check_vs_torch(got, q)


# ------------------------------------------------------------------------------------------------
# the previous accumulator, modelled: what the GPU test catches on it
# ------------------------------------------------------------------------------------------------
def parent_mean(q) -> np.float32:
    """The previous kernels' logged mean: to_fixed per quotient, int64 (wrapping) sum, / 2^32, / n."""
    q = np.asarray(q, dtype=np.float32)
    nan = pos = neg = False
    total = 0
    for v in q:
        if v != v:
            nan = True
        elif abs(v) >= np.float32(2.0 ** 20):
            pos, neg = pos or v > 0, neg or v < 0
        else:
            total += int(np.rint(np.float64(np.float32(v * np.float32(2.0 ** 32)))))  # __float2ll_rn(q * 2^32)
    total = (total + 2 ** 63) % 2 ** 64 - 2 ** 63
    if nan or (pos and neg):
        return np.float32("nan")
    if pos or neg:
        return np.float32(math.inf if pos else -math.inf)
    return np.float32(total * 2.0 ** -32 / len(q))


def test_previous_accumulator_wrapped_saturated_and_quantised(lib):
    wraps = np.full(65536, 40000.0, dtype=np.float32)
    assert parent_mean(wraps) == np.float32(-25536.0)
    assert logged(lib, wraps).mean(len(wraps)) == np.float32(40000.0)
    assert torch.from_numpy(wraps).mean().item() == 40000.0

    one_big = np.array([2.0 ** 20], dtype=np.float32)
    assert parent_mean(one_big) == np.float32(math.inf)
    assert logged(lib, one_big).mean(1) == np.float32(2.0 ** 20)

    tiny = np.array([1e-9], dtype=np.float32)
    assert abs(parent_mean(tiny) / np.float32(1e-9) - 1) > 0.06  # 9.31e-10
    assert logged(lib, tiny).mean(1) == np.float32(1e-9)
    denormal = np.array([DENORM_MIN * 5], dtype=np.float32)
    assert parent_mean(denormal) == 0.0
    assert logged(lib, denormal).mean(1) == denormal[0]


# ------------------------------------------------------------------------------------------------
# compact_kernel's launch geometry
# ------------------------------------------------------------------------------------------------
def _mask_words(num_envs: np.ndarray, tile: int) -> np.ndarray:
    """Mask words the post kernel leaves (one per warp of every slab, gfb200.cu)."""
    return (num_envs + tile - 1) // tile * (tile // 32)


def _geometry(lib, n_words: np.ndarray):
    n_words = np.ascontiguousarray(n_words, dtype=np.int32)
    nb, wpb = np.empty_like(n_words), np.empty_like(n_words)
    lib.compact_geometry_many(n_words.ctypes.data, len(n_words), nb.ctypes.data, wpb.ctypes.data)
    return nb.astype(np.int64), wpb.astype(np.int64)


def _parent_geometry(n_words: np.ndarray):
    nb = np.clip((n_words + 255) // 256, 1, 128)
    return nb, ((n_words + nb - 1) // nb + 255) // 256 * 256


@pytest.mark.parametrize("tile", [32, 64, 128, 256])
def test_compact_geometry_covers_the_mask_words_exactly(lib, tile):
    num_envs = np.arange(1, 4 * 2 ** 20 + 1, dtype=np.int64)
    n_words = np.unique(_mask_words(num_envs, tile))
    nb, wpb = _geometry(lib, n_words)
    assert (nb >= 1).all() and (nb <= 128).all() and (wpb % 256 == 0).all()
    # blocks b < nb cover [b * wpb, min((b + 1) * wpb, n_words)): together [0, n_words), every block non-empty,
    # so no block's prefix count (words [0, w0)) or scan reaches word n_words
    assert ((nb - 1) * wpb < n_words).all() and (nb * wpb >= n_words).all()
    # the words are within the allocation (ceil(N / 32) + 8 words)
    assert (_mask_words(num_envs, tile) <= (num_envs + 31) // 32 + 8).all()
    # around every multiple of 2^20 envs, explicitly
    around = np.array([m * 2 ** 20 + d for m in range(1, 5) for d in range(-64, 65)], dtype=np.int64)
    aw = _mask_words(around, tile)
    nb, wpb = _geometry(lib, aw)
    assert ((nb - 1) * wpb < aw).all() and (nb * wpb >= aw).all()


def test_previous_compact_geometry_started_blocks_past_the_mask():
    """N = 1,048,580 at tile 128: 32,772 words, yet block 127 started at word 65,024."""
    for n in (1_048_580, 1_500_000, 1_572_864, 2_097_156):
        w = _mask_words(np.array([n]), 128)
        nb, wpb = _parent_geometry(w)
        assert (nb - 1) * wpb >= w, n
    w = _mask_words(np.array([1_048_580]), 128)
    nb, wpb = _parent_geometry(w)
    assert int(w[0]) == 32_772 and int((nb[0] - 1) * wpb[0]) == 65_024
