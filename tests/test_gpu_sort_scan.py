"""-m gpu: `qed_sort_pairs` (own radix sort and the CUB baseline) and `qed_isect_scan` against plain CPU references.

Sort: numpy's stable argsort of `key & (2^end_bit - 1)` on uint64 (unsigned order, bits above end_bit ignored but kept
in the returned keys), at every size where the radix sort switches code path, every partial last digit, and under the
thread-local test hooks that select the other pass implementations (which must give the default's bytes).
Scan: torch.cumsum in int64, around the tile sizes of the three-phase scan and with totals beyond 2^31.
"""
import contextlib

import numpy as np
import pytest
import torch

from qed_splatter_b200 import _lib, ops
from qed_splatter_b200._lib import check, current_stream, ptr

pytestmark = pytest.mark.gpu

SORT_TILE = 4096                     # radix.cuh kSortTile
SMALL_TILES_MAX_N = 2 * 148 * 4096   # 1,212,416: half-size tiles (hook) up to 2 blocks of 4096 per SM
ONESWEEP_MAX_N = 3 * 148 * 4096      # 1,818,624: look-back passes up to 444 blocks, three kernels per pass above
# (onesweep, small_tiles) settings of the hooks; (1, 0) is the default
HOOK_MODES = [(0, 0), (0, 1), (1, 1), (2, 0), (2, 1)]
MODE2_MAX_N = 4_200_000              # look-back passes at every size: exercised up to here
DISTS = ("uniform", "equal", "two", "sorted", "reverse", "top_digit", "above")


@contextlib.contextmanager
def radix_hooks(onesweep, small_tiles):
    lib = _lib.load()
    old_o = lib.qed_debug_set_radix_onesweep(onesweep)
    old_s = lib.qed_debug_set_radix_small_tiles(small_tiles)
    try:
        yield
    finally:
        lib.qed_debug_set_radix_onesweep(old_o)
        lib.qed_debug_set_radix_small_tiles(old_s)


def _mask(end_bit):
    return np.uint64((1 << end_bit) - 1) if end_bit < 64 else np.uint64(0xFFFF_FFFF_FFFF_FFFF)


def make_keys(dist, n, end_bit, seed):
    """uint64 keys of a named distribution; only "above" (and every distribution at end_bit = 64) has bits above end_bit."""
    rng = np.random.default_rng(seed)
    full = rng.integers(0, 2**64, size=n, dtype=np.uint64)
    m = _mask(end_bit)
    low = full & m
    if dist == "uniform":
        return low
    if dist == "equal":
        return np.full(n, low[0], dtype=np.uint64)
    if dist == "two":
        return np.where(rng.random(n) < 0.5, low[0], low[-1]).astype(np.uint64)
    if dist == "sorted":
        return np.sort(low)
    if dist == "reverse":
        return np.ascontiguousarray(np.sort(low)[::-1])
    if dist == "top_digit":  # only the last (most significant) radix digit varies
        if end_bit == 0:
            return np.zeros(n, dtype=np.uint64)
        lo = np.uint64(8 * ((end_bit - 1) // 8))
        return ((low >> lo) << lo) & m
    if dist == "above":
        return full
    raise ValueError(dist)


def reference_sort(keys_u64, end_bit):
    order = np.argsort(keys_u64 & _mask(end_bit), kind="stable")
    return keys_u64[order], order.astype(np.int32)


def _sort(keys_i64, vals, end_bit, impl):
    return ops.sort_pairs(keys_i64, vals, end_bit, impl=impl)


def check_sort(cuda, keys_u64, end_bit, modes=HOOK_MODES, what=""):
    n = keys_u64.size
    ref_k, ref_v = reference_sort(keys_u64, end_bit)
    ref_k = torch.from_numpy(ref_k.view(np.int64))
    ref_v = torch.from_numpy(ref_v)
    keys = torch.from_numpy(keys_u64.view(np.int64)).to(cuda)
    vals = torch.arange(n, dtype=torch.int32, device=cuda)
    keys_before = keys.clone()
    default = None
    for impl in ("own", "cub"):
        ko, vo = _sort(keys, vals, end_bit, impl)
        assert torch.equal(ko.cpu(), ref_k), f"{what} {impl}: keys"
        assert torch.equal(vo.cpu(), ref_v), f"{what} {impl}: values (stable order)"
        if impl == "own":
            default = (ko, vo)
    assert torch.equal(keys, keys_before), f"{what}: the input keys were modified"
    for onesweep, small in modes:
        if onesweep == 2 and n > MODE2_MAX_N:
            continue
        with radix_hooks(onesweep, small):
            ko, vo = _sort(keys, vals, end_bit, "own")
        assert torch.equal(ko, default[0]) and torch.equal(vo, default[1]), f"{what}: hook mode onesweep={onesweep} small_tiles={small}"


@pytest.mark.timeout(120)
@pytest.mark.parametrize("dist", DISTS)
@pytest.mark.parametrize("end_bit", [0, 1, 7, 8, 9, 16, 17, 32, 33, 45, 63, 64])
def test_sort_pairs_end_bits_and_distributions(cuda, end_bit, dist):
    """Every partial last digit (end_bit % 8 != 0), zero passes (end_bit = 0), eight passes with negative int64 keys
    (end_bit = 64), and keys whose bits above end_bit must be ignored for the order but returned unchanged."""
    n = 70_001  # 18 blocks of 4096: one-kernel passes by default, half-size tiles and three kernels per pass through the hooks
    keys = make_keys(dist, n, end_bit, seed=1000 + end_bit)
    if end_bit == 64 and dist == "uniform":
        assert (keys.view(np.int64) < 0).mean() > 0.4, "negative int64 keys must be sorted in unsigned order"
    if dist == "above" and end_bit < 64:
        assert (keys >> np.uint64(end_bit)).any(), "keys with bits above end_bit"
    check_sort(cuda, keys, end_bit, what=f"n={n} end_bit={end_bit} {dist}")


@pytest.mark.timeout(300)
@pytest.mark.parametrize("n", [1, 4095, 4096, 4097, SMALL_TILES_MAX_N - 1, SMALL_TILES_MAX_N, SMALL_TILES_MAX_N + 1,
                               ONESWEEP_MAX_N, ONESWEEP_MAX_N + 1, 8_000_003])
def test_sort_pairs_sizes(cuda, n):
    """Sizes at the switches: one partial block, the half-size-tile limit of the hook, the last size that runs one
    kernel per pass (444 blocks) and the first that runs three, and a sort of 8 M pairs (S3-size lists).  A partial
    last digit with random bits above it, plus a few equal-key runs for the stability check."""
    nb = (n + SORT_TILE - 1) // SORT_TILE
    if n == ONESWEEP_MAX_N:
        assert nb == 444
    if n == ONESWEEP_MAX_N + 1:
        assert nb == 445
    if n in (SMALL_TILES_MAX_N, SMALL_TILES_MAX_N + 1):
        assert nb == (296 if n == SMALL_TILES_MAX_N else 297)
    keys = make_keys("above", n, 45, seed=n)
    keys[::5] = keys[0]  # ties across every block
    check_sort(cuda, keys, 45, what=f"n={n}")


@pytest.mark.timeout(300)
@pytest.mark.parametrize("dist,end_bit", [("uniform", 64), ("two", 33), ("reverse", 17), ("top_digit", 40)])
def test_sort_pairs_three_kernel_passes_distributions(cuda, dist, end_bit):
    """Degenerate distributions above the look-back limit (three kernels per pass by default, look-back at every size
    through the hook): a digit with every pair of a block, and full 64-bit keys."""
    n = ONESWEEP_MAX_N + 4097
    keys = make_keys(dist, n, end_bit, seed=end_bit)
    check_sort(cuda, keys, end_bit, modes=[(1, 0), (2, 0), (2, 1)], what=f"n={n} end_bit={end_bit} {dist}")


def scan(cuda, vals, pinned=True):
    lib = _lib.load()
    n = vals.numel()
    cum = torch.empty(max(n, 1), dtype=torch.int64, device=cuda)
    total = torch.full((1,), -1, dtype=torch.int64, device=cuda)
    host = torch.full((1,), -1, dtype=torch.int64).pin_memory() if pinned else None
    ws_bytes = lib.qed_isect_scan_workspace_bytes(n)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=cuda)
    check(lib.qed_isect_scan(n, ptr(vals) if n else None, ptr(cum) if n else None, ptr(total), ptr(host), ptr(ws), ws_bytes, current_stream()),
          "qed_isect_scan")
    torch.cuda.synchronize()
    return cum[:n], total, host


SCAN_TILE = 2048  # scan.cuh kScanTile


@pytest.mark.timeout(120)
@pytest.mark.parametrize("n", [0, 1, SCAN_TILE - 1, SCAN_TILE, SCAN_TILE + 1, 1024 * SCAN_TILE - 1, 1024 * SCAN_TILE, 1024 * SCAN_TILE + 1,
                               SCAN_TILE * SCAN_TILE])
@pytest.mark.parametrize("kind", ["counts", "large"])
def test_isect_scan_matches_cumsum(cuda, n, kind):
    """The three-phase scan (block sums, one-block scan of the sums, scan + add) == torch.cumsum in int64, with the
    total on the device and in pinned host memory.  `large`: values up to 2^31 - 1, so that the prefix sums leave the
    int32 range within the first few elements."""
    g = torch.Generator().manual_seed(n + (7 if kind == "large" else 0))
    if kind == "counts":
        v = torch.randint(0, 64, (n,), generator=g, dtype=torch.int32)
        v[torch.rand(n, generator=g) < 0.3] = 0  # culled entries
    else:
        v = torch.randint(0, 2**31 - 1, (n,), generator=g, dtype=torch.int32)
        if n:
            v[::97] = 2**31 - 1
    ref = torch.cumsum(v.to(torch.int64), 0)
    want_total = int(ref[-1]) if n else 0
    if kind == "large" and n > 2:
        assert want_total > 2**31
    cum, total, host = scan(cuda, v.to(cuda))
    assert torch.equal(cum.cpu(), ref)
    assert int(total.item()) == want_total and int(host[0]) == want_total
    if n == SCAN_TILE + 1:  # the pinned copy is optional
        cum, total, host = scan(cuda, v.to(cuda), pinned=False)
        assert torch.equal(cum.cpu(), ref) and int(total.item()) == want_total and host is None
