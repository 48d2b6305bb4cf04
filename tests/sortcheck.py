"""Independent answers for the outputs of a stable radix sort.

Three tools, none of which touches the library under test:

* ``radix_key`` / ``radix_key_torch``: the order-preserving map from typed key bits (signed, IEEE float, descending) to
  the unsigned key whose ascending order is the requested order -- the transform of the reference's HLSL path
  (GPUSortingD3D12/Shaders/SortCommon.hlsl:134-154 FloatToUint / IntToUint), with descending as the complement.
* ``stable_order`` (numpy, moderate n): the permutation a stable sort on the radix key (or on a bit range of it) applies.
* ``certify_stable_sort`` / ``certify_sorted_multiset`` (torch, any n, chunked int64 arithmetic on the tensors' own
  device): properties that together hold exactly when an output is THE stable sort of its input.  They bound their
  temporaries to a few chunks, so they work on outputs of more than 2^32 elements.
"""
from __future__ import annotations

import numpy as np
import torch

INT64_MIN = -(1 << 63)
U32 = 0xFFFFFFFF
DEFAULT_CHUNK = 1 << 27


# ---- the order: typed bits -> unsigned radix key -------------------------------------------------------------------
def radix_key(bits: np.ndarray, kind: str = "u", descending: bool = False) -> np.ndarray:
    """Unsigned key (same dtype as ``bits``: uint32 or uint64) whose ascending order is the requested order of the typed
    value: kind "u" unsigned, "i" two's complement, "f" IEEE float (total order: -NaN < -inf < ... < -0 < +0 < ... <
    +inf < +NaN, NaNs ordered by their payload bits)."""
    nb = bits.dtype.itemsize * 8
    u = bits.copy()
    sign = np.array(1 << (nb - 1), dtype=bits.dtype)
    if kind == "i":
        u ^= sign
    elif kind == "f":
        neg = (u >> np.array(nb - 1, dtype=bits.dtype)).astype(bool)
        u = np.where(neg, ~u, u | sign)
    if descending:
        u = ~u
    return u


def bit_field(u: np.ndarray, begin: int = 0, end: int | None = None) -> np.ndarray:
    """bits [begin, end) of unsigned keys, shifted down"""
    nb = u.dtype.itemsize * 8
    end = nb if end is None else end
    if end - begin == nb:
        return u
    return (u >> np.array(begin, dtype=u.dtype)) & np.array((1 << (end - begin)) - 1, dtype=u.dtype)


def stable_order(bits: np.ndarray, kind: str = "u", descending: bool = False, begin: int = 0,
                 end: int | None = None) -> np.ndarray:
    """Permutation applied by a stable sort of ``bits`` on bits [begin, end) of its radix key: the expected output is
    ``bits[order]`` and, for payload = input index, ``order`` itself."""
    return np.argsort(bit_field(radix_key(bits, kind, descending), begin, end), kind="stable")


def expected_plan(bits: np.ndarray, kind: str = "u", descending: bool = False, begin: int = 0, end: int | None = None,
                  skip: bool = True, hot: bool = True) -> tuple[int, int, int]:
    """(skip mask, hot mask, executed passes) the sort's device plan must report for this input: a digit place whose
    histogram has one non-empty bin is skipped; otherwise it is hot when one bin holds at least n/8 keys and n >= 2^22.
    Digits are taken from the radix key (what the histogram of a typed sort counts)."""
    u = radix_key(bits, kind, descending)
    nb = bits.dtype.itemsize * 8
    end = nb if end is None else end
    n = u.size
    skip_mask = hot_mask = 0
    places = (end - begin + 7) // 8
    for p in range(places):
        width = min(8, end - begin - 8 * p)
        d = bit_field(u, begin + 8 * p, begin + 8 * p + width).astype(np.int64)
        c = np.bincount(d, minlength=1 << width)
        if skip and c.max() == n:
            skip_mask |= 1 << p
        elif hot and n >= (1 << 22) and c.max() * 8 >= n:
            hot_mask |= 1 << p
    return skip_mask, hot_mask, places - bin(skip_mask).count("1")


def radix_key_torch(bits: torch.Tensor, kind: str = "u", descending: bool = False, begin: int = 0,
                    end: int | None = None) -> torch.Tensor:
    """Torch form of ``bit_field(radix_key(...))`` for 32-/64-bit containers (int32/int64 tensors holding the bits) on
    any device.  Returns int64 whose SIGNED ascending order is the requested order: 32-bit keys and bit ranges narrower
    than 64 bits come out as non-negative values, whole 64-bit keys with their top bit flipped."""
    if bits.element_size() == 4:
        u = bits.view(torch.int32).to(torch.int64) & U32
        sign, ones = 1 << 31, U32
        if kind == "i":
            u = u ^ sign
        elif kind == "f":
            u = torch.where(u >= sign, u ^ ones, u | sign)
        if descending:
            u = u ^ ones
        nb = 32
    else:
        t = bits.view(torch.int64)
        u = t
        if kind == "i":
            u = t ^ INT64_MIN
        elif kind == "f":
            u = torch.where(t < 0, ~t, t | INT64_MIN)
        if descending:
            u = ~u
        nb = 64
    end = nb if end is None else end
    if end - begin < nb:
        return (u >> begin) & ((1 << (end - begin)) - 1)  # non-negative: the mask drops any sign extension
    return u ^ INT64_MIN if nb == 64 else u


# ---- certificates ---------------------------------------------------------------------------------------------------
def _as_u32_index(p: torch.Tensor) -> torch.Tensor:
    return p.to(torch.int64) & U32 if p.dtype == torch.int32 else p.to(torch.int64)


def certify_nondecreasing(out_keys: torch.Tensor, kind: str = "u", descending: bool = False, begin: int = 0,
                          end: int | None = None, chunk: int = DEFAULT_CHUNK) -> None:
    """radix keys of ``out_keys`` never decrease, across chunk boundaries too"""
    n = out_keys.numel()
    for s in range(0, n, chunk):
        lo = max(s - 1, 0)
        r = radix_key_torch(out_keys[lo:min(s + chunk, n)], kind, descending, begin, end)
        bad = (r[1:] < r[:-1]).nonzero()
        assert bad.numel() == 0, f"order: output radix key decreases at index {lo + 1 + int(bad[0, 0])}"


def certify_stable_sort(in_keys: torch.Tensor, out_keys: torch.Tensor, out_payload: torch.Tensor, kind: str = "u",
                        descending: bool = False, begin: int = 0, end: int | None = None,
                        chunk: int = DEFAULT_CHUNK) -> None:
    """Raise AssertionError unless (out_keys, out_payload) is the stable sort of in_keys with payload = input index.

    Checks, chunk by chunk: (1) the output radix keys are non-decreasing; (2) the payload is a permutation of 0..n-1;
    (3) out_keys[j] == in_keys[payload[j]] bit for bit; (4) the payload ascends inside every run of equal radix keys.
    (2) and (3) make the output a rearrangement of the input that carries each key's origin, (1) makes it sorted and
    (4) puts equal keys in input order -- which is the definition of the stable sort."""
    n = in_keys.numel()
    assert out_keys.numel() == n and out_payload.numel() >= n, "sizes"
    assert in_keys.element_size() == out_keys.element_size(), "key widths"
    ik = in_keys.view(torch.int32 if in_keys.element_size() == 4 else torch.int64)
    ok = out_keys.view(ik.dtype)
    seen = torch.zeros(n, dtype=torch.bool, device=out_keys.device)
    for s in range(0, n, chunk):
        e = min(s + chunk, n)
        lo = max(s - 1, 0)
        p = _as_u32_index(out_payload[lo:e])
        pc = p[s - lo:]
        rng = ((pc < 0) | (pc >= n)).nonzero()
        assert rng.numel() == 0, f"permutation: payload {int(pc[int(rng[0, 0])])} at index {s + int(rng[0, 0])} is not an index"
        seen[pc] = True
        mism = (ik[pc] != ok[s:e]).nonzero()
        assert mism.numel() == 0, f"payload: output key at index {s + int(mism[0, 0])} is not the input key its payload names"
        r = radix_key_torch(ok[lo:e], kind, descending, begin, end)
        down = (r[1:] < r[:-1]).nonzero()
        assert down.numel() == 0, f"order: output radix key decreases at index {lo + 1 + int(down[0, 0])}"
        unstable = ((r[1:] == r[:-1]) & (p[1:] <= p[:-1])).nonzero()
        assert unstable.numel() == 0, f"stability: equal keys out of input order at index {lo + 1 + int(unstable[0, 0])}"
        del p, pc, r
    missing = (~seen).nonzero()
    assert missing.numel() == 0, f"permutation: input index {int(missing[0, 0])} never appears in the payload"


def bincount_chunked(t: torch.Tensor, bin_of, nbins: int, chunk: int = DEFAULT_CHUNK) -> torch.Tensor:
    """int64 counts of ``bin_of(chunk)`` over the whole tensor; every bin index must lie in [0, nbins)"""
    counts = torch.zeros(nbins, dtype=torch.int64, device=t.device)
    for s in range(0, t.numel(), chunk):
        b = bin_of(t[s:s + chunk])
        out = ((b < 0) | (b >= nbins)).nonzero()
        assert out.numel() == 0, f"multiset: element {s + int(out[0, 0])} falls outside the input's {nbins} values"
        counts += torch.bincount(b, minlength=nbins)
    return counts


def certify_sorted_multiset(in_counts: torch.Tensor, out_keys: torch.Tensor, bin_of, kind: str = "u",
                            descending: bool = False, chunk: int = DEFAULT_CHUNK) -> None:
    """Keys-only outputs: non-decreasing radix keys and the input's multiset, which together pin the output down.
    ``bin_of`` maps a chunk of keys to int64 bin indices and must be injective on all keys of that width (not only on the
    input's), e.g. a bijection onto a range the input fills; ``in_counts`` is ``bincount_chunked`` of the input."""
    certify_nondecreasing(out_keys, kind, descending, chunk=chunk)
    got = bincount_chunked(out_keys, bin_of, in_counts.numel(), chunk)
    diff = (got != in_counts).nonzero()
    assert diff.numel() == 0, f"multiset: value bin {int(diff[0, 0])} occurs {int(got[diff[0, 0]])} times, input had {int(in_counts[diff[0, 0]])}"
