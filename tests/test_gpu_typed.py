"""Typed keys and descending order (SURVEY 8f rank 1): the order-preserving bit transforms of the reference's HLSL path
(GPUSortingD3D12/Shaders/SortCommon.hlsl:134-154 FloatToUint / IntToUint, :594-656 descending) fused into the first
and last OneSweep pass.  Oracle: numpy restatement of those transforms + a stable argsort.  -m gpu"""
import zlib

import numpy as np
import pytest
import torch

from tests.sortcheck import radix_key as to_radix

pytestmark = pytest.mark.gpu


CASES = [("u32", np.uint32, "u"), ("i32", np.uint32, "i"), ("f32", np.uint32, "f"),
         ("u64", np.uint64, "u"), ("i64", np.uint64, "i"), ("f64", np.uint64, "f")]


def make_bits(rng, n, dtype, kind):
    if kind == "f":
        f = rng.standard_normal(n).astype(np.float32 if dtype == np.uint32 else np.float64) * 1e3
        f[:8] = [0.0, -0.0, np.inf, -np.inf, 1.0, -1.0, 1e-30, -1e-30]
        f[8:16] = f[:8]  # duplicates
        return f.view(dtype).copy()
    hi = np.iinfo(dtype).max
    b = rng.integers(0, hi, n, dtype=dtype, endpoint=True)
    b[:4] = [0, hi, hi >> 1, (hi >> 1) + 1]
    return b


@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("name,dtype,kind", CASES)
def test_typed_keys(name, dtype, kind, descending):
    import gpusorting_b200 as g

    rng = np.random.default_rng(zlib.crc32(name.encode()) & 0xFFFF)  # the same seed in every process
    kb = np.dtype(dtype).itemsize
    s = g.OneSweepSorter(1 << 20, kb, 0)
    T = s.info("tile_keys")
    for n in (1, 2, 1000, T + 17, 3 * T + 5, 1 << 20):
        n = max(n, 16)
        bits = make_bits(rng, n, dtype, kind)
        want = bits[np.argsort(to_radix(bits, kind, descending), kind="stable")]
        t = torch.from_numpy(bits.view(np.int32 if kb == 4 else np.int64).copy()).cuda()
        s.sort_keys_typed(t, name, descending)
        got = t.cpu().numpy().view(dtype)
        assert np.array_equal(got, want), f"{name} desc={descending} n={n}"
        if kind == "f":  # sanity against numpy's own float sort (no NaNs here)
            fl = got.view(np.float32 if kb == 4 else np.float64)
            assert np.all(fl[1:] <= fl[:-1]) if descending else np.all(fl[1:] >= fl[:-1])
    s.close()


@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("name,kind", [("i32", "i"), ("f32", "f"), ("u32", "u")])
def test_typed_pairs_are_stable_both_directions(name, kind, descending):
    import gpusorting_b200 as g

    rng = np.random.default_rng(7)
    n = 300007
    s = g.OneSweepSorter(n, 4, 4)
    if kind == "f":
        bits = rng.integers(-50, 50, n).astype(np.float32).view(np.uint32).copy()  # many ties, both signs, +-0
    else:
        bits = (rng.integers(0, 200, n).astype(np.int64) - 100).astype(np.int32).view(np.uint32).copy()
        if kind == "u":
            bits &= np.uint32(0xFF)
    order = np.argsort(to_radix(bits, kind, descending), kind="stable")
    tk = torch.from_numpy(bits.view(np.int32).copy()).cuda()
    tv = torch.arange(n, dtype=torch.int32, device="cuda")
    s.sort_pairs_typed(tk, tv, name, descending)
    assert np.array_equal(tk.cpu().numpy().view(np.uint32), bits[order])
    assert np.array_equal(tv.cpu().numpy().astype(np.int64), order)  # ties keep input order in BOTH directions
    s.close()


def test_typed_argument_checks():
    import gpusorting_b200 as g

    s = g.OneSweepSorter(1024, 4, 0)
    t = torch.zeros(64, dtype=torch.int32, device="cuda")
    with pytest.raises(g.OneSweepError):
        s.sort_keys_typed(t, "i64")  # width mismatch
    s.set_option("variant", 0)
    with pytest.raises(g.OneSweepError):
        s.sort_keys_typed(t, "i32")  # only the default kernel carries the codec
    s.close()
