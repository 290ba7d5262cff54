"""CPU checks of the exact-marginal entry points: the two C-ABI exports are declared, exported and bound, and a NumPy restatement
of the kernel's work split (``marginal_args`` in qb_api.cu, ``marginal_kernel`` / ``marginal_reduce_kernel`` in qb_kernels.cuh)
adds every amplitude into exactly the bin ``Statevector.probabilities(qargs)`` puts it in, for any bit order, with rank bits."""
import numpy as np
import pytest

from tests.test_native_abi import header_functions

NEW = ("qb_marginal_probabilities", "qb_marginal_device")
ITEM_BITS = 16  # qb::kMargItemBits


def test_marginal_exports():
    import __graft_entry__ as entry

    entry.build()
    from queasars_b200 import _native

    lib = _native.load()
    declared = header_functions()
    for name in NEW:
        assert name in declared and name in _native.EXPORTED_SYMBOLS and hasattr(lib, name)
        assert getattr(lib, name).argtypes, f"{name} has no argument types"


def marginal_args(n_bits, index_offset, pos):
    """Mirror of qb_api.cu's marginal_args."""
    out_of = {p: j for j, p in enumerate(pos)}
    a = {"lane_bin": [0] * 5, "lane_sum": 0, "bin_fixed": 0, "fixed_mask": 0, "h": [], "v": []}
    for p in range(64):
        j = out_of.get(p, -1)
        if p < 5:
            if j >= 0:
                a["lane_bin"][p] = 1 << j
            elif p < n_bits:
                a["lane_sum"] |= 1 << p
        elif p < n_bits:
            (a["h"] if j >= 0 else a["v"]).append((p - 5, j))
        elif j >= 0:
            a["bin_fixed"] |= ((index_offset >> p) & 1) << j
            a["fixed_mask"] |= 1 << j
    a["slice_bits"] = min(len(a["v"]), max(0, ITEM_BITS - len(a["h"])))
    return a


def kernel_marginal(p, n_bits, index_offset, pos):
    """marginal_kernel (+ marginal_reduce_kernel) over the amplitudes' probabilities p, item by item."""
    a = marginal_args(n_bits, index_offset, pos)
    m, S, h, v = len(pos), a["slice_bits"], a["h"], a["v"]
    v_mask = sum(1 << c for c, _ in v)
    part = np.full((1 << m, 1 << S), np.nan)
    length = 1 << (len(v) - S)
    for item in range(1 << (len(h) + S)):
        t, s = item >> S, item & ((1 << S) - 1)
        hc = sum(1 << c for i, (c, _) in enumerate(h) if (t >> i) & 1)
        hb = sum(1 << j for i, (_, j) in enumerate(h) if (t >> i) & 1)
        start = s * length
        vc = sum(1 << c for i, (c, _) in enumerate(v) if (start >> i) & 1)
        acc = np.zeros(32)
        for _ in range(length):
            acc += p[((hc | vc) << 5) + np.arange(32)]
            vc = ((vc | ~v_mask) + 1) & v_mask
        for b in range(5):  # butterfly over the unmeasured lane bits
            if (a["lane_sum"] >> b) & 1:
                acc = acc + acc[np.arange(32) ^ (1 << b)]
        for lane in range(32):
            if lane & a["lane_sum"] == 0:
                bin_ = a["bin_fixed"] | hb | sum(a["lane_bin"][b] for b in range(5) if (lane >> b) & 1)
                assert np.isnan(part[bin_, s]), "a bin slot written twice"
                part[bin_, s] = acc[lane]
    bins = np.arange(1 << m)
    live = (bins & a["fixed_mask"]) == a["bin_fixed"]
    assert not np.isnan(part[live]).any(), "a bin of this shard was never written"
    return np.where(live, np.nan_to_num(part).sum(axis=1), 0.0)


def reference(p, n_bits, index_offset, pos):
    k = np.arange(p.size, dtype=np.int64) | index_offset
    b = np.zeros_like(k)
    for j, q in enumerate(pos):
        b |= ((k >> q) & 1) << j
    return np.bincount(b, weights=p, minlength=1 << len(pos))


@pytest.mark.parametrize("n_bits", [8, 11])
def test_work_split_covers_every_amplitude_once(n_bits):
    rng = np.random.default_rng(n_bits)
    p = rng.random(1 << n_bits)
    cases = [[0], [n_bits - 1], list(range(n_bits)), list(range(n_bits - 1, -1, -1)), [3, n_bits - 3, 1], [5, 6, 7],
             [int(q) for q in rng.permutation(n_bits)[:4]], [4, 0, n_bits - 2]]
    for pos in cases:
        assert np.allclose(kernel_marginal(p, n_bits, 0, pos), reference(p, n_bits, 0, pos), rtol=1e-13, atol=0), pos
    # a shard: rank bits n_bits and n_bits + 1 measured, this shard's pattern is 0b10
    offset = 2 << n_bits
    for pos in ([n_bits + 1, 0, n_bits], [n_bits, 2], [n_bits + 1] + list(range(n_bits))):
        got = kernel_marginal(p, n_bits, offset, pos)
        assert np.allclose(got, reference(p, n_bits, offset, pos), rtol=1e-13, atol=0), pos
