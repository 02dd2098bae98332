"""Parity of the hand-written sm_100a kernels (through the C ABI) against the CPU oracle.

Bars: bit-exact for tree contents, sampled indices and gathered bytes; GAE within rtol=atol=1e-5 of the
float64 evaluation of the recurrence (and exactly the reference's own tolerance 1e-4 against the golden
vectors produced by the reference's two fp32 code paths).
"""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import per_oracle as po

pytestmark = pytest.mark.gpu
GOLD = Path(__file__).parent / "golden"


def dev():
    return torch.device("cuda", 0)


# ---------------------------------------------------------------------------------------------------- trees
def _heap_equal(dev_tree, orc_tree):
    got = dev_tree.values.cpu().numpy()
    want = orc_tree.values()
    np.testing.assert_array_equal(got[1:], want[1:])


@pytest.mark.parametrize("size", [1, 2, 7, 16, 100, 1000, 1024, 4097, 100_000])
def test_tree_update_matches_oracle_bitwise(cuda_backend, size):
    from rl_b200.data.segment_tree import MinSegmentTreeFp32, SumSegmentTreeFp32

    rng = np.random.default_rng(size)
    ds, dm = SumSegmentTreeFp32(size, dev()), MinSegmentTreeFp32(size, dev())
    os_, om = po.OracleTree(size, False), po.OracleTree(size, True)
    assert ds.capacity == os_.capacity
    _heap_equal(ds, os_)
    _heap_equal(dm, om)
    for n in [1, 3, 33, 256, 1000, 1024, 1025, 5000]:
        idx = rng.integers(0, size, n).astype(np.int64)  # duplicates: last writer must win
        val = (rng.random(n, dtype=np.float32) * 3 + 1e-3).astype(np.float32)
        for t in (os_, om):
            t[idx] = val
        ti, tv = torch.from_numpy(idx).to(dev()), torch.from_numpy(val).to(dev())
        ds[ti] = tv
        dm[ti] = tv
        _heap_equal(ds, os_)
        _heap_equal(dm, om)
    # scalar value overload + negative ("skip") indices
    idx = rng.integers(0, size, 17).astype(np.int64)
    os_[idx] = 0.25
    ds[torch.from_numpy(idx).to(dev())] = torch.tensor(0.25, device=dev())
    _heap_equal(ds, os_)


@pytest.mark.parametrize("size", [1, 2, 7, 16, 1000, 4097, 100_000, 1_000_000])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_tree_update_range_matches_oracle_bitwise(cuda_backend, size, dtype):
    """rlb_tree_update_range (closed-form fill + boundary chain) against the reference's index-by-index update: whole
    heaps bit-equal, for plain / wrapping / full / single-slot ranges on top of random earlier contents."""
    from rl_b200 import ops
    from rl_b200.data.segment_tree import (MinSegmentTreeFp32, MinSegmentTreeFp64, SumSegmentTreeFp32,
                                           SumSegmentTreeFp64)

    f64 = dtype == torch.float64
    rng = np.random.default_rng(size + f64)
    ds = (SumSegmentTreeFp64 if f64 else SumSegmentTreeFp32)(size, dev())
    dm = (MinSegmentTreeFp64 if f64 else MinSegmentTreeFp32)(size, dev())
    npdt = np.float64 if f64 else np.float32

    class NpTree:
        """fp64 has no compiled reference here: every node an update touches ends as op(children)
        (segment_tree.h:83-139), so the heap is rebuilt level by level from the leaves; untouched nodes keep the
        identity, which op(identity, identity) reproduces."""

        def __init__(self, is_min):
            self.is_min = is_min
            self.h = np.full(2 * ds.capacity, np.finfo(np.float64).max if is_min else 0.0)

        def __setitem__(self, ix, v):
            cap = ds.capacity
            self.h[cap + ix] = v
            w = cap // 2
            while w >= 1:
                a, b = self.h[2 * w:4 * w:2], self.h[2 * w + 1:4 * w:2]
                self.h[w:2 * w] = np.minimum(a, b) if self.is_min else a + b
                w //= 2

        def values(self):
            return self.h

    os_, om = (NpTree(False), NpTree(True)) if f64 else (po.OracleTree(size, False), po.OracleTree(size, True))
    n0 = min(size, 5000)
    idx = rng.integers(0, size, n0).astype(np.int64)
    val = (rng.random(n0) * 3 + 1e-3).astype(npdt)
    for t in (os_, om):
        t[idx] = val
    ds[torch.from_numpy(idx).to(dev())] = torch.from_numpy(val).to(dev())
    dm[torch.from_numpy(idx).to(dev())] = torch.from_numpy(val).to(dev())
    cases = [(0, 1), (size - 1, 1), (0, size), (size // 2, size), (size // 3, max(1, size // 2)), (size - 1, 2),
             (0, max(1, size - 1)), (size // 2, max(1, size // 2 + 1))]
    cases += [(int(rng.integers(0, size)), int(rng.integers(1, size + 1))) for _ in range(6)]
    for start, n in cases:
        n = min(n, size)
        v = npdt(rng.random() * 2 + 1e-3)
        ix = (start + np.arange(n, dtype=np.int64)) % size
        for t in (os_, om):
            t[ix] = v
        value = torch.tensor(v, dtype=dtype, device=dev())
        cuda_backend.tree_update_range(ops.RangeUpdate(ds.values, dm.values, ds.capacity, ops.RANGE_VALUE, value),
                                       start, n, size)
        _heap_equal(ds, os_)
        _heap_equal(dm, om)
    # a single tree (the segment-tree classes' own use)
    cuda_backend.tree_update_range(ops.RangeUpdate(ds.values, None, ds.capacity, ops.RANGE_VALUE,
                                                   torch.tensor(0.5, dtype=dtype, device=dev())), 0, size, size)
    os_[np.arange(size, dtype=np.int64)] = npdt(0.5)
    _heap_equal(ds, os_)
    _heap_equal(dm, om)


@pytest.mark.parametrize("alpha", [0.6, 0.5, 1.0])
def test_range_default_priority_matches_oracle_sampler(cuda_backend, alpha):
    """mark_update of writer batches through the range kernel (default priority computed in the kernel, double pow,
    running max through the ticket) == the restated reference sampler, leaf for leaf, across many extends."""
    from rl_b200.data import PrioritizedSampler

    N = 5000
    smp = PrioritizedSampler(N, alpha, 0.4, device=dev())
    orc = po.OraclePrioritizedSampler(N, alpha, 0.4)
    rng = np.random.default_rng(3)
    cursor = 0
    for it in range(12):
        n = int(rng.integers(1, 3000))
        smp.mark_update_range(cursor, n, N)
        orc.mark_update(torch.arange(cursor, cursor + n) % N)
        cursor = (cursor + n) % N
        got_s, got_m = smp._sum_tree.values.cpu().numpy(), smp._min_tree.values.cpu().numpy()
        if alpha == 1.0:            # no transcendental: the CPU restatement is exact.  (torch's CPU sqrt / pow are not
                                    # correctly rounded -- 0.7 % of fp32 inputs differ from IEEE sqrt -- so for any
                                    # other alpha CPU and CUDA leaves differ by an ulp in the reference itself)
            np.testing.assert_array_equal(got_s[1:], orc._sum_tree.values()[1:])
            np.testing.assert_array_equal(got_m[1:], orc._min_tree.values()[1:])
            assert float(smp._max_priority_buf[0]) == float(torch.as_tensor(orc._max_priority, dtype=torch.float32))
        else:                       # CUDA powf vs glibc powf: leaves agree to an ulp, the heap is exact for ITS leaves
            cap = smp._sum_tree.capacity
            np.testing.assert_allclose(got_s[cap:cap + N], orc._sum_tree.values()[cap:cap + N], rtol=1e-6)
            ts, tm = po.OracleTree(N, False), po.OracleTree(N, True)
            ts.load_leaves(got_s[cap:cap + N])
            tm.load_leaves(got_m[cap:cap + N])
            np.testing.assert_array_equal(got_s[1:], ts.values()[1:])
            np.testing.assert_array_equal(got_m[1:], tm.values()[1:])
            np.testing.assert_allclose(float(smp._max_priority_buf[0]), float(orc._max_priority), rtol=1e-6)
        if it % 3 == 2:       # raise / keep the running max so that the default priority moves
            k = int(rng.integers(1, 200))
            idx = torch.from_numpy(rng.integers(0, N, k))
            pr = torch.from_numpy((rng.random(k) * (it + 1)).astype(np.float32))
            smp.update_priority(idx.to(dev()), pr.to(dev()))
            orc.update_priority(idx, pr)
    assert int(smp._range_ticket.item()) == 0


def test_range_default_follows_the_running_max_on_replay(cuda_backend):
    """The range kernel decides "no priority seen yet" on the device: a launch captured before any priority exists
    gives the initial default, and the SAME graph replayed after a write-back gives (max + eps) ** alpha; updates made of
    "skip" markers only leave the max unset, as in the reference."""
    from rl_b200.data import PrioritizedSampler

    N = 1000
    smp = PrioritizedSampler(N, 1.0, 0.4, device=dev())
    smp.update_priority(torch.tensor([-1, -1], device=dev()), torch.tensor([3.0, 4.0], device=dev()))   # skips only
    side = torch.cuda.Stream(dev())
    gr = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        with torch.cuda.graph(gr, stream=side):
            smp.mark_update_range(0, 100, N)
    gr.replay()
    torch.cuda.synchronize()
    eps = np.float32(1e-8)
    first = np.float32(np.float32(1 + 1e-8) + eps)
    leaves = smp._sum_tree.dump_leaves().cpu().numpy()
    assert (leaves[:100] == first).all() and (leaves[100:] == 0).all()
    smp.update_priority(torch.tensor([5], device=dev()), torch.tensor([7.0], device=dev()))
    gr.replay()
    torch.cuda.synchronize()
    leaves = smp._sum_tree.dump_leaves().cpu().numpy()
    want = np.float32(np.float32(np.float32(7.0) + eps) + eps)
    assert (leaves[:100] == want).all()
    assert float(smp._max_priority_buf[0]) == float(np.float32(np.float32(7.0) + eps))   # the default itself is a raw priority


@pytest.mark.parametrize("size", [3, 1000, 2047, 2048, 4095, 5000, 1_000_000, 3_000_000])
def test_tree_rebuild_matches_oracle(cuda_backend, size):
    """rlb_tree_rebuild (eleven levels per launch over 2048-leaf tiles, dense levels above, single-CTA top) from random
    leaves: every internal node bit-equal to the reference tree holding the same leaves; fp64 against numpy."""
    from rl_b200.data.segment_tree import (MinSegmentTreeFp32, MinSegmentTreeFp64, SumSegmentTreeFp32,
                                           SumSegmentTreeFp64)

    rng = np.random.default_rng(size)
    leaves = (rng.random(size) * 5 + 1e-3).astype(np.float32)
    for cls, is_min in ((SumSegmentTreeFp32, False), (MinSegmentTreeFp32, True)):
        t = cls(size, dev())
        t.load_leaves(torch.from_numpy(leaves).to(dev()))
        o = po.OracleTree(size, is_min)
        o.load_leaves(leaves)
        np.testing.assert_array_equal(t.values.cpu().numpy()[1:], o.values()[1:])
    l64 = rng.random(size) * 5 + 1e-3
    for cls, is_min in ((SumSegmentTreeFp64, False), (MinSegmentTreeFp64, True)):
        t = cls(size, dev())
        t.load_leaves(torch.from_numpy(l64).to(dev()))
        cap = t.capacity
        h = np.full(2 * cap, np.finfo(np.float64).max if is_min else 0.0)
        h[cap:cap + size] = l64
        w = cap // 2
        while w >= 1:
            a, b = h[2 * w:4 * w:2], h[2 * w + 1:4 * w:2]
            h[w:2 * w] = np.minimum(a, b) if is_min else a + b
            w //= 2
        np.testing.assert_array_equal(t.values.cpu().numpy()[1:], h[1:])


def test_tree_kat_and_queries(cuda_backend):
    # test/rb/test_prioritized.py:113-140
    from rl_b200.data.segment_tree import MinSegmentTreeFp32, SumSegmentTreeFp32

    s, m = SumSegmentTreeFp32(16, dev()), MinSegmentTreeFp32(16, dev())
    idx = torch.tensor([0, 3, 4, 7, 12, 15], device=dev())
    val = torch.tensor([1, 2, 4, 8, 16, 32], dtype=torch.float32, device=dev())
    s[idx] = val
    m[idx] = val
    assert s.capacity == 32
    l = torch.tensor([0, 3, 4, 7], device=dev())
    r = torch.tensor([16, 8, 13, 16], device=dev())
    assert s.query(l, r).tolist() == [63, 14, 28, 56]
    assert m.query(l, r).tolist() == [1, 2, 4, 8]
    assert s.query(l, r, root_fast_path=False).tolist() == [63, 14, 28, 56]
    assert s.scan_lower_bound(torch.tensor([0.5, 1.0, 2.9, 7.1, 30.0], device=dev())).tolist() == [0, 0, 3, 7, 12]
    assert s.scan_lower_bound(64.0) == 16
    assert s.query(0, 16) == 63.0 and s[3] == 2.0
    np.testing.assert_array_equal(s[np.array([0, 3, 15])], [1, 2, 32])


@pytest.mark.parametrize("size", [5, 1000, 70_000, 1_000_000])
def test_scan_query_at_match_oracle(cuda_backend, size):
    from rl_b200.data.segment_tree import MinSegmentTreeFp32, SumSegmentTreeFp32

    rng = np.random.default_rng(size + 1)
    leaves = (rng.random(size, dtype=np.float32) ** 3 + 1e-6).astype(np.float32)
    leaves[rng.integers(0, size, max(size // 50, 1))] = 0.0  # some empty slots
    ds, dm = SumSegmentTreeFp32(size, dev()), MinSegmentTreeFp32(size, dev())
    os_, om = po.OracleTree(size, False), po.OracleTree(size, True)
    for t in (os_, om):
        t.load_leaves(leaves)
    ds.load_leaves(torch.from_numpy(leaves))
    dm.load_leaves(torch.from_numpy(leaves))
    _heap_equal(ds, os_)
    _heap_equal(dm, om)
    root = np.float32(os_.query(0, size))
    mass = (rng.random(20_000, dtype=np.float32) * root * np.float32(1.02)).astype(np.float32)
    got = ds.scan_lower_bound(torch.from_numpy(mass).to(dev())).cpu().numpy()
    np.testing.assert_array_equal(got, os_.scan_lower_bound(mass))
    l = rng.integers(0, size, 300).astype(np.int64)
    r = np.minimum(l + rng.integers(1, size + 1, 300), size).astype(np.int64)
    tl, tr = torch.from_numpy(l).to(dev()), torch.from_numpy(r).to(dev())
    np.testing.assert_array_equal(ds.query(tl, tr).cpu().numpy(), os_.query(l, r))
    np.testing.assert_array_equal(dm.query(tl, tr).cpu().numpy(), om.query(l, r))
    np.testing.assert_array_equal(ds.query(tl, tr, root_fast_path=False).cpu().numpy(), os_.query(l, r, walk=True))
    probe = rng.integers(0, size, 100).astype(np.int64)
    np.testing.assert_array_equal(ds[torch.from_numpy(probe).to(dev())].cpu().numpy(), os_[probe])


def test_tree_fp64(cuda_backend):
    from rl_b200.data.segment_tree import SumSegmentTreeFp64

    size = 3000
    rng = np.random.default_rng(0)
    t = SumSegmentTreeFp64(size, dev())
    leaves = rng.random(size)
    t[torch.arange(size, device=dev())] = torch.from_numpy(leaves).to(dev())
    heap = t.values.cpu().numpy()
    cap = t.capacity
    want = np.zeros(2 * cap)
    want[cap:cap + size] = leaves
    for i in range(cap - 1, 0, -1):
        want[i] = want[2 * i] + want[2 * i + 1]
    np.testing.assert_array_equal(heap[1:], want[1:])
    mass = rng.random(500) * want[1]
    got = t.scan_lower_bound(torch.from_numpy(mass).to(dev())).cpu().numpy()
    ref = []
    for v in mass:
        node, cur = 1, v
        while node < cap:
            node <<= 1
            if cur > want[node]:
                cur -= want[node]
                node |= 1
        ref.append(node ^ cap)
    np.testing.assert_array_equal(got, ref)


# ---------------------------------------------------------------------------------------------------- PER sample
def test_per_sample_golden(cuda_backend):
    """Committed golden vectors from the compiled reference trees (tests/golden/make_golden.py)."""
    from rl_b200.data.samplers import PrioritizedSampler
    from rl_b200.data.storages import Storage

    z = np.load(GOLD / "per_golden.npz")
    for k in sorted({n.split("/")[0] for n in z.files}):
        N, filled, B = (int(x) for x in z[f"{k}/meta"])
        alpha, beta = (float(x) for x in z[f"{k}/ab"])
        smp = PrioritizedSampler(N, alpha, beta, device=dev())
        # replay the same writes: default priorities for [0, filled) then the explicit update (with duplicates)
        smp.mark_update(torch.arange(filled, device=dev()))
        smp.update_priority(torch.from_numpy(z[f"{k}/upd_index"]).to(dev()),
                            torch.from_numpy(z[f"{k}/upd_priority"]).to(dev()))
        got_leaves = smp._sum_tree.dump_leaves().cpu().numpy()
        # leaves come from powf on the device vs SLEEF pow in the reference: allow 1-ulp, then force identical
        # leaves so that the index comparison is exact
        np.testing.assert_allclose(got_leaves, z[f"{k}/leaves"], rtol=3e-7, atol=0)
        smp._sum_tree.load_leaves(torch.from_numpy(z[f"{k}/leaves"]))
        min_leaves = z[f"{k}/leaves"].copy()
        min_leaves[filled:] = np.finfo(np.float32).max
        smp._min_tree.load_leaves(torch.from_numpy(min_leaves))
        u = torch.from_numpy(z[f"{k}/u"]).to(dev())
        idx, w, leaf, pp = cuda_backend.per_sample(smp._sum_tree.values, smp._min_tree.values, N,
                                                   smp._sum_tree.capacity, filled, u, beta, True, want_aux=True)
        assert pp[0].item() == z[f"{k}/p_sum"] and pp[1].item() == z[f"{k}/p_min"], k
        np.testing.assert_array_equal(idx.cpu().numpy(), z[f"{k}/index"])       # index-exact
        np.testing.assert_allclose(w.cpu().numpy(), z[f"{k}/weight"], rtol=2e-6)  # powf vs SLEEF


@pytest.mark.parametrize("size,filled,B", [(16, 16, 64), (1000, 313, 256), (1_000_000, 1_000_000, 256),
                                           (1_000_000, 400_000, 4096), (3_000_000, 3_000_000, 65536),
                                           # group-cooperative descent: 1 / 2 / 3 / 4 samples per single-warp CTA (groups
                                           # of 32 / 16 / 8 lanes), tree depths that leave 1 .. 15 levels below the staged top
                                           (6_250_000, 6_250_000, 256), (6_250_000, 5_000_000, 512), (600, 600, 300),
                                           (1100, 1100, 37), (3000, 2999, 800), (300_000, 300_000, 1100),
                                           (70_000, 70_000, 128), (2_100_000, 2_100_000, 600)])
@pytest.mark.parametrize("cpu_sem", [True, False])
def test_per_sample_matches_oracle(cuda_backend, size, filled, B, cpu_sem):
    from rl_b200.data.segment_tree import MinSegmentTreeFp32, SumSegmentTreeFp32

    rng = np.random.default_rng(size + B)
    leaves = np.zeros(size, dtype=np.float32)
    leaves[:filled] = ((rng.random(filled, dtype=np.float32) + 1e-8) ** np.float32(0.6)).astype(np.float32)
    if filled > 100:
        leaves[rng.integers(0, filled, filled // 100)] = 0.0
    leaves[0] = 0.5  # u == 0 lands on leaf 0; keep it positive so the CPU back-off loop cannot underflow
    ds, dm = SumSegmentTreeFp32(size, dev()), MinSegmentTreeFp32(size, dev())
    os_, om = po.OracleTree(size, False), po.OracleTree(size, True)
    min_leaves = np.where(np.arange(size) < filled, np.maximum(leaves, np.float32(1e-6)), np.finfo(np.float32).max)
    min_leaves = min_leaves.astype(np.float32)
    os_.load_leaves(leaves)
    om.load_leaves(min_leaves)
    ds.load_leaves(torch.from_numpy(leaves))
    dm.load_leaves(torch.from_numpy(min_leaves))
    u = rng.random(B, dtype=np.float32)
    u[:3] = [0.0, np.float32(1.0) - np.float32(2 ** -24), 0.5]
    want_idx, want_w, p_sum, p_min = po.per_sample_c(os_, om, filled, u, 0.4, cpu_checks=cpu_sem,
                                                     walk_query=not cpu_sem)
    idx, w, leaf, pp = cuda_backend.per_sample(ds.values, dm.values, size, ds.capacity, filled,
                                               torch.from_numpy(u).to(dev()), 0.4, cpu_sem, want_aux=True)
    assert pp[0].item() == p_sum and pp[1].item() == p_min
    np.testing.assert_array_equal(idx.cpu().numpy(), want_idx)
    np.testing.assert_allclose(w.cpu().numpy(), want_w, rtol=2e-6)
    # the weight is torch's own CUDA pow on the same operands, bit for bit.  CPU semantics: a true division (what the
    # reference's CPU branch computes); CUDA semantics: p_min is a Python float there, and ATen's CUDA division by a
    # CPU scalar multiplies by its reciprocal
    tw = torch.pow(leaf / pp[1], -0.4) if cpu_sem else torch.pow(leaf / pp[1].item(), -0.4)
    assert torch.equal(tw, w)


def test_fused_pow_is_torch_pow(cuda_backend):
    """(p + eps) ** alpha inside rlb_per_update == torch.pow on the device, bitwise, incl. the special exponents."""
    from rl_b200.data.samplers import PrioritizedSampler

    N = 50_000
    g = torch.Generator(device=dev()).manual_seed(0)
    p = torch.rand(N, device=dev(), generator=g) * 5
    for alpha in (0.6, 0.7, 0.5, 1.0, 2.0, 0.0, 3.0):
        smp = PrioritizedSampler(N, alpha, 0.4, device=dev())
        smp.update_priority(torch.arange(N, device=dev()), p)
        want = torch.pow(p + 1e-8, alpha)
        assert torch.equal(smp._sum_tree.dump_leaves(), want), alpha
        assert smp._max_priority[0].item() == p.max().item()


# ---------------------------------------------------------------------------------------------------- gather / scatter
SHAPES = [((4, 84, 84), torch.uint8), ((), torch.float32), ((1,), torch.int64), ((), torch.bool),
          ((17,), torch.float32), ((376,), torch.float32), ((3, 5), torch.float16), ((7,), torch.uint8),
          ((33,), torch.int16), ((2, 3), torch.float64)]


def _rand_leaf(n, shape, dtype, g):
    if dtype in (torch.uint8, torch.int16, torch.int64):
        return torch.randint(0, 100, (n, *shape), device=dev(), generator=g).to(dtype)
    if dtype == torch.bool:
        return torch.rand((n, *shape), device=dev(), generator=g) < 0.5
    return torch.randn((n, *shape), device=dev(), generator=g).to(dtype)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("N,B", [(50, 1), (300, 7), (5000, 256), (5000, 1024), (20000, 4099)])
def test_gather_matches_torch_indexing(cuda_backend, mode, N, B):
    g = torch.Generator(device=dev()).manual_seed(N + B)
    leaves = [_rand_leaf(N, s, d, g) for s, d in SHAPES]
    length = N - N // 7
    idx = torch.randint(-length, length, (B,), device=dev(), generator=g)
    status = torch.zeros(1, dtype=torch.int32, device=dev())
    out = cuda_backend.gather(leaves, idx, length, mode=mode, status=status)
    for leaf, o in zip(leaves, out):
        assert o.dtype == leaf.dtype and torch.equal(o, leaf[:length][idx])
    assert status.item() == 0
    # byte-level C restatement on one leaf
    np.testing.assert_array_equal(out[0].cpu().numpy(),
                                  po.gather_rows(leaves[0].cpu().numpy(), idx.cpu().numpy(), length))


def test_gather_oob_is_reported(cuda_backend):
    src = [torch.arange(100, device=dev(), dtype=torch.float32).reshape(50, 2)]
    status = torch.zeros(1, dtype=torch.int32, device=dev())
    cuda_backend.gather(src, torch.tensor([0, 49, 50], device=dev()), 50, status=status)
    assert status.item() & 1


def test_gather_strided_rows(cuda_backend):
    # storage leaf that is a column-slice view: rows are contiguous but the row stride is larger
    base = torch.randn(1000, 64, device=dev())
    view = base[:, :32]
    idx = torch.randint(0, 1000, (300,), device=dev())
    (o,) = cuda_backend.gather([view], idx, 1000)
    assert torch.equal(o, view[idx])


@pytest.mark.parametrize("B", [256, 4096])
def test_gather_atari_full_rows(cuda_backend, B):
    """C2-shaped: the bulk-DMA role on 28 224-byte rows, pixels + next pixels + small leaves in one launch."""
    N = 20_000
    g = torch.Generator(device=dev()).manual_seed(B)
    pix = torch.randint(0, 255, (N, 4, 84, 84), device=dev(), generator=g, dtype=torch.uint8)
    nxt = torch.randint(0, 255, (N, 4, 84, 84), device=dev(), generator=g, dtype=torch.uint8)
    act = torch.randint(0, 18, (N, 1), device=dev(), generator=g)
    rew = torch.randn(N, device=dev(), generator=g)
    done = torch.rand(N, 1, device=dev(), generator=g) < 0.1
    leaves = [pix, nxt, act, rew, done]
    idx = torch.randint(0, N, (B,), device=dev(), generator=g)
    for mode in (0, 1, 2):
        out = cuda_backend.gather(leaves, idx, N, mode=mode)
        for leaf, o in zip(leaves, out):
            assert torch.equal(o, leaf[idx]), mode


def test_scatter_matches_index_put(cuda_backend):
    g = torch.Generator(device=dev()).manual_seed(3)
    N, B = 4000, 777
    leaves = [_rand_leaf(N, s, d, g) for s, d in SHAPES]
    want = [l.clone() for l in leaves]
    data = [_rand_leaf(B, s, d, g) for s, d in SHAPES]
    idx = torch.randperm(N, device=dev(), generator=g)[:B]
    cuda_backend.scatter(leaves, data, idx, N)
    for w, d, l in zip(want, data, leaves):
        w[idx] = d
        assert torch.equal(w, l)


# ---------------------------------------------------------------------------------------------------- GAE
def _gae_inputs(shape, seed, p=0.05, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    v, nv, r = (torch.randn(*shape, generator=g, dtype=dtype) for _ in range(3))
    term = torch.rand(*shape, generator=g) < p
    done = term | (torch.rand(*shape, generator=g) < p)
    return v, nv, r, done, term


@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 5, 1), (3, 200, 1), (7, 3, 3, 1), (64, 128, 1), (9, 131, 1),
                                   (2, 1000, 1), (4096, 128, 1), (5, 33, 3), (16, 64, 40), (300, 500, 1),
                                   # few rows / long T: CTA per row, warp per tile (benchmarks/test_objectives_benchmarks.py:122-153),
                                   # several chunks of 16 tiles, ragged last tile, scalar (unaligned T) path, warp-per-CTA rows
                                   (32, 512, 1), (1, 512, 1), (3, 4100, 1), (2, 2049, 1), (5, 257, 1), (700, 129, 1),
                                   (400, 64, 1),
                                   # narrow feature dims: a warp per (row, feature) column; short T and wide F: the column kernel
                                   (37, 300, 2), (256, 128, 4), (3, 1000, 16), (11, 15, 4), (6, 40, 17), (5, 64, 3), (9, 516, 3), (2, 132, 4),
                                   (7, 130, 2)])
@pytest.mark.parametrize("gamma,lmbda", [(0.99, 0.95), (0.5, 0.1)])
def test_gae_matches_f64_oracle(cuda_backend, shape, gamma, lmbda):
    from rl_b200.objectives.value import generalized_advantage_estimate, vec_generalized_advantage_estimate

    v, nv, r, done, term = _gae_inputs(shape, sum(shape))
    g, l = torch.tensor(gamma), torch.tensor(lmbda)
    fa, ft = po.gae_f64(g, l, v, nv, r, done, term)
    cu = [x.to(dev()) for x in (v, nv, r, done, term)]
    a, t = vec_generalized_advantage_estimate(g, l, *cu[:3], done=cu[3], terminated=cu[4])
    torch.testing.assert_close(a.cpu().double(), fa, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(t.cpu().double(), ft, rtol=1e-5, atol=1e-5)
    # and against the reference's own fp32 loop semantics (C restatement, bit-exact to the reference)
    la, lt = po.gae_f32(g, l, v, nv, r, done, term)
    torch.testing.assert_close(a.cpu(), la, rtol=1e-5, atol=1e-5)
    a2, t2 = generalized_advantage_estimate(g, l, *cu[:3], done=cu[3], terminated=cu[4])
    assert torch.equal(a, a2) and torch.equal(t, t2)


def test_gae_golden(cuda_backend):
    from rl_b200.objectives.value import vec_generalized_advantage_estimate

    z = np.load(GOLD / "gae_golden.npz")
    for k in sorted({n.split("/")[0] for n in z.files}):
        gt = lambda n: torch.from_numpy(z[f"{k}/{n}"])
        cu = [gt(n).to(dev()) for n in ("v", "nv", "r", "done", "term")]
        a, t = vec_generalized_advantage_estimate(gt("gamma"), gt("lmbda"), *cu[:3], done=cu[3], terminated=cu[4])
        torch.testing.assert_close(a.cpu(), gt("loop_adv"), rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(t.cpu(), gt("loop_tgt"), rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(a.cpu(), gt("vec_adv"), rtol=1e-4, atol=1e-4)   # the reference's own bar
        torch.testing.assert_close(t.cpu(), gt("vec_tgt"), rtol=1e-4, atol=1e-4)


def test_gae_unaligned_and_time_dim(cuda_backend):
    from rl_b200.objectives.value import vec_generalized_advantage_estimate

    # a view that is NOT 16-B aligned and whose T is not a multiple of 4 -> scalar path
    v, nv, r, done, term = _gae_inputs((6, 51, 1), 5)
    g, l = 0.97, 0.9
    fa, ft = po.gae_f64(g, l, v, nv, r, done, term)
    pad = lambda x: torch.cat([x.flatten()[:1], x.flatten()]).to(dev())[1:].view(x.shape)
    a, t = vec_generalized_advantage_estimate(g, l, pad(v), pad(nv), pad(r), done=pad(done), terminated=pad(term))
    torch.testing.assert_close(a.cpu().double(), fa, rtol=1e-5, atol=1e-5)
    # time_dim = -1 on [B, T] inputs and time_dim=0 on [T, B, 1]
    v2, nv2, r2, d2, t2 = (x.squeeze(-1).to(dev()) for x in (v, nv, r, done, term))
    a2, tt2 = vec_generalized_advantage_estimate(g, l, v2, nv2, r2, done=d2, terminated=t2, time_dim=-1)
    assert a2.shape == v2.shape
    torch.testing.assert_close(a2.cpu().double(), fa.squeeze(-1), rtol=1e-5, atol=1e-5)
    v3, nv3, r3, d3, t3 = (x.transpose(0, 1).contiguous().to(dev()) for x in (v, nv, r, done, term))
    a3, _ = vec_generalized_advantage_estimate(g, l, v3, nv3, r3, done=d3, terminated=t3, time_dim=0)
    torch.testing.assert_close(a3.cpu().double(), fa.transpose(0, 1), rtol=1e-5, atol=1e-5)


def test_gae_fp64(cuda_backend):
    from rl_b200.objectives.value import vec_generalized_advantage_estimate

    v, nv, r, done, term = _gae_inputs((33, 77, 1), 11, dtype=torch.float64)
    g, l = 0.99, 0.95
    cu = [x.to(dev()) for x in (v, nv, r, done, term)]
    a, t = vec_generalized_advantage_estimate(g, l, *cu[:3], done=cu[3], terminated=cu[4])
    # float64 python loop
    adv = torch.zeros_like(v)
    prev = torch.zeros(33, 1, dtype=torch.float64)
    for s in range(76, -1, -1):
        delta = r[:, s] + g * (~term[:, s]).double() * nv[:, s] - v[:, s]
        prev = delta + g * l * (~done[:, s]).double() * prev
        adv[:, s] = prev
    torch.testing.assert_close(a.cpu(), adv, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(t.cpu(), adv + v, rtol=1e-12, atol=1e-12)


def test_successive_traj_gae(cuda_backend):
    """test/objectives/test_values.py:1775-1857: a rollout with a mid-trajectory `terminated` equals the
    concatenation of the two halves computed separately."""
    from rl_b200.objectives.value import vec_generalized_advantage_estimate

    T, cut = 200, 77
    g = torch.Generator().manual_seed(0)
    v, nv, r = (torch.randn(1, T, 1, generator=g).to(dev()) for _ in range(3))
    done = torch.zeros(1, T, 1, dtype=torch.bool, device=dev())
    done[0, cut - 1] = True
    done[0, -1] = True
    a, t = vec_generalized_advantage_estimate(0.99, 0.95, v, nv, r, done=done, terminated=done.clone())
    a1, t1 = vec_generalized_advantage_estimate(0.99, 0.95, v[:, :cut], nv[:, :cut], r[:, :cut],
                                                done=done[:, :cut], terminated=done[:, :cut])
    a2, t2 = vec_generalized_advantage_estimate(0.99, 0.95, v[:, cut:], nv[:, cut:], r[:, cut:],
                                                done=done[:, cut:], terminated=done[:, cut:])
    torch.testing.assert_close(a, torch.cat([a1, a2], 1), rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(t, torch.cat([t1, t2], 1), rtol=1e-6, atol=1e-6)


# ---------------------------------------------------------------------------------------------------- peer broadcast
@pytest.mark.parametrize("mode", [0, 1])
def test_gather_peer_replication_single_gpu(cuda_backend, mode):
    """rlb_gather / rlb_shard_pack with peer_delta: every destination byte also lands at dst + delta[p].  On one
    GPU the 'peers' are three slices of one buffer (the multi-GPU run, tests/mgpu_check.py, passes the offsets of the
    NVLink symmetric receive buffers instead)."""
    from rl_b200.data.sharded import _PackedLayout

    N, B = 5000, 96
    g = torch.Generator(device=dev()).manual_seed(4)
    leaves = [torch.randint(0, 255, (N, 4, 84, 84), dtype=torch.uint8, device=dev(), generator=g),
              torch.randn(N, 17, device=dev(), generator=g), torch.randint(0, 9, (N, 1), device=dev(), generator=g),
              torch.rand(N, 1, device=dev(), generator=g) < 0.5]
    lay = _PackedLayout(leaves)
    buf = torch.zeros((3, B, lay.row), dtype=torch.uint8, device=dev())
    step = B * lay.row
    idx = torch.randint(0, N, (B,), device=dev(), generator=g)
    cuda_backend.gather(leaves, idx, N, mode=mode, out=lay.leaf_views(buf[0]), peer_delta=[0, step, 2 * step])
    leaf_p = torch.rand(B, device=dev(), generator=g)
    pp = torch.tensor([3.5, 0.25], device=dev())
    cuda_backend.shard_pack(buf[0], lay.meta, idx, leaf_p, pp, 1000, peer_delta=[0, step, 2 * step])
    for c in range(3):
        for leaf, view in zip(leaves, lay.leaf_views(buf[c])):
            assert torch.equal(view, leaf[idx]), c
        gi, p, S, m = lay.meta_views(buf[c])
        assert torch.equal(gi, idx + 1000) and torch.equal(p, leaf_p)
        assert torch.all(S == 3.5) and torch.all(m == 0.25)
    assert torch.equal(buf[0], buf[1]) and torch.equal(buf[0], buf[2])
    w, gidx = cuda_backend.shard_weights(buf[1], lay.meta, 0.4)
    torch.testing.assert_close(w, torch.pow((leaf_p / 3.5) / (0.25 / 3.5), -0.4), rtol=1e-6, atol=0)
    assert torch.equal(gidx, idx + 1000)


def test_shard_flag_exchange_single_gpu(cuda_backend):
    """The split-phase exchange's flags on one GPU: three 'ranks' are three regions [flags | rows] of one buffer.
    rlb_shard_pack(rank=r) release-stores its sequence number into slot r of every region's flags; rlb_shard_weights
    waits until all slots have reached its own call count; a missing rank trips the bounded wait and the status bit."""
    from rl_b200 import ops
    from rl_b200.data.sharded import _PackedLayout

    N, B, W = 2000, 64, 3
    g = torch.Generator(device=dev()).manual_seed(14)
    leaves = [torch.randn(N, 24, device=dev(), generator=g), torch.randint(0, 9, (N, 1), device=dev(), generator=g)]
    lay = _PackedLayout(leaves)
    region = 256 + W * B * lay.row
    region += (-region) % 256
    raw = torch.zeros(W * region, dtype=torch.uint8, device=dev())
    flags = [raw[r * region:r * region + 256].view(torch.int64)[:W] for r in range(W)]
    rows = [raw[r * region + 256:r * region + 256 + W * B * lay.row].view(W * B, lay.row) for r in range(W)]
    ctr = torch.zeros((W, 2), dtype=torch.int64, device=dev())
    status = torch.zeros(1, dtype=torch.int32, device=dev())
    pp = torch.tensor([2.0, 0.5], device=dev())
    for seq in (1, 2):
        idxs = []
        for r in range(W):
            idx = torch.randint(0, N, (B,), device=dev(), generator=g)
            idxs.append(idx)
            mine = rows[r][r * B:(r + 1) * B]
            peers = [(q - r) * region for q in range(W)]
            cuda_backend.gather(leaves, idx, N, out=lay.leaf_views(mine), peer_delta=peers)
            cuda_backend.shard_pack(mine, lay.meta, idx, torch.rand(B, device=dev(), generator=g) + 0.5, pp, r * N,
                                    peer_delta=peers, flags=flags[r], seq_counter=ctr[r, 0:1], rank=r)
            if r == W - 2 and seq == 2:
                # rank W-1 has not published draw 2 yet: a wait on region 0 must time out and say so
                w, gi = cuda_backend.shard_weights(rows[0], lay.meta, 0.4, flags=flags[0], wait_counter=ctr[0, 1:2],
                                                   n_ranks=W, timeout_s=0.05, status=status)
                torch.cuda.synchronize()
                assert int(status.item()) & ops.STATUS_EXCHANGE_TIMEOUT
                status.zero_()
                ctr[0, 1] -= 1   # that wait did not pair with a complete draw
        for r in range(W):
            assert flags[r].tolist() == [seq] * W
            w, gi = cuda_backend.shard_weights(rows[r], lay.meta, 0.4, flags=flags[r], wait_counter=ctr[r, 1:2],
                                               n_ranks=W, timeout_s=5.0, status=status)
            assert torch.equal(gi, torch.cat([idxs[q] + q * N for q in range(W)]))
            for leaf, view in zip(leaves, lay.leaf_views(rows[r])):
                assert torch.equal(view, torch.cat([leaf[idxs[q]] for q in range(W)]))
        assert int(status.item()) == 0
    assert ctr[:, 0].tolist() == [2] * W and ctr[:, 1].tolist() == [2] * W


def test_update_priority_chunked_under_capture(cuda_backend):
    """More than 1024 priorities inside a CUDA graph: applied as <=1024-item chunks, same heap as the eager call."""
    from rl_b200.data import PrioritizedSampler

    N, n = 100_000, 3000
    g = torch.Generator(device=dev()).manual_seed(8)
    idx = torch.randint(0, N, (n,), device=dev(), generator=g)
    idx[::7] = idx[0]  # duplicates across chunk boundaries: the last one must win
    pr = torch.rand(n, device=dev(), generator=g) + 0.1
    a, b = PrioritizedSampler(N, 0.6, 0.4, device=dev()), PrioritizedSampler(N, 0.6, 0.4, device=dev())
    for s in (a, b):
        s.update_priority(torch.arange(N, device=dev()), torch.ones(N, device=dev()))
    a.update_priority(idx, pr)  # eager: stamp-dedupe general path
    s_ = torch.cuda.Stream(dev())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s_):
        b.update_priority(idx[:8], pr[:8])  # lazy init outside capture
        b.update_priority(idx[:8], torch.ones(8, device=dev()))
        s_.synchronize()
        with torch.cuda.graph(graph, stream=s_):
            b.update_priority(idx, pr)
        graph.replay()
        s_.synchronize()
    assert torch.equal(a._sum_tree.values[1:], b._sum_tree.values[1:])
    assert torch.equal(a._min_tree.values[1:], b._min_tree.values[1:])


# ---------------------------------------------------------------------------------------------------- TD(lambda)
@pytest.mark.parametrize("shape", [(1, 1, 1), (3, 200, 1), (9, 131, 1), (4096, 128, 1), (5, 33, 3), (2, 1000, 1),
                                   (3, 4100, 1), (300, 500, 1)])
@pytest.mark.parametrize("gamma,lmbda", [(0.99, 0.95), (0.97, 1.0), (0.9, 0.0)])
def test_td_lambda_matches_f64_oracle(cuda_backend, shape, gamma, lmbda):
    from rl_b200.objectives.value import td1_return_estimate, vec_td_lambda_advantage_estimate, vec_td_lambda_return_estimate

    v, nv, r, done, term = _gae_inputs(shape, sum(shape) + 1)
    f64 = po.td_lambda(gamma, lmbda, nv, r, done, term, f64=True)
    loop = po.td_lambda(gamma, lmbda, nv, r, done, term)           # bit-equal to the reference loop
    cu = [x.to(dev()) for x in (v, nv, r, done, term)]
    got = vec_td_lambda_return_estimate(gamma, lmbda, cu[1], cu[2], cu[3], cu[4])
    torch.testing.assert_close(got.cpu().double(), f64, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(got.cpu(), loop, rtol=1e-5, atol=1e-5)
    adv = vec_td_lambda_advantage_estimate(gamma, lmbda, cu[0], cu[1], cu[2], cu[3], cu[4])
    assert torch.equal(adv, got - cu[0])
    if lmbda == 1.0:
        assert torch.equal(td1_return_estimate(gamma, cu[1], cu[2], cu[3], cu[4]), got)


def test_td_lambda_golden(cuda_backend):
    from rl_b200.objectives.value import vec_td_lambda_return_estimate

    z = np.load(GOLD / "td_lambda_golden.npz")
    for k in sorted({n.split("/")[0] for n in z.files}):
        gt = lambda n: torch.from_numpy(z[f"{k}/{n}"])
        got = vec_td_lambda_return_estimate(float(gt("gamma")), float(gt("lmbda")), gt("nv").to(dev()), gt("r").to(dev()),
                                            gt("done").to(dev()), gt("term").to(dev()))
        torch.testing.assert_close(got.cpu(), gt("loop"), rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(got.cpu(), gt("vec"), rtol=1e-4, atol=1e-4)   # the reference's own bar


@pytest.mark.parametrize("shape", [(16, 80, 1), (3, 1000, 1), (5, 33, 3), (2, 3, 7, 1), (300, 5, 1), (1, 1, 1),
                                   (2, 2300, 1)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_affine_scan_matches_oracle(cuda_backend, shape, dtype):
    """rlb_affine_scan against the C recurrence: fp64 to 1e-12, fp32 within the 1e-5 bar of the fp64 recurrence."""
    g = torch.Generator().manual_seed(sum(shape))
    d = torch.randn(*shape, generator=g, dtype=dtype)
    c = torch.rand(*shape, generator=g, dtype=dtype) * (torch.rand(*shape, generator=g) > 0.05)
    rows, T, F = int(np.prod(shape[:-2])), shape[-2], shape[-1]
    got = cuda_backend.affine_scan(d.to(dev()), c.to(dev()), rows, T, F).cpu()
    ref64 = po.affine_scan(d.double(), c.double())
    if dtype == torch.float64:
        torch.testing.assert_close(got, ref64, rtol=1e-12, atol=1e-12)
    else:
        torch.testing.assert_close(got.double(), ref64, rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(got, po.affine_scan(d, c), rtol=1e-5, atol=1e-5)


def test_vtrace_and_per_step_gae_golden(cuda_backend):
    """V-trace and GAE with per-step gamma / lmbda tensors on the device against the reference's outputs
    (tests/golden/vtrace_golden.npz) and the oracle; time_dim variants too."""
    from rl_b200.objectives.value import reward2go, vec_generalized_advantage_estimate, vtrace_advantage_estimate

    z = np.load(GOLD / "vtrace_golden.npz")
    for k in sorted({n.split("/")[0] for n in z.files}):
        gt = lambda n: torch.from_numpy(z[f"{k}/{n}"])
        cu = lambda n: gt(n).to(dev())
        args = (float(gt("gamma")), cu("log_pi"), cu("log_mu"), cu("v"), cu("nv"), cu("r"), cu("done"), cu("term"),
                float(gt("rho_thresh")), float(gt("c_thresh")))
        adv, vs = vtrace_advantage_estimate(*args)
        torch.testing.assert_close(vs.cpu(), gt("vs"), rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(adv.cpu(), gt("adv"), rtol=1e-5, atol=1e-5)
        ga, gtg = vec_generalized_advantage_estimate(cu("gammas"), cu("lmbdas"), cu("v"), cu("nv"), cu("r"), cu("done"),
                                                     cu("term"))
        oa, ot = po.gae_per_step(gt("gammas").double(), gt("lmbdas").double(), gt("v").double(), gt("nv").double(),
                                 gt("r").double(), gt("done"), gt("term"))
        torch.testing.assert_close(ga.cpu().double(), oa, rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(gtg.cpu().double(), ot, rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(ga.cpu(), gt("gae_adv"), rtol=1e-4, atol=1e-4)     # the reference's own bar
        torch.testing.assert_close(reward2go(cu("r"), cu("done"), float(gt("gamma"))).cpu(), gt("r2g"), rtol=1e-5,
                                   atol=1e-5)
        if gt("v").ndim == 3 and gt("v").shape[-1] == 1:
            sq = lambda t: t.squeeze(-1) if isinstance(t, torch.Tensor) else t
            adv_t, vs_t = vtrace_advantage_estimate(*[sq(a) for a in args], time_dim=-1)
            # [B, T] with time last runs as one [T, F=B] problem (serial column kernel), not B warp scans
            torch.testing.assert_close(adv_t, adv.squeeze(-1), rtol=1e-5, atol=1e-5)
            torch.testing.assert_close(vs_t, vs.squeeze(-1), rtol=1e-5, atol=1e-5)


# ---------------------------------------------------------------------------------------------------- trajectory slices
@pytest.mark.parametrize("L", [1, 2, 7, 2048, 2049, 5000, 100_000, 1_000_003])
@pytest.mark.parametrize("by_id", [False, True])
def test_traj_table_matches_oracle(cuda_backend, L, by_id):
    """rlb_traj_table (tile scan with last-CTA prefix, emit, compaction) against the restated reference
    (_find_start_stop_traj / _end_to_start_stop): every table row and both counters, bit-exact, over densities from
    "no end at all" to "every slot ends", partial and full rings, with and without the cursor rule and the length filter."""
    from oracle import slice_oracle as so

    rng = np.random.default_rng(L + by_id)
    table = torch.empty((3, L), dtype=torch.int64, device=dev())
    counts = torch.zeros(2, dtype=torch.int64, device=dev())
    ws = cuda_backend.traj_workspace(L, dev())
    for density in [0.0, 0.002, 0.05, 0.6, 1.0]:
        for at_capacity in (False, True):
            for cursor in (-1, int(rng.integers(0, L))):
                if by_id:
                    sig = np.cumsum(rng.random(L) < density).astype(np.int64) + 5
                    kw = dict(trajectory=sig)
                else:
                    sig = rng.random(L) < density
                    kw = dict(end=sig)
                start, stop, length = so.traj_table(at_capacity=at_capacity, cursor=None if cursor < 0 else cursor, **kw)
                for min_len, keep in ((0, False), (4, False), (4, True), (L + 1, True)):
                    cuda_backend.traj_table(torch.from_numpy(sig).to(dev()), by_id, L, at_capacity, cursor, min_len, keep,
                                            table, counts, ws)
                    long_enough = length >= min_len
                    assert counts.tolist() == [len(start), int(long_enough.sum())]
                    sel = long_enough if keep else slice(None)
                    want = np.stack([start[sel], stop[sel], length[sel]])
                    np.testing.assert_array_equal(table[:, :want.shape[1]].cpu().numpy(), want)
    assert int(ws.view(torch.int32)[:2].abs().sum()) == 0        # both tickets are back at zero


def test_slice_index_golden_and_large(cuda_backend):
    """rlb_slice_index with the draws the reference made (tests/golden/slice_golden.npz, produced by the unmodified
    SliceSampler): index / truncated / mask bit-equal; then BASELINE-scale shapes against the oracle."""
    from oracle import slice_oracle as so

    z = np.load(GOLD / "slice_golden.npz")
    for k in sorted({n.split("/")[0] for n in z.files}):
        gt = lambda n: z[f"{k}/{n}"]
        length, max_size, cursor, seq, num_slices, strict, pad, by_id = (int(x) for x in gt("meta"))
        sig = torch.from_numpy(gt("signal")[:length]).to(dev())
        table = torch.empty((3, max_size), dtype=torch.int64, device=dev())
        counts = torch.zeros(2, dtype=torch.int64, device=dev())
        cuda_backend.traj_table(sig, bool(by_id), length, length == max_size, cursor, seq, bool(strict), table, counts,
                                cuda_backend.traj_workspace(max_size, dev()))
        n_all, n_long = counts.tolist()
        assert n_all == gt("table").shape[1]
        if not strict:
            np.testing.assert_array_equal(table[:, :n_all].cpu().numpy(), gt("table"))
        n_traj, variable = (n_long, False) if strict else (n_all, n_long < n_all)
        traj, u = torch.from_numpy(gt("traj_draw")).to(dev()), torch.from_numpy(gt("u")).to(dev())
        args = (table[0], table[2], n_traj, traj, u, seq, max_size)
        if variable and not pad:
            sq = cuda_backend.slice_index(*args, variable=True, want_index=False)[3]
            ends_at = sq.cumsum(0)
            index, trunc, mask, _ = cuda_backend.slice_index(*args, variable=True, out_offset=ends_at - sq,
                                                             total=int(ends_at[-1]))
        else:
            index, trunc, mask, _ = cuda_backend.slice_index(*args, variable=variable, pad_output=bool(pad))
        np.testing.assert_array_equal(index.cpu().numpy(), gt("index"))
        np.testing.assert_array_equal(trunc.cpu().numpy().reshape(-1), gt("truncated"))
        if pad:
            np.testing.assert_array_equal(mask.cpu().numpy(), gt("mask"))
    # 10M-slot ring, 4096 slices of 64 steps
    L, S, T = 10_000_000, 4096, 64
    rng = np.random.default_rng(0)
    end = rng.random(L) < 1 / 300
    start, stop, length = so.traj_table(end=end, at_capacity=True, cursor=None)
    ks, _, kl = so.valid_trajectories(start, stop, length, T, True)
    table = torch.empty((3, L), dtype=torch.int64, device=dev())
    counts = torch.zeros(2, dtype=torch.int64, device=dev())
    cuda_backend.traj_table(torch.from_numpy(end).to(dev()), False, L, True, -1, T, True, table, counts,
                            cuda_backend.traj_workspace(L, dev()))
    assert counts.tolist() == [len(start), len(ks)]
    np.testing.assert_array_equal(table[0, :len(ks)].cpu().numpy(), ks)
    g = torch.Generator(device=dev()).manual_seed(0)
    traj = torch.randint(len(ks), (S,), device=dev(), generator=g)
    u = torch.rand(S, device=dev(), generator=g)
    index, trunc, _, _ = cuda_backend.slice_index(table[0], table[2], len(ks), traj, u, T, L)
    oi, otr, _, _ = so.slice_index(ks, kl, seq_length=T, num_slices=S, storage_length=L, traj_draw=traj.cpu().numpy(),
                                   u=u.cpu().numpy())
    np.testing.assert_array_equal(index.cpu().numpy(), oi)
    np.testing.assert_array_equal(trunc.cpu().numpy().reshape(-1), otr)
    # size-independent property: every slice is S consecutive ring slots inside ONE trajectory
    ix = index.view(S, T).cpu().numpy()
    assert ((ix[:, 1:] - ix[:, :-1]) % L == 1).all()
    assert not end[ix[:, :-1]].any()


def test_prioritized_slice_golden(cuda_backend):
    """PrioritizedSliceSampler's draw on the device -- masked copy of the leaves (rlb_slice_mask_starts), rebuild, the
    ordinary PER sample -- with the leaves and uniform draws of the unmodified reference (tests/golden/pslice_golden.npz):
    the masked heap is, node for node, the reference's zero-and-recompute tree, and the sampled starts are its starts."""
    from oracle import slice_oracle as so
    from rl_b200.data import PrioritizedSliceSampler

    z = np.load(GOLD / "pslice_golden.npz")
    for k in sorted({n.split("/")[0] for n in z.files}):
        gt = lambda n: z[f"{k}/{n}"]
        L, filled, S, T = (int(x) for x in gt("meta"))
        smp = PrioritizedSliceSampler(L, 0.7, 0.9, num_slices=S, end_key=("next", "done"), device=dev())
        smp._sum_tree.load_leaves(torch.from_numpy(gt("sum_leaves")).to(dev()))
        smp._min_tree.load_leaves(torch.from_numpy(gt("min_leaves")).to(dev()))
        cap = smp._sum_tree.capacity
        done = torch.from_numpy(gt("done")[:filled]).to(dev())
        table = torch.empty((3, L), dtype=torch.int64, device=dev())
        counts = torch.zeros(2, dtype=torch.int64, device=dev())
        cuda_backend.traj_table(done, False, filled, filled == L, -1, T, False, table, counts,
                                cuda_backend.traj_workspace(L, dev()))
        n_all = int(counts[0])
        masked = smp._sum_tree.values.clone()
        cuda_backend.slice_mask_starts(masked, cap, table[1], table[2], n_all, T, filled)
        cuda_backend.tree_rebuild(masked, cap, False)
        start, stop, length = so.traj_table(end=gt("done")[:filled], at_capacity=filled == L, cursor=None)
        ot = po.OracleTree(L, False)
        leaves = gt("sum_leaves").copy()
        leaves[so.invalid_starts(stop, length, T, filled)] = 0
        ot.load_leaves(leaves)
        np.testing.assert_array_equal(masked.cpu().numpy()[1:], ot.values()[1:])
        for d in range(gt("u").shape[0]):
            u = torch.from_numpy(gt("u")[d]).to(dev())
            starts, w = cuda_backend.per_sample(masked, smp._min_tree.values, L, cap, filled, u, 0.9, True)
            np.testing.assert_array_equal(starts.cpu().numpy(), gt("index")[d].reshape(S, T)[:, 0])
            np.testing.assert_allclose(w.cpu().numpy(), gt("weight")[d].reshape(S, T)[:, 0], rtol=2e-6)


# ---------------------------------------------------------------------------------------------------- edge cases
def test_empty_and_degenerate_inputs(cuda_backend):
    """Empty batches / rows / time axes are no-ops that return correctly shaped empties; arguments are validated."""
    from rl_b200.data import PrioritizedSampler
    from rl_b200.data.segment_tree import SumSegmentTreeFp32
    from rl_b200.objectives.value import vec_generalized_advantage_estimate, vec_td_lambda_return_estimate

    src = [torch.randn(10, 3, device=dev()), torch.zeros(10, 0, device=dev())]          # a zero-width leaf too
    out = cuda_backend.gather(src, torch.empty(0, dtype=torch.long, device=dev()), 10)
    assert out[0].shape == (0, 3) and out[1].shape == (0, 0)
    out = cuda_backend.gather(src, torch.tensor([9, 0], device=dev()), 10)
    assert torch.equal(out[0], src[0][[9, 0]]) and out[1].shape == (2, 0)
    with pytest.raises(RuntimeError, match="empty storage"):
        cuda_backend.gather(src, torch.tensor([0], device=dev()), 0)
    t = SumSegmentTreeFp32(8, dev())
    t[torch.empty(0, dtype=torch.long, device=dev())] = torch.empty(0, device=dev())    # n == 0
    assert t.query(0, 8) == 0.0
    assert t.scan_lower_bound(torch.empty(0, device=dev())).shape == (0,)
    smp = PrioritizedSampler(8, 0.6, 0.4, device=dev())
    smp.update_priority(torch.tensor([-1, -1], device=dev()), torch.tensor([3.0, 4.0], device=dev()))  # all skipped
    assert smp._sum_tree.query(0, 8) == 0.0 and float(smp._max_priority_buf) == float("-inf")
    e = torch.empty(0, 5, 1, device=dev())
    a, tg = vec_generalized_advantage_estimate(0.9, 0.9, e, e, e, done=e.bool())
    assert a.shape == (0, 5, 1) and tg.shape == (0, 5, 1)
    e = torch.empty(3, 0, 1, device=dev())
    assert vec_td_lambda_return_estimate(0.9, 0.9, e, e, e.bool()).shape == (3, 0, 1)
    with pytest.raises(RuntimeError, match="expected a CUDA tensor|no CPU path"):
        cuda_backend.gather([torch.randn(4, 2)], torch.tensor([0]), 4)
    # single-element tree / batch, capacity rule for a power-of-two size
    one = SumSegmentTreeFp32(1, dev())
    one[torch.tensor([0], device=dev())] = torch.tensor([2.5], device=dev())
    assert one.capacity == 2 and one.query(0, 1) == 2.5 and one.scan_lower_bound(1.0) == 0


# ------------------------------------------------------------------------- the reference's OWN CUDA path, end to end
def test_sampler_matches_reference_cuda_path_without_leaf_injection(cuda_backend, ref_cuda):
    """The closing leg of the parity loop: this repo's PrioritizedSampler against the reference's CUDA branch --
    the UNMODIFIED csrc/cuda_segment_tree.cu (oracle/_ref/cuda/_torchrl.so: CudaSum/MinSegmentTreeFp32) driven by the
    glue of samplers.py:895-956 / :1054-1078 restated line by line, with torch.pow / torch.rand on the device.  Nothing
    is injected: both sides start from raw priorities, apply (p + eps) ** alpha themselves (torch.pow there, the fused
    kernel here), and must produce the same leaves, the same query results and the same sampled indices and weights
    through several rounds of sample -> write-back with duplicate indices (shape of test/rb/test_prioritized.py:103-140)."""
    from rl_b200.data import PrioritizedSampler

    ext = ref_cuda
    N, n_filled, B, alpha, beta, eps = 50_000, 41_234, 256, 0.6, 0.4, 1e-8
    d = dev()
    rs, rm = ext.CudaSumSegmentTreeFp32(N, d), ext.CudaMinSegmentTreeFp32(N, d)
    ours = PrioritizedSampler(N, alpha, beta, eps=eps, device=d, semantics="cuda")

    class _St:  # what the sampler needs from a storage (benchmarks/test_replaybuffer_benchmark.py:95-105)
        ndim, shape, device = 1, (n_filled,), d

        def __len__(self):
            return n_filled

    st = _St()

    def ref_update(index, priority):           # samplers.py:1076-1078 on the CUDA branch
        leaf = torch.pow(priority + eps, alpha)
        rs[index] = leaf
        rm[index] = leaf

    def ref_sample(gen):                       # samplers.py:899-953 on the CUDA branch
        left = torch.zeros((), dtype=torch.long, device=d)
        right = torch.full((), n_filled, dtype=torch.long, device=d)
        p_sum, p_min = rs.query(left, right), rm.query(left, right)
        mass = torch.rand(B, device=d, generator=gen) * p_sum
        index = rs.scan_lower_bound(mass)
        index.clamp_max_(n_filled - 1)
        # NB: p_sum / p_min come back as PYTHON FLOATS here -- pybind accepts a 0-d integer tensor for the (int64, int64)
        # overload of query through __index__ -- so this division is ATen's CUDA "multiply by the reciprocal of a CPU
        # scalar"; semantics="cuda" reproduces exactly that
        weight = torch.pow(rs[index] / p_min, -beta)
        return index, weight, p_sum, p_min

    g = torch.Generator(device=d).manual_seed(3)
    all_idx = torch.arange(n_filled, device=d)
    p0 = torch.rand(n_filled, device=d, generator=g) * 3
    p0[::97] = 0.0                                        # eps keeps zero priorities positive
    ref_update(all_idx, p0)
    ours.update_priority(all_idx, p0)
    g_ref, g_our = torch.Generator(device=d).manual_seed(9), torch.Generator(device=d).manual_seed(9)
    ours._rng = g_our
    for rnd in range(6):
        assert torch.equal(rs[all_idx], ours._sum_tree[all_idx]), rnd           # leaves, bit for bit
        assert torch.equal(rm[all_idx], ours._min_tree[all_idx]), rnd
        lq = torch.randint(0, n_filled // 2, (64,), device=d, generator=g)
        rq = lq + torch.randint(1, n_filled // 2, (64,), device=d, generator=g)
        assert torch.equal(rs.query(lq, rq), ours._sum_tree.query(lq, rq, root_fast_path=False))  # internal nodes
        assert torch.equal(rm.query(lq, rq), ours._min_tree.query(lq, rq, root_fast_path=False))
        ri, rw, p_sum, p_min = ref_sample(g_ref)
        oi, info = ours.sample(st, B)
        assert torch.equal(ri, oi), rnd
        ow = info["priority_weight"]
        if not torch.equal(rw, ow):
            bad = (rw != ow).nonzero().flatten()[:5]
            op = ours._min_tree.query(torch.zeros(1, dtype=torch.long, device=d),
                                      torch.full((1,), n_filled, dtype=torch.long, device=d), root_fast_path=False)
            raise AssertionError(f"round {rnd}: {int((rw != ow).sum())} of {B} weights differ; ref p_min={float(p_min).hex()} "
                                 f"ours p_min={op.item().hex()}; first: " + "; ".join(
                                     f"i={int(i)} leaf={rs[ri[i:i + 1]].item().hex()} ref={rw[i].item().hex()} "
                                     f"ours={ow[i].item().hex()} torch.pow(leaf/p_min)={torch.pow(rs[ri[i:i + 1]] / op, -beta).item().hex()}"
                                     for i in bad))
        # write-back with duplicates (last writer wins on both sides) and fresh priorities
        wi = torch.cat([oi, oi[:32], oi[5:9]])
        wp = torch.rand(wi.numel(), device=d, generator=g) * 2
        ref_update(wi, wp)
        ours.update_priority(wi, wp)
    torch.cuda.synchronize()


@pytest.mark.parametrize("span", [(-1, 0), (0, -1), (-1, -1), (3, 0), (0, 5), (2, 7), (-1, 4)])
@pytest.mark.parametrize("pad", [False, True])
def test_slice_index_span_matches_oracle(cuda_backend, span, pad):
    """SliceSampler(span=...) in rlb_slice_index (samplers.py:2071-2118): the slice may start before its trajectory
    (left) or run past its end (right); the part outside is cut off.  Index / truncated / mask / lengths bit-equal to the
    restatement (itself pinned to the unmodified reference in tests/test_host_logic.py) for the same draws."""
    from oracle import slice_oracle as so

    L, S, T = 200_000, 512, 16
    rng = np.random.default_rng(100 + 7 * span[0] + span[1])
    end = np.zeros(L, dtype=bool)
    end[np.cumsum(rng.integers(8, 60, L // 30))[:-1] % L] = True      # trajectories of 8..59 steps: longer than any span
    start, stop, length = so.traj_table(end=end, at_capacity=True, cursor=None)
    table = torch.empty((3, L), dtype=torch.int64, device=dev())
    counts = torch.zeros(2, dtype=torch.int64, device=dev())
    cuda_backend.traj_table(torch.from_numpy(end).to(dev()), False, L, True, -1, T, False, table, counts,
                            cuda_backend.traj_workspace(L, dev()))
    n_all = int(counts[0])
    assert n_all == len(start)
    g = torch.Generator(device=dev()).manual_seed(1)
    traj = torch.randint(n_all, (S,), device=dev(), generator=g)
    u = torch.rand(S, device=dev(), generator=g)
    args = (table[0], table[2], n_all, traj, u, T, L)
    oi, otr, omask, oseq = so.slice_index(start, length, seq_length=T, num_slices=S, storage_length=L,
                                          traj_draw=traj.cpu().numpy(), u=u.cpu().numpy(), strict_length=False,
                                          pad_output=pad, span=span, force_variable=True)
    if pad:
        index, trunc, mask, sq = cuda_backend.slice_index(*args, variable=True, pad_output=True, span=span)
        np.testing.assert_array_equal(mask.cpu().numpy(), omask)
    else:
        sq = cuda_backend.slice_index(*args, variable=True, want_index=False, span=span)[3]
        ends_at = sq.cumsum(0)
        index, trunc, mask, _ = cuda_backend.slice_index(*args, variable=True, out_offset=ends_at - sq,
                                                         total=int(ends_at[-1]), span=span)
    np.testing.assert_array_equal(sq.cpu().numpy(), oseq)
    np.testing.assert_array_equal(index.cpu().numpy(), oi)
    np.testing.assert_array_equal(trunc.cpu().numpy().reshape(-1), otr)
    assert (oseq < T).any() and (oseq >= 0).all()                                # some slices were cut


@pytest.mark.parametrize("n", [1025, 4096, 8192])
def test_update_rounds_in_one_launch(cuda_backend, n):
    """Batches above 1024 items: rounds of 1024 inside ONE cluster launch (no epoch stamp, capturable).  A 6.25M-slot
    shard (BASELINE configs[4]: capacity 2^23), heavy duplication inside and ACROSS rounds -- the last writer of a leaf
    must win -- against the oracle; then the same call captured in a CUDA graph and replayed on fresh priorities."""
    from rl_b200.data import PrioritizedSampler

    N = 6_250_000
    rng = np.random.default_rng(n)
    smp = PrioritizedSampler(N, 0.6, 0.4, device=dev())
    base = rng.integers(0, N, 2000)
    idx = np.concatenate([rng.integers(0, N, n - n // 4), rng.choice(base, n // 4)]).astype(np.int64)
    rng.shuffle(idx)
    idx[-5:] = idx[:5]                                 # duplicates that span the first and the last round
    pr = (rng.random(n, dtype=np.float32) * 4).astype(np.float32)
    ti, tp = torch.from_numpy(idx).to(dev()), torch.from_numpy(pr).to(dev())
    smp.update_priority(ti, tp)
    leaves = torch.pow(tp + 1e-8, 0.6)                 # the fused pow is torch's (test_fused_pow_is_torch_pow)
    os_, om = po.OracleTree(N, False), po.OracleTree(N, True)
    os_[idx] = leaves.cpu().numpy()
    om[idx] = leaves.cpu().numpy()
    np.testing.assert_array_equal(smp._sum_tree.values.cpu().numpy()[1:], os_.values()[1:])
    np.testing.assert_array_equal(smp._min_tree.values.cpu().numpy()[1:], om.values()[1:])
    assert smp._max_priority[0].item() == pr.max()
    # captured: one graph node per call, replay-safe
    tp2 = torch.empty_like(tp)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            smp.update_priority(ti, tp2)
    for rep in range(2):
        pr2 = (rng.random(n, dtype=np.float32) * 4).astype(np.float32)
        tp2.copy_(torch.from_numpy(pr2))
        g.replay()
        torch.cuda.synchronize()
        l2 = torch.pow(tp2 + 1e-8, 0.6).cpu().numpy()
        os_[idx] = l2
        om[idx] = l2
        np.testing.assert_array_equal(smp._sum_tree.values.cpu().numpy()[1:], os_.values()[1:])
        np.testing.assert_array_equal(smp._min_tree.values.cpu().numpy()[1:], om.values()[1:])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["one-range", "two-ranges", "sharded", "fp64-plain"])
def test_update_split_over_clusters_skewed(cuda_backend, shape):
    """The multi-cluster split of large batches with lopsided leaf ranges: every item in ONE cluster's range (the others
    get empty shares, that one runs several rounds), two far-apart ranges, global indices of a sharded buffer (entries
    outside the shard are skipped), and the plain fp64 tree update -- all bit-exact against the oracle."""
    rng = np.random.default_rng(7)
    n = 4096
    if shape == "fp64-plain":
        from rl_b200.data import SumSegmentTreeFp64

        N = 3_000_000
        tree = SumSegmentTreeFp64(N, dev())
        idx = rng.integers(0, N, n).astype(np.int64)
        idx[100:200] = idx[:100]
        val = rng.random(n)
        tree[torch.from_numpy(idx).to(dev())] = torch.from_numpy(val).to(dev())
        cap = tree.capacity
        want = np.zeros(2 * cap)
        want[cap + idx] = val                                         # (numpy fancy assignment: the last duplicate wins)
        level = want[cap:]
        while len(level) > 1:                                         # every node = left child + right child, in fp64
            level = level[0::2] + level[1::2]
            want[len(level):2 * len(level)] = level
        np.testing.assert_array_equal(tree.values.cpu().numpy()[1:], want[1:])
        return
    from rl_b200.data import PrioritizedSampler

    N = 6_250_000
    smp = PrioritizedSampler(N, 0.6, 0.4, device=dev())
    base, limit = 0, N
    if shape == "one-range":
        idx = rng.integers(5_000_000, 5_000_000 + 3000, n)          # heavy duplication inside 1/16 of the leaves
    elif shape == "two-ranges":
        idx = np.concatenate([rng.integers(0, 40_000, n // 2), rng.integers(6_000_000, N, n // 2)])
        rng.shuffle(idx)
    else:
        base, limit = 3 * N, N                                        # this shard owns [3N, 4N) of a 8N global buffer
        idx = rng.integers(0, 8 * N, n)
        idx[: n // 2] = rng.integers(3 * N, 4 * N, n // 2)
        rng.shuffle(idx)
    idx = idx.astype(np.int64)
    pr = (rng.random(n, dtype=np.float32) * 4).astype(np.float32)
    ti, tp = torch.from_numpy(idx).to(dev()), torch.from_numpy(pr).to(dev())
    for rep in range(2):                                              # (the ticket must be back at zero for the second call)
        smp.update_priority(ti, tp, index_base=base, index_limit=limit) if shape == "sharded" else smp.update_priority(ti, tp)
    torch.cuda.synchronize()
    mine = (idx >= base) & (idx < base + limit)
    leaves = torch.pow(tp + 1e-8, 0.6).cpu().numpy()
    os_, om = po.OracleTree(N, False), po.OracleTree(N, True)
    os_[idx[mine] - base] = leaves[mine]
    om[idx[mine] - base] = leaves[mine]
    np.testing.assert_array_equal(smp._sum_tree.values.cpu().numpy()[1:], os_.values()[1:])
    np.testing.assert_array_equal(smp._min_tree.values.cpu().numpy()[1:], om.values()[1:])
    assert smp._max_priority[0].item() == pr[mine].max()
