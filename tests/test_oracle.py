"""Pins the CPU oracle: reference KATs, the compiled reference trees, the imported reference GAE.

Runs on CPU (`-m "not gpu"`).  If these fail the oracle is wrong and no parity claim stands.
"""
import numpy as np
import pytest
import torch

from oracle import per_oracle as po
from oracle import gae_torch


# --------------------------------------------------------------------------- segment tree KATs
def _kat_trees(factory):
    # test/rb/test_prioritized.py:113-140 (test_cuda_segment_tree_parity)
    s, m = factory(16, False), factory(16, True)
    idx = np.array([0, 3, 4, 7, 12, 15], dtype=np.int64)
    val = np.array([1, 2, 4, 8, 16, 32], dtype=np.float32)
    s[idx] = val
    m[idx] = val
    return s, m


def test_tree_kat_oracle():
    s, m = _kat_trees(po.OracleTree)
    assert s.capacity == 32  # strictly-greater power of two, csrc/segment_tree.h:46
    l = np.array([0, 3, 4, 7]); r = np.array([16, 8, 13, 16])
    np.testing.assert_array_equal(s.query(l, r), [63, 14, 28, 56])
    np.testing.assert_array_equal(m.query(l, r), [1, 2, 4, 8])
    np.testing.assert_array_equal(s.query(l, r, walk=True), [63, 14, 28, 56])
    np.testing.assert_array_equal(
        s.scan_lower_bound(np.array([0.5, 1.0, 2.9, 7.1, 30.0], dtype=np.float32)), [0, 0, 3, 7, 12])
    # value > root -> size (segment_tree.h:250-252)
    assert s.scan_lower_bound(np.float32(64.0)) == 16


def test_tree_kat_reference(ref_cpu):
    s, m = _kat_trees(lambda n, is_min: (ref_cpu.MinSegmentTreeFp32 if is_min else ref_cpu.SumSegmentTreeFp32)(n))
    assert s.capacity == 32
    l = np.array([0, 3, 4, 7]); r = np.array([16, 8, 13, 16])
    np.testing.assert_array_equal(s.query(l, r), [63, 14, 28, 56])
    np.testing.assert_array_equal(m.query(l, r), [1, 2, 4, 8])
    np.testing.assert_array_equal(
        s.scan_lower_bound(np.array([0.5, 1.0, 2.9, 7.1, 30.0], dtype=np.float32)), [0, 0, 3, 7, 12])


def test_writer_kat():
    # test/rb/test_rb_core.py:598-600: 50 default-priority items in a 100-slot tree
    smp = po.OraclePrioritizedSampler(100, alpha=0.7, beta=0.5)
    smp.mark_update(torch.arange(50))
    assert smp._sum_tree.query(0, 10) == 10
    assert smp._sum_tree.query(0, 50) == 50
    assert smp._sum_tree.query(0, 70) == 50


@pytest.mark.parametrize("size", [1, 2, 7, 16, 100, 1000, 4097, 100_000])
def test_tree_matches_reference_random(ref_cpu, size):
    rng = np.random.default_rng(size)
    os_, om = po.OracleTree(size, False), po.OracleTree(size, True)
    rs, rm = ref_cpu.SumSegmentTreeFp32(size), ref_cpu.MinSegmentTreeFp32(size)
    assert os_.capacity == rs.capacity
    for _ in range(4):
        n = int(rng.integers(1, 4 * size + 2))
        idx = rng.integers(0, size, n).astype(np.int64)          # duplicates on purpose
        val = rng.random(n, dtype=np.float32) * 3 + 1e-3
        for t in (os_, om, rs, rm):
            t[idx] = val
        l = rng.integers(0, size, 64).astype(np.int64)
        r = np.minimum(l + rng.integers(1, size + 1, 64), size).astype(np.int64)
        np.testing.assert_array_equal(os_.query(l, r), rs.query(l, r))
        np.testing.assert_array_equal(om.query(l, r), rm.query(l, r))
        assert os_.query(0, size) == rs.query(0, size)
        mass = (rng.random(257, dtype=np.float32) * np.float32(os_.query(0, size)) * np.float32(1.05))
        np.testing.assert_array_equal(os_.scan_lower_bound(mass), rs.scan_lower_bound(mass))
        probe = rng.integers(0, size, 33).astype(np.int64)
        np.testing.assert_array_equal(os_[probe], rs[probe])
    # scalar-value overload
    idx = rng.integers(0, size, 9).astype(np.int64)
    os_[idx] = 0.25; rs[idx] = 0.25
    assert os_.query(0, size) == rs.query(0, size)
    # whole heap equals leaves reloaded bottom-up (LoadValues, segment_tree.h:200-207)
    t2 = po.OracleTree(size, False); t2.load_leaves(os_.dump_leaves())
    np.testing.assert_array_equal(t2.values()[1:], os_.values()[1:])


def test_sampler_glue_matches_reference_tree(ref_cpu):
    """OraclePrioritizedSampler over C trees == the same glue over the compiled reference trees."""
    N, B = 5000, 512
    a = po.OraclePrioritizedSampler(N, alpha=0.6, beta=0.4)
    b = po.OraclePrioritizedSampler(N, alpha=0.6, beta=0.4, tree_factory=lambda n, is_min: (
        ref_cpu.MinSegmentTreeFp32 if is_min else ref_cpu.SumSegmentTreeFp32)(n))
    g = torch.Generator().manual_seed(0)
    for smp in (a, b):
        smp.mark_update(torch.arange(3000))
    pr = torch.rand(3000, generator=g) * 4
    ids = torch.randperm(3000, generator=g)
    for smp in (a, b):
        smp.update_priority(ids, pr)
    assert float(a.default_priority) == float(b.default_priority)
    ga, gb = torch.Generator().manual_seed(7), torch.Generator().manual_seed(7)
    ia, wa = a.sample(3000, B, generator=ga)
    ib, wb = b.sample(3000, B, generator=gb)
    assert torch.equal(ia, ib) and torch.equal(wa, wb)
    # and the all-C sample path gives the same thing for the same uniforms
    u = torch.rand(B, generator=torch.Generator().manual_seed(7)).numpy()
    ic, wc, _, _ = po.per_sample_c(a._sum_tree, a._min_tree, 3000, u, 0.4)
    np.testing.assert_array_equal(ic, ia.numpy())
    np.testing.assert_array_equal(wc, wa.numpy())


@pytest.mark.parametrize("alpha,beta", [(0.6, 0.4), (0.7, 0.5), (1.0, 1.0)])
def test_sampler_restatement_equals_live_reference_sampler(ref_samplers, alpha, beta):
    """The REAL torchrl PrioritizedSampler (samplers.py imported unmodified, on the compiled reference trees) against
    oracle.OraclePrioritizedSampler through the same life cycle: writer marks, TD-error write-backs with duplicates and
    negative ("skip") indices, scalar priorities, draws from one CPU generator.  Indices, weights, default priority and
    the running max agree exactly -- this pins the restatement every GPU parity test leans on."""
    N = 1000
    ref = ref_samplers.mod.PrioritizedSampler(N, alpha, beta)
    st = ref_samplers.make_storage({"obs": torch.zeros(N)}, 0, N)
    orc = po.OraclePrioritizedSampler(N, alpha, beta)
    g = torch.Generator().manual_seed(11)
    ref._rng = torch.Generator().manual_seed(5)
    og = torch.Generator().manual_seed(5)
    filled = 0
    for it in range(8):
        n = int(torch.randint(1, 300, (), generator=g))
        idx = (filled + torch.arange(n)) % N
        filled = min(N, filled + n)
        st._len = filled
        ref.mark_update(idx, storage=st)
        orc.mark_update(idx)
        k = int(torch.randint(1, 200, (), generator=g))
        ix = torch.randint(0, filled, (k,), generator=g)
        ix[::17] = -1
        pr = torch.rand(k, generator=g) * (it + 1)
        ref.update_priority(ix, pr, storage=st)
        orc.update_priority(ix, pr)
        if it % 3 == 0:
            ref.update_priority(ix[:5].clamp_min(0), 0.25, storage=st)
            orc.update_priority(ix[:5].clamp_min(0), 0.25)
        assert float(ref.default_priority) == float(orc.default_priority)
        assert float(ref._max_priority[0]) == float(orc._max_priority)
        ri, rinfo = ref.sample(st, 64)
        oi, ow = orc.sample(filled, 64, generator=og)
        assert torch.equal(ri, oi)
        assert torch.equal(rinfo["priority_weight"], ow)


def test_double_pow_quirk():
    # SURVEY 8(a'): mark_update passes the already-powered default priority through update_priority
    s = po.OraclePrioritizedSampler(8, alpha=0.6, beta=0.4)
    s.update_priority(torch.tensor([0]), torch.tensor([4.0]))
    s.mark_update(torch.tensor([1]))
    leaf = s._sum_tree[np.array([0, 1])]
    np.testing.assert_allclose(leaf, [2.29740, 1.64718], rtol=1e-5)


# --------------------------------------------------------------------------- GAE
def _gae_inputs(shape, seed, p=0.1, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    v, nv, r = (torch.randn(*shape, generator=g, dtype=dtype) for _ in range(3))
    term = torch.rand(*shape, generator=g) < p
    done = term | (torch.rand(*shape, generator=g) < p)
    return v, nv, r, done, term


@pytest.mark.parametrize("shape", [(1, 5, 1), (3, 200, 1), (7, 3, 3, 1), (4, 17, 5)])
@pytest.mark.parametrize("gamma,lmbda", [(0.99, 0.95), (0.5, 0.1), (0.1, 0.99)])
def test_gae_c_oracle_is_reference_loop(ref_funcs, shape, gamma, lmbda):
    v, nv, r, done, term = _gae_inputs(shape, 1)
    g, l = torch.tensor(gamma), torch.tensor(lmbda)
    ra, rt = ref_funcs.generalized_advantage_estimate(g, l, v, nv, r, done=done, terminated=term)
    oa, ot = po.gae_f32(g, l, v, nv, r, done, term)
    assert torch.equal(oa, ra) and torch.equal(ot, rt)      # bit-exact: same op order, no FMA
    ta, tt = gae_torch.loop_gae(g, l, v, nv, r, done, term)
    assert torch.equal(ta, ra) and torch.equal(tt, rt)
    fa, ft = po.gae_f64(g, l, v, nv, r, done, term)
    torch.testing.assert_close(ra.double(), fa, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("shape", [(1, 5, 1), (3, 200, 1), (7, 3, 3, 1), (64, 128, 1)])
def test_gae_torch_restatement_matches_reference(ref_funcs, shape):
    v, nv, r, done, term = _gae_inputs(shape, 2)
    g, l = torch.tensor(0.99), torch.tensor(0.95)
    ra, rt = ref_funcs.vec_generalized_advantage_estimate(g, l, v, nv, r, done=done, terminated=term)
    ta, tt = gae_torch.vec_gae(g, l, v, nv, r, done, term)
    assert torch.equal(ta, ra) and torch.equal(tt, rt)


def test_gae_golden_fixture():
    """Committed golden vectors made by the imported reference (tests/golden/make_golden.py)."""
    from pathlib import Path

    f = Path(__file__).parent / "golden" / "gae_golden.npz"
    z = np.load(f)
    for k in sorted({n.split("/")[0] for n in z.files}):
        gt = lambda n: torch.from_numpy(z[f"{k}/{n}"])
        g, l = gt("gamma"), gt("lmbda")
        v, nv, r, done, term = gt("v"), gt("nv"), gt("r"), gt("done"), gt("term")
        oa, ot = po.gae_f32(g, l, v, nv, r, done, term)
        assert torch.equal(oa, gt("loop_adv")) and torch.equal(ot, gt("loop_tgt")), k
        fa, ft = po.gae_f64(g, l, v, nv, r, done, term)
        torch.testing.assert_close(gt("vec_adv").double(), fa, rtol=1e-4, atol=1e-4)  # reference's own bar
        torch.testing.assert_close(gt("loop_adv").double(), fa, rtol=1e-5, atol=1e-5)


def test_gather_oracle_is_torch_indexing():
    rng = np.random.default_rng(0)
    src = rng.integers(0, 255, (100, 4, 7, 3), dtype=np.uint8)
    idx = rng.integers(-60, 60, 33)
    out = po.gather_rows(src, idx, 60)
    assert np.array_equal(out, torch.from_numpy(src)[:60][torch.from_numpy(idx)].numpy())
    with pytest.raises(IndexError):
        po.gather_rows(src, np.array([60]), 60)


# --------------------------------------------------------------------------- TD(lambda) / TD(1)
@pytest.mark.parametrize("shape", [(1, 5, 1), (3, 100, 1), (4, 17, 5), (2, 3, 7, 1)])
@pytest.mark.parametrize("gamma,lmbda", [(0.99, 0.95), (0.9, 1.0), (0.5, 0.0)])
def test_td_lambda_c_oracle_is_reference_loop(ref_funcs, shape, gamma, lmbda):
    v, nv, r, done, term = _gae_inputs(shape, 3)
    ref = ref_funcs.td_lambda_return_estimate(gamma, lmbda, nv, r, done=done, terminated=term)
    got = po.td_lambda(gamma, lmbda, nv, r, done, term)
    assert torch.equal(got, ref)                                   # bit-exact: same op order, no FMA
    f64 = po.td_lambda(gamma, lmbda, nv, r, done, term, f64=True)
    torch.testing.assert_close(ref.double(), f64, rtol=1e-5, atol=1e-5)
    if lmbda == 1.0:                                                # TD(1) loop (functional.py:464-570) agrees
        td1 = ref_funcs.td1_return_estimate(gamma, nv, r, done=done, terminated=term)
        torch.testing.assert_close(td1.double(), f64, rtol=1e-5, atol=1e-5)


def test_td_lambda_golden_fixture():
    from pathlib import Path

    z = np.load(Path(__file__).parent / "golden" / "td_lambda_golden.npz")
    for k in sorted({n.split("/")[0] for n in z.files}):
        gt = lambda n: torch.from_numpy(z[f"{k}/{n}"])
        got = po.td_lambda(gt("gamma"), gt("lmbda"), gt("nv"), gt("r"), gt("done"), gt("term"))
        assert torch.equal(got, gt("loop")), k
        f64 = po.td_lambda(gt("gamma"), gt("lmbda"), gt("nv"), gt("r"), gt("done"), gt("term"), f64=True)
        torch.testing.assert_close(gt("vec").double(), f64, rtol=1e-4, atol=1e-4)


def test_vtrace_golden_fixture():
    """The scan oracle against the reference's V-trace loop (bit-equal: same ops in the same order) and its
    per-step-gamma GAE (cumprod + conv in the reference, recurrence here: the reference's own 1e-4 bar)."""
    from pathlib import Path

    z = np.load(Path(__file__).parent / "golden" / "vtrace_golden.npz")
    names = sorted({n.split("/")[0] for n in z.files})
    assert len(names) == 4
    for k in names:
        gt = lambda n: torch.from_numpy(z[f"{k}/{n}"])
        adv, vs = po.vtrace(float(gt("gamma")), gt("log_pi"), gt("log_mu"), gt("v"), gt("nv"), gt("r"), gt("done"),
                            gt("term"), float(gt("rho_thresh")), float(gt("c_thresh")))
        assert torch.equal(vs, gt("vs")), k
        assert torch.equal(adv, gt("adv")), k
        ga, gtg = po.gae_per_step(gt("gammas"), gt("lmbdas"), gt("v"), gt("nv"), gt("r"), gt("done"), gt("term"))
        torch.testing.assert_close(ga, gt("gae_adv"), rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(gtg, gt("gae_tgt"), rtol=1e-4, atol=1e-4)
        r2g = po.affine_scan(gt("r"), (~gt("done")).float() * float(gt("gamma")))       # reward2go, :1385-1460
        torch.testing.assert_close(r2g, gt("r2g"), rtol=1e-5, atol=1e-5)
        # the recurrence in float64 agrees with the fp32 one far inside the bar
        ga64, _ = po.gae_per_step(gt("gammas").double(), gt("lmbdas").double(), gt("v").double(), gt("nv").double(),
                                  gt("r").double(), gt("done"), gt("term"))
        torch.testing.assert_close(ga.double(), ga64, rtol=1e-5, atol=1e-5)


def test_vtrace_oracle_matches_live_reference(ref_funcs):
    g = torch.Generator().manual_seed(5)
    shape = (3, 17, 2)
    v, nv, r, lp, lm = (torch.randn(*shape, generator=g) for _ in range(5))
    term = torch.rand(*shape, generator=g) < 0.1
    done = term | (torch.rand(*shape, generator=g) < 0.1)
    ref = ref_funcs.vtrace_advantage_estimate(0.95, lp, lm, v, nv, r, done, term, 0.8, 1.2)
    got = po.vtrace(0.95, lp, lm, v, nv, r, done, term, 0.8, 1.2)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    ref = ref_funcs.vtrace_advantage_estimate(0.95, lp, lm, v, nv, r, done)       # terminated=None
    got = po.vtrace(0.95, lp, lm, v, nv, r, done)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])


# ------------------------------------------------------------------------------------------ SliceSampler (SURVEY 8f-3)
from _slice_cases import (_oracle_slice, _pslice_scenarios, _ref_pslice_run, _ref_slice_run,  # noqa: E402
                          _slice_cases)


@pytest.mark.parametrize("case", sorted(_slice_cases()))
def test_slice_oracle_equals_live_reference(ref_samplers, case):
    kwargs, data, length, max_size, last_cursor, batch_size = _slice_cases()[case]
    for seed in range(4):
        index, info, rec = _ref_slice_run(ref_samplers, kwargs, data, length, max_size, last_cursor, batch_size, seed)
        oi, otr, omask, _ = _oracle_slice(kwargs, data, length, max_size, last_cursor, batch_size, rec)
        np.testing.assert_array_equal(index.numpy(), oi)
        np.testing.assert_array_equal(info[("next", "truncated")].numpy().reshape(-1), otr)
        stored_done = data[("next", "done")][oi].numpy().reshape(-1) if ("next", "done") in data else np.zeros_like(otr)
        np.testing.assert_array_equal(info[("next", "done")].numpy().reshape(-1), stored_done | otr)
        if omask is not None:
            np.testing.assert_array_equal(info[("collector", "mask")].numpy(), omask)
        else:
            assert ("collector", "mask") not in info


def test_slice_golden_fixture():
    """tests/golden/slice_golden.npz (made by the unmodified reference) against the restatement -- runs anywhere."""
    from pathlib import Path

    from oracle import slice_oracle as so

    z = np.load(Path(__file__).parent / "golden" / "slice_golden.npz")
    names = sorted({n.split("/")[0] for n in z.files})
    assert len(names) >= 11
    for k in names:
        gt = lambda n: z[f"{k}/{n}"]
        length, max_size, cursor, seq, num_slices, strict, pad, by_traj = (int(x) for x in gt("meta"))
        sig = gt("signal")[:length]
        kw = dict(at_capacity=length == max_size, cursor=None if cursor < 0 else cursor)
        start, stop, lens = so.traj_table(trajectory=sig, **kw) if by_traj else so.traj_table(end=sig, **kw)
        np.testing.assert_array_equal(np.stack([start, stop, lens]), gt("table"))
        start, stop, lens = so.valid_trajectories(start, stop, lens, seq, bool(strict))
        oi, otr, omask, _ = so.slice_index(start, lens, seq_length=seq, num_slices=num_slices, storage_length=max_size,
                                           traj_draw=gt("traj_draw"), u=gt("u"), strict_length=bool(strict),
                                           pad_output=bool(pad))
        np.testing.assert_array_equal(oi, gt("index"))
        np.testing.assert_array_equal(otr, gt("truncated"))
        if pad:
            np.testing.assert_array_equal(omask, gt("mask"))


def _oracle_pslice(done, sum_leaves, min_leaves, L, filled, S, T, u, strict=True):
    from oracle import slice_oracle as so

    orc = po.OraclePrioritizedSampler(L, 0.7, 0.9)
    orc._sum_tree.load_leaves(sum_leaves)
    orc._min_tree.load_leaves(min_leaves)
    start, stop, length = so.traj_table(end=done[:filled], at_capacity=filled == L, cursor=None)
    return so.prioritized_slice_sample(orc, start, stop, length, seq_length=T, num_slices=S, storage_len=filled, u=u,
                                       strict_length=strict)


@pytest.mark.parametrize("strict", [True, False])
@pytest.mark.parametrize("name", sorted(_pslice_scenarios()))
def test_prioritized_slice_oracle_equals_live_reference(ref_samplers, name, strict):
    L, filled, S, T, seed = _pslice_scenarios()[name]
    done, sl, ml, draws = _ref_pslice_run(ref_samplers, L, filled, S, T, seed, strict=strict)
    for u, index, weight, truncated in draws:
        oi, ow, otr, _ = _oracle_pslice(done, sl, ml, L, filled, S, T, u, strict=strict)
        np.testing.assert_array_equal(oi, index)
        np.testing.assert_array_equal(ow, weight)
        np.testing.assert_array_equal(otr, truncated)


def test_prioritized_slice_golden_fixture():
    from pathlib import Path

    z = np.load(Path(__file__).parent / "golden" / "pslice_golden.npz")
    names = sorted({n.split("/")[0] for n in z.files})
    assert len(names) == len(_pslice_scenarios())
    for k in names:
        gt = lambda n: z[f"{k}/{n}"]
        L, filled, S, T = (int(x) for x in gt("meta"))
        for d in range(gt("u").shape[0]):
            oi, ow, otr, _ = _oracle_pslice(gt("done"), gt("sum_leaves"), gt("min_leaves"), L, filled, S, T, gt("u")[d])
            np.testing.assert_array_equal(oi, gt("index")[d])
            np.testing.assert_array_equal(ow, gt("weight")[d])


def test_slice_oracle_randomized_against_live_reference(ref_samplers):
    """Sixty random SliceSampler configurations (ring length, fill level, cursor, end density, flags vs trajectory ids,
    num_slices vs slice_len, strict / loose / padded) through the unmodified reference and through the restatement."""
    rng = np.random.default_rng(123)
    done_cases = 0
    for trial in range(60):
        L = int(rng.integers(8, 300))
        filled = L if rng.random() < 0.6 else int(rng.integers(4, L + 1))
        density = float(rng.choice([0.0, 0.02, 0.1, 0.4]))
        by_traj = bool(rng.random() < 0.3)
        done = torch.from_numpy(rng.random((L, 1)) < density)
        traj = torch.from_numpy(np.cumsum(rng.random(L) < max(density, 0.02)))
        seq = int(rng.integers(1, 12))
        S = int(rng.integers(1, 9))
        kwargs = dict(traj_key="episode") if by_traj else dict(end_key=("next", "done"))
        kwargs.update(dict(num_slices=S) if rng.random() < 0.5 else dict(slice_len=seq))
        mode = rng.integers(0, 3)
        if mode == 1:
            kwargs["strict_length"] = False
        elif mode == 2:
            kwargs.update(strict_length=False, pad_output=True)
        cursor = None
        if filled == L and rng.random() < 0.5:
            cursor = int(rng.integers(0, L)) if rng.random() < 0.5 else torch.arange(3, int(rng.integers(4, L + 1)))
        data = {("next", "done"): done, "episode": traj}
        try:
            index, info, rec = _ref_slice_run(ref_samplers, kwargs, data, filled, L, cursor, S * seq, seed=trial)
        except RuntimeError as err:                       # no trajectory long enough: the restatement must agree
            assert "sufficient length" in str(err)
            from oracle import slice_oracle as so

            c = None if cursor is None else int(cursor[-1] if isinstance(cursor, torch.Tensor) else cursor)
            start, stop, lens = (so.traj_table(trajectory=traj[:filled].numpy(), at_capacity=filled == L, cursor=c)
                                 if by_traj else so.traj_table(end=done[:filled].numpy(), at_capacity=filled == L, cursor=c))
            assert (lens < seq).all()
            continue
        oi, otr, omask, _ = _oracle_slice(kwargs, data, filled, L, cursor, S * seq, rec)
        np.testing.assert_array_equal(index.numpy(), oi, err_msg=f"trial {trial}: {kwargs}")
        np.testing.assert_array_equal(info[("next", "truncated")].numpy().reshape(-1), otr)
        if omask is not None:
            np.testing.assert_array_equal(info[("collector", "mask")].numpy(), omask)
        done_cases += 1
    assert done_cases >= 40


def test_framestack_oracle_rebuilds_what_was_written():
    """oracle/framestack_oracle.py: the plain-loop frame log, read back, equals the materialised stacks for every padding
    mode / layout / episode-start signal, and reports evictions when a ring is lapped."""
    from oracle import framestack_oracle as fo

    for n_envs, layout, pad, use_init in ((1, 0, "same", True), (3, 0, "constant", False), (4, 1, "same", False)):
        k, steps, per = 4, 96, 12
        obs, nxt, done, init = fo.make_stream(n_envs, steps, k, (3, 2), seed=5 + n_envs, pad=pad, min_len=1, max_len=15)
        ring = steps * (k + 1)
        pool = np.zeros((n_envs * ring, 3, 2), dtype=np.uint8)
        head, last = np.zeros(n_envs, dtype=np.int64), np.ones(n_envs, dtype=np.uint8)
        words, flat_o, flat_x = [], [], []
        for t0 in range(0, steps, per):
            def flat(a):
                a = a[t0:t0 + per]
                if layout == 0:
                    a = np.swapaxes(a, 0, 1)
                return np.ascontiguousarray(a).reshape(-1, *a.shape[2:])
            o, x, d, i = flat(obs), flat(nxt), flat(done), flat(init)
            words.append(fo.push(pool, head, last, o, x, i if use_init else None, d, n_envs=n_envs, layout=layout, k=k, ring=ring))
            flat_o.append(o)
            flat_x.append(x)
        w = np.concatenate(words)
        ro, rx, evicted = fo.rebuild(pool, head, w, k=k, ring=ring)
        assert not evicted.any()
        np.testing.assert_array_equal(ro, np.concatenate(flat_o))
        np.testing.assert_array_equal(rx, np.concatenate(flat_x))
        assert (w >> fo.ENV_SHIFT).max() == n_envs - 1
    # a lapped ring is reported
    obs, nxt, done, init = fo.make_stream(1, 40, 4, (2, 2), seed=1, min_len=1, max_len=1)
    pool = np.zeros((30, 2, 2), dtype=np.uint8)
    head, last = np.zeros(1, dtype=np.int64), np.ones(1, dtype=np.uint8)
    w = np.concatenate([fo.push(pool, head, last, obs[t:t + 5, 0], nxt[t:t + 5, 0], None, done[t:t + 5, 0], n_envs=1, layout=0,
                                k=4, ring=30) for t in range(0, 40, 5)])
    _, _, evicted = fo.rebuild(pool, head, w, k=4, ring=30)
    assert evicted[:30].all() and not evicted[-5:].any()
