"""Host-side logic of the TorchRL-facing mirror (cursors, lengths, key plumbing, bookkeeping quirks, error
behaviour), exercised on CPU with the oracle-backed emulator standing in for the CUDA library
(tests/_emul.py).  The arithmetic itself is checked on the GPU in tests/test_gpu_kernels.py; here the
expected values come from the compiled reference trees / the restated reference glue (oracle/)."""
import numpy as np
import pytest
import torch

from oracle import per_oracle as po
from rl_b200 import ops
from rl_b200.data import (LazyTensorStorage, ListStorage, PrioritizedReplayBuffer, PrioritizedSampler, RandomSampler,
                          ReplayBuffer, RoundRobinWriter, TensorDict, TensorDictPrioritizedReplayBuffer,
                          TensorDictReplayBuffer, TensorStorage)
from rl_b200.objectives.value import GAE, vec_generalized_advantage_estimate


# ------------------------------------------------------------------------------------------- C1 plumbing
def test_config1_liststorage_randomsampler_cartpole():
    """BASELINE configs[0]: ListStorage + RandomSampler, 10k cap, CartPole-shaped, batch 32, CPU.  Pure host
    plumbing -- no kernel is involved, so it runs without any backend."""
    torch.manual_seed(0)
    g = torch.Generator().manual_seed(0)
    rb = ReplayBuffer(storage=ListStorage(10_000), sampler=RandomSampler(), batch_size=32, generator=g)
    items = [TensorDict({"obs": torch.randn(4), "action": torch.randint(0, 2, (1,))}, []) for _ in range(500)]
    for it in items[:10]:
        rb.add(it)
    idx = rb.extend(items[10:])
    assert len(rb) == 500 and idx.tolist() == list(range(10, 500))
    batch, info = rb.sample(return_info=True)
    assert batch.batch_size == torch.Size([32])
    assert batch.get("obs").shape == (32, 4) and batch.get("action").dtype == torch.int64
    want = torch.stack([items[i].get("obs") for i in info["index"].tolist()])
    assert torch.equal(batch.get("obs"), want)
    # same generator state => same indices (test/rb/test_rb_core.py:113-131 style)
    g.manual_seed(5)
    a = rb.sample(return_info=True)[1]["index"]
    g.manual_seed(5)
    b = rb.sample(return_info=True)[1]["index"]
    assert torch.equal(a, b)
    with pytest.raises(RuntimeError, match="batch_size not specified"):
        ReplayBuffer(storage=ListStorage(10)).sample()
    with pytest.raises(RuntimeError, match="Cannot sample from an empty storage"):
        ReplayBuffer(storage=ListStorage(10), batch_size=2).sample()


def test_liststorage_semantics():
    st = ListStorage(3)
    st.set(0, "a")
    st.set(1, "b")
    with pytest.raises(RuntimeError, match="more than one item away"):
        st.set(3, "d")
    st.set(2, "c")
    with pytest.raises(RuntimeError, match="maximum capacity"):
        st.set(3, "d")
    assert st.get([0, 2]) == ["a", "c"] and st.get(torch.tensor([1])) == ["b"] and len(st) == 3
    rb = ReplayBuffer(storage=ListStorage(5), batch_size=2)
    rb.extend(list(range(7)))  # wraps round-robin
    assert rb.storage._storage == [5, 6, 2, 3, 4]


def test_no_cpu_fallback_in_product_path():
    """Without the emulator a tensor-index read of a TensorStorage must fail loudly on this GPU-less box."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    ops.set_backend(None)
    st = TensorStorage(torch.arange(10.0))
    assert st.get(3) == 3.0  # views need no kernel
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        st.get(torch.tensor([1, 2]))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        PrioritizedSampler(10, 0.6, 0.4, device="cpu")


# ------------------------------------------------------------------------------------------- storages / writers
def test_lazy_tensor_storage_bookkeeping(emul):
    st = LazyTensorStorage(10, device="cpu")
    assert len(st) == 0 and not st.initialized
    with pytest.raises(RuntimeError, match="non-initialized"):
        st.get(0)
    w = RoundRobinWriter()
    w.register_storage(st)
    data = TensorDict({"a": torch.arange(6.0).reshape(6, 1), "n": {"b": torch.arange(6)}}, [6])
    idx = w.extend(data)
    assert idx.tolist() == list(range(6)) and len(st) == 6 and w._cursor == 6 and w._write_count == 6
    assert st.shape == torch.Size([6]) and not st._is_full
    idx = w.extend(data)  # wraps: 6..9, 0, 1  -> scatter path
    assert idx.tolist() == [6, 7, 8, 9, 0, 1] and len(st) == 10 and w._cursor == 2 and st._is_full
    got = st.get(torch.tensor([0, 1, 2, 6, 9]))
    assert got.get(("n", "b")).tolist() == [4, 5, 2, 0, 3]
    assert got.batch_size == torch.Size([5])
    assert st.get(slice(0, 3)).get("a").squeeze(-1).tolist() == [4.0, 5.0, 2.0]
    assert st[7].get(("n", "b")).item() == 1
    # negative indices wrap by len (torch indexing semantics)
    assert st.get(torch.tensor([-1])).get(("n", "b")).item() == 3
    st._empty()
    assert len(st) == 0
    # pytree (tuple) storage and plain tensors
    st2 = LazyTensorStorage(8, device="cpu")
    rb = ReplayBuffer(storage=st2, batch_size=4)
    rb.extend((torch.arange(5), torch.arange(5.0).unsqueeze(-1)))
    out = rb[torch.tensor([4, 0])]
    assert isinstance(out, tuple) and out[0].tolist() == [4, 0] and out[1].shape == (2, 1)
    st3 = TensorStorage(torch.arange(12.0).reshape(6, 2))
    assert len(st3) == 6 and torch.equal(st3.get(torch.tensor([5, 0])), torch.tensor([[10.0, 11.0], [0.0, 1.0]]))
    with pytest.raises(ValueError, match="max-size and the storage shape mismatch"):
        TensorStorage(torch.zeros(4), max_size=5)


def test_shared_storage_prioritized_sampler(emul):
    """test/rb/test_rb_core.py:577-601: a second buffer on the same storage sees the writes (mark_update)."""
    n = 100
    storage = LazyTensorStorage(n, device="cpu")
    writer = RoundRobinWriter()
    rb0 = ReplayBuffer(storage=storage, writer=writer, sampler=RandomSampler(), batch_size=10)
    rb1 = ReplayBuffer(storage=storage, writer=writer, sampler=PrioritizedSampler(max_capacity=n, alpha=0.7, beta=1.1),
                       batch_size=10)
    rb0.extend(TensorDict({"a": torch.arange(50)}, [50]))
    assert len(rb0) == 50 and len(storage) == 50 and len(rb1) == 50
    rb0.sample()
    rb1.sample()
    assert rb1._sampler._sum_tree.query(0, 10) == 10
    assert rb1._sampler._sum_tree.query(0, 50) == 50
    assert rb1._sampler._sum_tree.query(0, 70) == 50


# ------------------------------------------------------------------------------------------- PER glue vs reference
def _oracle_sampler(N, alpha, beta, ref_cpu):
    f = lambda n, is_min: (ref_cpu.MinSegmentTreeFp32 if is_min else ref_cpu.SumSegmentTreeFp32)(n)  # noqa: E731
    return po.OraclePrioritizedSampler(N, alpha, beta, tree_factory=f)


def test_prioritized_buffer_matches_reference_glue(emul, ref_cpu):
    """extend (default priorities + td_error write-back), sample under a fixed seed, update_tensordict_priority:
    indices, weights and tree leaves equal the reference sampler glue over the compiled reference trees."""
    N, B = 2000, 128
    alpha, beta = 0.6, 0.4
    g = torch.Generator().manual_seed(3)
    rb = TensorDictPrioritizedReplayBuffer(alpha=alpha, beta=beta, storage=LazyTensorStorage(N, device="cpu"),
                                           batch_size=B, generator=g)
    ref = _oracle_sampler(N, alpha, beta, ref_cpu)
    gd = torch.Generator().manual_seed(11)
    for n in (700, 900, 650):  # the last one wraps around
        td_err = torch.rand(n, generator=gd) * 3
        data = TensorDict({"obs": torch.randn(n, 4, generator=gd), "td_error": td_err}, [n])
        cur = rb.writer._cursor
        idx = rb.extend(data)
        want_idx = torch.arange(cur, cur + n) % N
        assert torch.equal(idx, want_idx) and torch.equal(data.get("index"), want_idx)
        ref.mark_update(want_idx)               # writer -> mark_update            (writers.py:232-235)
        ref.update_priority(want_idx, td_err)   # then the td_error of the new data (replay_buffers.py:1903-1907)
    smp = rb.sampler
    np.testing.assert_array_equal(smp._sum_tree.dump_leaves().numpy(), ref._sum_tree[np.arange(N)])
    np.testing.assert_array_equal(smp._min_tree.dump_leaves().numpy(), ref._min_tree[np.arange(N)])
    assert float(smp._max_priority[0]) == float(ref._max_priority)
    assert float(smp.default_priority) == float(ref.default_priority)
    for _ in range(3):
        state = g.get_state()
        sample = rb.sample()
        g2 = torch.Generator()
        g2.set_state(state)
        want_idx, want_w = ref.sample(len(rb), B, generator=g2)
        assert torch.equal(sample.get("index"), want_idx)
        assert torch.equal(sample.get("priority_weight"), want_w)
        assert torch.equal(sample.get("obs"), rb.storage.get(slice(None)).get("obs")[want_idx])
        new_td = torch.rand(B, generator=gd) * 2
        sample.set("td_error", new_td)
        rb.update_tensordict_priority(sample)
        ref.update_priority(want_idx, new_td)
        np.testing.assert_array_equal(smp._sum_tree.values.numpy()[1:2], [np.float32(ref._sum_tree.query(0, N))])


def test_double_pow_quirk_and_default_priority(emul):
    rb = ReplayBuffer(storage=LazyTensorStorage(8, device="cpu"),
                      sampler=PrioritizedSampler(8, alpha=0.6, beta=0.4), batch_size=2)
    assert rb.sampler.default_priority == (1 + 1e-8) ** 0.6
    idx = rb.extend(torch.arange(2.0))
    rb.update_priority(idx[:1], torch.tensor([4.0]))
    rb.extend(torch.arange(1.0))  # new item gets ((4+eps)^a + eps)^a, not (4+eps)^a   (SURVEY 8a')
    leaves = rb.sampler._sum_tree.dump_leaves()
    np.testing.assert_allclose(leaves[[0, 2]].numpy(), [2.29740, 1.64718], rtol=1e-5)
    assert float(rb.sampler._max_priority[0]) == 4.0


def test_prb_update_max_priority(emul):
    """test/rb/test_samplers.py:1152-1188 (value part; the argmax index is only kept with
    max_priority_within_buffer=True, like the reference's CUDA branch)."""
    for within in (True, False):
        rb = ReplayBuffer(storage=LazyTensorStorage(11, device="cpu"),
                          sampler=PrioritizedSampler(max_capacity=11, alpha=1.0, beta=1.0,
                                                     max_priority_within_buffer=within))
        for data in torch.arange(20):
            idx = rb.add(data)
            rb.update_priority(idx, 21 - data)
            if data <= 10 or not within:
                assert rb.sampler._max_priority[0] == 21
            else:
                leaves = rb.sampler._sum_tree.dump_leaves()
                assert rb.sampler._max_priority[0] == leaves.max()
                assert rb.sampler._max_priority[1] == leaves.argmax()
        idx = rb.extend(torch.arange(10))
        rb.update_priority(idx, 12)
        assert rb.sampler._max_priority[0] == (12 if within else 21)


def test_priority_weight_formula(emul):
    """test/rb/test_prioritized.py:278-338: priority_weight == ((p+eps)^alpha / min)^(-beta), obs == index."""
    size, B, alpha, beta, eps = 64, 16, 0.7, 0.5, 1e-8
    pr = torch.linspace(0.1, 2.0, size)
    tree_p = (pr + eps).pow(alpha)
    rb = TensorDictReplayBuffer(storage=LazyTensorStorage(size, device="cpu"),
                                sampler=PrioritizedSampler(size, alpha, beta, eps, device="cpu"), batch_size=B,
                                priority_key="td_error")
    rb.extend(TensorDict({"obs": torch.arange(size), "td_error": pr}, [size]))
    for _ in range(8):
        s = rb.sample()
        i = s.get("index")
        torch.testing.assert_close(s.get("obs"), i)
        torch.testing.assert_close(s.get("td_error"), pr[i])
        torch.testing.assert_close(s.get("priority_weight"), (tree_p[i] / tree_p.min()).pow(-beta))


def test_prb_rng(emul):
    """test/rb/test_rb_core.py:113-131: same generator state => identical PER sample."""
    g = torch.Generator().manual_seed(0)
    rb = PrioritizedReplayBuffer(alpha=0.7, beta=0.9, storage=LazyTensorStorage(50, device="cpu"), batch_size=8,
                                 generator=g)
    rb.extend(torch.arange(50.0))
    rb.update_priority(torch.arange(50), torch.rand(50))
    st = g.get_state()
    a = rb.sample()
    b = rb.sample()
    g.set_state(st)
    c = rb.sample()
    assert torch.equal(a, c) and not torch.equal(a, b)


def test_update_priority_shapes_and_negative_index(emul):
    smp = PrioritizedSampler(16, 1.0, 1.0, device="cpu")
    smp.update_priority(torch.arange(4), 2.0)                       # scalar priority
    smp.update_priority(3, torch.tensor(5.0))                        # int index, 0-d priority
    smp.update_priority(torch.tensor([5, -1, 6]), torch.tensor([1.0, 100.0, 3.0]))  # -1 = skip
    leaves = smp._sum_tree.dump_leaves()
    assert leaves[:7].tolist() == pytest.approx([2, 2, 2, 5, 0, 1, 3], rel=1e-6)
    assert float(smp._max_priority[0]) == 5.0   # the skipped 100 must not count
    with pytest.raises(RuntimeError, match="priority should be a number or an iterable"):
        smp.update_priority(torch.arange(4), torch.ones(3))
    with pytest.raises(ValueError, match="alpha must be greater or equal than 0"):
        PrioritizedSampler(4, -1.0, 1.0)
    with pytest.raises(ValueError, match="beta must be greater or equal to 0"):
        PrioritizedSampler(4, 1.0, -1.0)


def test_sampler_dumps_loads_reference_layout(emul, tmp_path):
    """On-disk layout of samplers.py:1120-1204: float64 leaves memmaps + json metadata."""
    smp = PrioritizedSampler(37, 0.6, 0.4, device="cpu")
    smp.update_priority(torch.arange(30), torch.rand(30) + 0.1)
    smp.dumps(tmp_path / "s")
    mm = np.memmap(tmp_path / "s" / "sumtree.memmap", dtype=np.float64, mode="r", shape=(37,))
    np.testing.assert_array_equal(np.asarray(mm), smp._sum_tree.dump_leaves().double().numpy())
    other = PrioritizedSampler(37, 0.1, 0.1, device="cpu")
    other.loads(tmp_path / "s")
    assert torch.equal(other._sum_tree.values[1:], smp._sum_tree.values[1:])
    assert torch.equal(other._min_tree.values[1:], smp._min_tree.values[1:])
    assert other.alpha == 0.6 and float(other._max_priority[0]) == float(smp._max_priority[0])
    sd = smp.state_dict()
    third = PrioritizedSampler(37, 0.6, 0.4, device="cpu")
    third.load_state_dict(sd)
    assert torch.equal(third._sum_tree.values[1:], smp._sum_tree.values[1:])


def test_buffer_dumps_loads(emul, tmp_path):
    g = torch.Generator().manual_seed(1)
    mk = lambda: TensorDictPrioritizedReplayBuffer(alpha=0.6, beta=0.4, storage=LazyTensorStorage(20, device="cpu"),
                                                   batch_size=5, generator=torch.Generator().manual_seed(1))
    rb = mk()
    rb.extend(TensorDict({"x": torch.randn(13, 3, generator=g), "td_error": torch.rand(13, generator=g)}, [13]))
    rb.dumps(tmp_path / "rb")
    rb2 = mk()
    rb2.extend(TensorDict({"x": torch.zeros(1, 3), "td_error": torch.zeros(1)}, [1]))  # initialise the layout
    rb2.loads(tmp_path / "rb")
    assert len(rb2) == 13 and rb2.writer._cursor == 13
    a, b = rb.sample(), rb2.sample()
    assert torch.equal(a.get("index"), b.get("index")) and torch.equal(a.get("x"), b.get("x"))


# ------------------------------------------------------------------------------------------- GAE plumbing
def _gae_td(B, T, seed=0):
    g = torch.Generator().manual_seed(seed)
    term = torch.rand(B, T, 1, generator=g) < 0.05
    return TensorDict({
        "state_value": torch.randn(B, T, 1, generator=g),
        "next": {"state_value": torch.randn(B, T, 1, generator=g), "reward": torch.randn(B, T, 1, generator=g),
                 "done": term | (torch.rand(B, T, 1, generator=g) < 0.05), "terminated": term},
    }, [B, T])


def test_gae_module_keys_and_values(emul, ref_funcs):
    td = _gae_td(5, 40)
    mod = GAE(gamma=0.99, lmbda=0.95, value_network=None)
    out = mod(td)
    assert out is td and td.get("advantage").shape == (5, 40, 1)
    ra, rt = ref_funcs.generalized_advantage_estimate(
        mod.gamma, mod.lmbda, td.get("state_value"), td.get(("next", "state_value")), td.get(("next", "reward")),
        done=td.get(("next", "done")), terminated=td.get(("next", "terminated")))
    assert torch.equal(td.get("advantage"), ra) and torch.equal(td.get("value_target"), rt)
    # custom keys, average_gae, skip_existing
    mod2 = GAE(gamma=0.9, lmbda=0.8, value_network=None, average_gae=True, skip_existing=True)
    mod2.set_keys(advantage="adv", value_target=("tgt", "v"))
    td2 = _gae_td(3, 17, 1)
    mod2(td2)
    assert abs(td2.get("adv").mean()) < 1e-5 and td2.get(("tgt", "v")).shape == (3, 17, 1)
    before = td2.get("adv").clone()
    td2.set(("next", "reward"), torch.zeros(3, 17, 1))
    mod2(td2)  # skip_existing: untouched
    assert torch.equal(td2.get("adv"), before)
    with pytest.raises(ValueError, match="is missing, and no value network was provided"):
        GAE(gamma=0.9, lmbda=0.9, value_network=None)(TensorDict({"next": {"reward": torch.zeros(2, 3, 1),
                                                                        "done": torch.zeros(2, 3, 1, dtype=torch.bool)}},
                                                                 [2, 3]))
    with pytest.raises(NotImplementedError):
        GAE(gamma=0.9, lmbda=0.9, value_network=None, differentiable=True)
    # a critic callable is invoked on the data and on data["next"]
    calls = []

    def critic(t):
        calls.append(1)
        t.set("state_value", torch.ones(*t.batch_size, 1))

    td3 = _gae_td(2, 6, 2)
    GAE(gamma=0.99, lmbda=0.95, value_network=critic)(td3)
    assert len(calls) == 2 and td3.get("value_target").shape == (2, 6, 1)


def test_gae_functional_errors_and_time_dim(emul, ref_funcs):
    v = torch.randn(4, 9, 1)
    with pytest.raises(RuntimeError, match="must share a unique shape"):
        vec_generalized_advantage_estimate(0.9, 0.9, v, v[:, :8], v, torch.zeros(4, 9, 1, dtype=torch.bool))
    nd = torch.zeros(4, 9, 1, dtype=torch.bool)          # a constant per-step gamma tensor == the scalar path
    a_t, _ = vec_generalized_advantage_estimate(torch.full((4, 9, 1), 0.9), 0.9, v, v, v, nd)
    a_s, _ = vec_generalized_advantage_estimate(0.9, 0.9, v, v, v, nd)
    torch.testing.assert_close(a_t, a_s, rtol=1e-5, atol=1e-5)
    g = torch.Generator().manual_seed(0)
    v, nv, r = (torch.randn(6, 11, generator=g) for _ in range(3))
    done = torch.rand(6, 11, generator=g) < 0.1
    a, t = vec_generalized_advantage_estimate(0.99, 0.95, v, nv, r, done=done, time_dim=-1)
    ra, rt = ref_funcs.generalized_advantage_estimate(0.99, 0.95, v, nv, r, done=done, time_dim=-1)
    assert a.shape == (6, 11) and torch.equal(a, ra) and torch.equal(t, rt)
    a, t = vec_generalized_advantage_estimate(0.99, 0.95, v.t().unsqueeze(-1), nv.t().unsqueeze(-1),
                                              r.t().unsqueeze(-1), done=done.t().unsqueeze(-1), time_dim=0)
    assert a.shape == (11, 6, 1) and torch.equal(a.squeeze(-1).t(), ra)
    # python-float vs tensor gamma/lmbda are rounded the way the reference rounds them
    from rl_b200.objectives.value.functional import gae_scalars

    gm, gl = gae_scalars(torch.tensor(0.99), torch.tensor(0.95), torch.float32)
    assert gl == float(torch.tensor(0.99) * torch.tensor(0.95))
    gm2, gl2 = gae_scalars(0.99, 0.95, torch.float32)
    assert gl2 == float(torch.tensor(0.99 * 0.95, dtype=torch.float32))


def test_td_estimators_plumbing(emul, ref_funcs):
    """TD(0)/TD(1)/TD(lambda) functionals: signatures, shape errors, time_dim, advantage = return - value."""
    from rl_b200.objectives.value import (td0_advantage_estimate, td0_return_estimate, td1_return_estimate,
                                          td_lambda_advantage_estimate, vec_td1_advantage_estimate,
                                          vec_td_lambda_return_estimate)

    g = torch.Generator().manual_seed(0)
    v, nv, r = (torch.randn(4, 12, 1, generator=g) for _ in range(3))
    term = torch.rand(4, 12, 1, generator=g) < 0.1
    done = term | (torch.rand(4, 12, 1, generator=g) < 0.1)
    ref = ref_funcs.td_lambda_return_estimate(0.99, 0.9, nv, r, done=done, terminated=term)
    got = vec_td_lambda_return_estimate(0.99, 0.9, nv, r, done, term)
    assert torch.equal(got, ref)      # the emulator runs the C restatement, bit-equal to the reference loop
    adv = td_lambda_advantage_estimate(0.99, 0.9, v, nv, r, done, term)
    assert torch.equal(adv, ref - v)
    ref1 = ref_funcs.td1_return_estimate(0.99, nv, r, done=done, terminated=term)
    torch.testing.assert_close(td1_return_estimate(0.99, nv, r, done, term), ref1, rtol=1e-5, atol=1e-5)
    assert torch.equal(vec_td1_advantage_estimate(0.99, v, nv, r, done, term), td1_return_estimate(0.99, nv, r, done, term) - v)
    assert torch.equal(td0_return_estimate(0.99, nv, r, term), ref_funcs.td0_return_estimate(0.99, nv, r, term))
    assert torch.equal(td0_advantage_estimate(0.99, v, nv, r, done, term),
                       ref_funcs.td0_advantage_estimate(0.99, v, nv, r, done, term))
    got_t = vec_td_lambda_return_estimate(0.99, 0.9, nv.squeeze(-1), r.squeeze(-1), done.squeeze(-1), term.squeeze(-1),
                                          time_dim=-1)
    assert torch.equal(got_t, ref.squeeze(-1))
    with pytest.raises(RuntimeError, match="must share a unique shape"):
        vec_td_lambda_return_estimate(0.99, 0.9, nv, r[:, :5], done, term)
    with pytest.raises(NotImplementedError, match="tensor-valued"):
        vec_td_lambda_return_estimate(torch.full((4, 12, 1), 0.9), 0.9, nv, r, done, term)
    with pytest.raises(RuntimeError, match="rolling_gamma=False"):
        vec_td_lambda_return_estimate(0.99, 0.9, nv, r, done, term, rolling_gamma=False)


def test_vtrace_and_per_step_gae_plumbing(emul, ref_funcs):
    """vtrace_advantage_estimate / tensor-valued gamma, lmbda: signature, time_dim, shape errors, values."""
    from rl_b200.objectives.value import vec_generalized_advantage_estimate, vtrace_advantage_estimate

    g = torch.Generator().manual_seed(1)
    shape = (4, 12, 1)
    v, nv, r, lp, lm = (torch.randn(*shape, generator=g) for _ in range(5))
    term = torch.rand(*shape, generator=g) < 0.1
    done = term | (torch.rand(*shape, generator=g) < 0.1)
    ref = ref_funcs.vtrace_advantage_estimate(0.99, lp, lm, v, nv, r, done, term, 1.0, 0.9)
    got = vtrace_advantage_estimate(0.99, lp, lm, v, nv, r, done, term, 1.0, 0.9)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])     # emulator = C scan, same op order
    ref = ref_funcs.vtrace_advantage_estimate(0.99, lp, lm, v, nv, r, done, rho_thresh=torch.tensor(0.5))
    got = vtrace_advantage_estimate(0.99, lp, lm, v, nv, r, done, rho_thresh=torch.tensor(0.5))
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    sq = lambda t: t.squeeze(-1)
    ref_t = ref_funcs.vtrace_advantage_estimate(0.99, sq(lp), sq(lm), sq(v), sq(nv), sq(r), sq(done), sq(term),
                                                time_dim=-1)
    got_t = vtrace_advantage_estimate(0.99, sq(lp), sq(lm), sq(v), sq(nv), sq(r), sq(done), sq(term), time_dim=-1)
    assert got_t[0].shape == ref_t[0].shape == (4, 12)
    assert torch.equal(got_t[0], ref_t[0]) and torch.equal(got_t[1], ref_t[1])
    with pytest.raises(RuntimeError, match="must share a unique shape"):
        vtrace_advantage_estimate(0.99, lp, lm, v, nv, r[:, :5], done, term)

    gammas = 0.9 + 0.1 * torch.rand(*shape, generator=g)
    lmbdas = 0.8 + 0.2 * torch.rand(*shape, generator=g)
    ref = ref_funcs.vec_generalized_advantage_estimate(gammas, lmbdas, v, nv, r, done=done, terminated=term)
    got = vec_generalized_advantage_estimate(gammas, lmbdas, v, nv, r, done, term)
    torch.testing.assert_close(got[0], ref[0], rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(got[1], ref[1], rtol=1e-4, atol=1e-4)
    ref = ref_funcs.vec_generalized_advantage_estimate(gammas, 0.95, v, nv, r, done=done, terminated=term)
    got = vec_generalized_advantage_estimate(gammas, 0.95, v, nv, r, done, term)     # tensor gamma, scalar lmbda
    torch.testing.assert_close(got[0], ref[0], rtol=1e-4, atol=1e-4)
    ref_t = ref_funcs.vec_generalized_advantage_estimate(sq(gammas), sq(lmbdas), sq(v), sq(nv), sq(r), done=sq(done),
                                                         terminated=sq(term), time_dim=-1)
    got_t = vec_generalized_advantage_estimate(sq(gammas), sq(lmbdas), sq(v), sq(nv), sq(r), sq(done), sq(term),
                                               time_dim=-1)
    assert got_t[0].shape == ref_t[0].shape
    torch.testing.assert_close(got_t[0], ref_t[0], rtol=1e-4, atol=1e-4)
    with pytest.raises(NotImplementedError, match="forward-only"):
        vec_generalized_advantage_estimate(gammas.requires_grad_(), lmbdas, v, nv, r, done, term)

    from rl_b200.objectives.value import reward2go
    for shp, tdim in [((4, 20, 1), -2), ((4, 20, 3), -2), ((2, 3, 20, 1), -2), ((20, 2), -2), ((5, 20), -1),
                      ((4, 20, 1), 1)]:
        rr = torch.randn(*shp, generator=g)
        dd = torch.rand(*shp, generator=g) < 0.15
        ref = ref_funcs.reward2go(rr, dd, 0.97, time_dim=tdim)
        got = reward2go(rr, dd, 0.97, time_dim=tdim)
        assert got.shape == ref.shape == rr.shape
        torch.testing.assert_close(got, ref, rtol=1e-5, atol=1e-5)
    ones, dn = torch.ones(1, 10), torch.zeros(1, 10, dtype=torch.bool)       # the docstring example, :1408-1422
    dn[:, [3, 7]] = True
    torch.testing.assert_close(reward2go(ones, dn, 0.99, time_dim=-1).flatten(),
                               torch.tensor([3.9404, 2.9701, 1.99, 1.0, 3.9404, 2.9701, 1.99, 1.0, 1.99, 1.0]),
                               rtol=1e-4, atol=1e-4)
    with pytest.raises(ValueError, match="must share the same shape"):
        reward2go(ones, dn[:, :5], 0.99)


@pytest.mark.parametrize("drop_last", [True, False])
@pytest.mark.parametrize("shuffle", [True, False])
def test_sampler_without_replacement(emul, drop_last, shuffle):
    """samplers.py:221-362 / test/rb/test_samplers.py: every item once per sweep, ran_out ends __iter__,
    a PPO-style epoch loop over GAE output runs through the same buffer."""
    from rl_b200.data import SamplerWithoutReplacement

    n, B = 23, 5
    rb = TensorDictReplayBuffer(storage=LazyTensorStorage(n, device="cpu"),
                                sampler=SamplerWithoutReplacement(drop_last=drop_last, shuffle=shuffle), batch_size=B,
                                generator=torch.Generator().manual_seed(0))
    td = _gae_td(1, n)
    GAE(gamma=0.99, lmbda=0.95, value_network=None)(td)
    rb.extend(td.reshape(n))
    for epoch in range(2):
        seen = [b.get("index") for b in rb]
        flat = torch.cat(seen)
        if drop_last:
            assert len(seen) == n // B and all(s.numel() == B for s in seen) and flat.unique().numel() == flat.numel()
        else:
            assert len(seen) == -(n // -B) and sorted(flat.tolist()) == list(range(n))
        if not shuffle:
            assert flat.tolist() == list(range(flat.numel()))
    b = rb.sample()
    assert torch.equal(b.get("advantage"), td.get("advantage").reshape(n, 1)[b.get("index")])
    with pytest.raises(ValueError, match="greater than the storage capacity"):
        ReplayBuffer(storage=LazyTensorStorage(3, device="cpu"), sampler=SamplerWithoutReplacement(drop_last=True),
                     batch_size=8)._sampler.sample(type("S", (), {"__len__": lambda s: 3, "ndim": 1, "device": "cpu"})(), 8)


@pytest.mark.parametrize("case", ["end_full", "end_partial", "traj_full", "strict_filter", "loose_variable", "loose_padded",
                                  "with_terminated", "with_is_init", "no_end_full"])
def test_slice_sampler_equals_live_reference(emul, ref_samplers, case):
    """rl_b200 SliceSampler inside a TensorDictReplayBuffer (kernels emulated by the oracle) against the UNMODIFIED
    reference sampler on the same contents with the same CPU generator seed: same slices, same info, same rows."""
    from _slice_cases import _slice_cases
    from rl_b200.data import SliceSampler

    kwargs, data, length, max_size, last_cursor, batch_size = _slice_cases()[case]
    td = TensorDict({k: v[:length] for k, v in data.items()}, [length])
    td.set("obs", torch.arange(length, dtype=torch.float32).unsqueeze(-1))
    rb = TensorDictReplayBuffer(storage=LazyTensorStorage(max_size, device="cpu"), sampler=SliceSampler(**kwargs),
                                batch_size=batch_size, generator=torch.Generator().manual_seed(3))
    rb.extend(td)
    ref = ref_samplers.mod.SliceSampler(**kwargs)
    ref._rng = torch.Generator().manual_seed(3)
    cursor = rb.storage._last_cursor
    st = ref_samplers.make_storage({**{k: v for k, v in data.items()}, "obs": td.get("obs") if length == max_size else
                                    torch.cat([td.get("obs"), torch.zeros(max_size - length, 1)])}, length, max_size,
                                   range(cursor.start, cursor.stop) if isinstance(cursor, slice) else cursor)
    for _ in range(3):
        want_index, want_info = ref.sample(st, batch_size)
        got = rb.sample()
        assert torch.equal(got.get("index").reshape(-1), want_index[0])
        for k, v in want_info.items():
            assert torch.equal(got.get(k).reshape(v.shape), v), k
        assert torch.equal(got.get("obs").reshape(-1), want_index[0].float())     # the rows are the indexed rows


def test_slice_sampler_contract(emul):
    from rl_b200.data import SliceSampler

    with pytest.raises(TypeError, match="Either num_slices or slice_len"):
        SliceSampler()
    with pytest.raises(ValueError, match="pad_output=True is incompatible"):
        SliceSampler(num_slices=2, pad_output=True)
    assert SliceSampler(num_slices=2, span=True)._span_code == (-1, -1)
    assert SliceSampler(num_slices=2, span=(False, 3))._span_code == (0, 3)
    with pytest.raises(RuntimeError, match="requires `cache_values`"):
        SliceSampler(num_slices=2, ends=torch.zeros(10, dtype=torch.bool))
    L = 60
    done = torch.zeros(L, 1, dtype=torch.bool)
    done[[9, 29, 59]] = True
    rb = TensorDictReplayBuffer(storage=LazyTensorStorage(L, device="cpu"), batch_size=12,
                                sampler=SliceSampler(num_slices=3, end_key=("next", "done"), cache_values=True))
    rb.extend(TensorDict({("next", "done"): done, "t": torch.arange(L)}, [L]))
    b = rb.sample()
    t = b.get("t").reshape(3, 4)
    assert (t[:, 1:] - t[:, :-1] == 1).all()                      # consecutive steps of one trajectory
    assert b.get(("next", "truncated")).reshape(3, 4)[:, -1].all()
    assert ("table", 4) in rb.sampler._cache
    rb.extend(TensorDict({("next", "done"): done[:5], "t": torch.arange(5)}, [5]))
    assert not rb.sampler._cache                                  # a write drops the cached table
    with pytest.raises(RuntimeError, match="divisible by the number of slices"):
        rb.sample(10)
    with pytest.raises(RuntimeError, match="sufficient length"):
        rb.sample(3 * 40)
    # ends= given up front: the table never depends on the storage contents
    rb2 = TensorDictReplayBuffer(storage=LazyTensorStorage(L, device="cpu"), batch_size=8,
                                 sampler=SliceSampler(slice_len=4, ends=done.squeeze(-1), cache_values=True))
    rb2.extend(TensorDict({"t": torch.arange(L)}, [L]))
    t = rb2.sample().get("t").reshape(2, 4)
    assert (t[:, 1:] - t[:, :-1] == 1).all()


@pytest.mark.parametrize("strict", [True, False])
@pytest.mark.parametrize("filled", [400, 250])
def test_prioritized_slice_sampler_equals_live_reference(emul, ref_samplers, filled, strict):
    """PrioritizedSliceSampler in a TensorDictReplayBuffer (kernels emulated) against the UNMODIFIED reference class:
    same starts, slices, per-step weights and flags for the same CPU generator seed, through writes, TD-error
    write-backs and repeated draws."""
    from rl_b200.data import PrioritizedSliceSampler

    L, S, T = 400, 8, 10
    g = torch.Generator().manual_seed(0)
    done = torch.rand(L, 1, generator=g) < 0.06
    kw = dict(num_slices=S, end_key=("next", "done"), strict_length=strict)
    rb = TensorDictReplayBuffer(storage=LazyTensorStorage(L, device="cpu"), batch_size=S * T,
                                sampler=PrioritizedSliceSampler(L, 0.7, 0.9, **kw),
                                generator=torch.Generator().manual_seed(2), priority_key="td_error")
    ref = ref_samplers.mod.PrioritizedSliceSampler(L, 0.7, 0.9, **kw)
    ref._rng = torch.Generator().manual_seed(2)
    obs = torch.arange(L, dtype=torch.float32).unsqueeze(-1)
    rb.extend(TensorDict({("next", "done"): done[:filled], "obs": obs[:filled]}, [filled]))
    st = ref_samplers.make_storage({("next", "done"): done, "obs": obs}, filled, L, range(0, filled))   # _last_cursor
    ref.mark_update(torch.arange(filled), storage=st)
    for rep in range(4):
        ix = torch.randint(0, filled, (50,), generator=g)
        pr = torch.rand(50, generator=g) * 3
        rb.update_priority(ix, pr)
        ref.update_priority(ix, pr, storage=st)
        want_index, want_info = ref.sample(st, S * T)
        got = rb.sample()
        assert torch.equal(got.get("index").reshape(-1), want_index[0])
        assert torch.equal(got.get("priority_weight").reshape(-1), want_info["priority_weight"])
        for k in (("next", "truncated"), ("next", "done"), ("next", "terminated")):
            assert torch.equal(got.get(k).reshape(-1), want_info[k].reshape(-1)), k
        assert torch.equal(got.get("obs").reshape(-1), obs[want_index[0]].reshape(-1))
        if strict:
            t = got.get("obs").reshape(S, T)
            assert (t[:, 1:] - t[:, :-1] == 1).all() and not done[:filled][got.get("index").reshape(S, T)[:, :-1]].any()
    # the true priorities were never altered by sampling
    orc_leaves = torch.tensor([ref._sum_tree[i] for i in range(filled)])
    assert torch.equal(rb.sampler._sum_tree.dump_leaves()[:filled].cpu(), orc_leaves)


@pytest.mark.parametrize("case", ["end_full", "strict_filter", "loose_variable", "traj_partial"])
@pytest.mark.parametrize("shuffle", [True, False])
def test_slice_sampler_without_replacement_equals_live_reference(emul, ref_samplers, case, shuffle):
    """SliceSamplerWithoutReplacement against the UNMODIFIED reference class, same CPU generator: a full sweep over the
    trajectories and into the next one -- same slices, same ran_out sequence."""
    from _slice_cases import _slice_cases
    from rl_b200.data import SliceSamplerWithoutReplacement

    kwargs, data, length, max_size, last_cursor, batch_size = _slice_cases()[case]
    kwargs = {k: v for k, v in kwargs.items() if k != "pad_output"}
    td = TensorDict({k: v[:length] for k, v in data.items()}, [length])
    td.set("obs", torch.arange(length, dtype=torch.float32).unsqueeze(-1))
    rb = TensorDictReplayBuffer(storage=LazyTensorStorage(max_size, device="cpu"), batch_size=batch_size,
                                sampler=SliceSamplerWithoutReplacement(shuffle=shuffle, **kwargs),
                                generator=torch.Generator().manual_seed(4))
    rb.extend(td)
    ref = ref_samplers.mod.SliceSamplerWithoutReplacement(shuffle=shuffle, **kwargs)
    ref._rng = torch.Generator().manual_seed(4)
    cursor = rb.storage._last_cursor
    st = ref_samplers.make_storage({k: v for k, v in data.items()}, length, max_size,
                                   range(cursor.start, cursor.stop) if isinstance(cursor, slice) else cursor)
    raised = 0
    for _ in range(12):
        try:
            want_index, want_info = ref.sample(st, batch_size)
        except RuntimeError as err:      # a batch of trajectories that are all too short: the reference gives up, so do we
            assert "sufficient length" in str(err)
            with pytest.raises(RuntimeError, match="sufficient length"):
                rb.sample()
            raised += 1
            continue
        got = rb.sample()
        assert torch.equal(got.get("index").reshape(-1), want_index[0])
        assert torch.equal(got.get(("next", "truncated")).reshape(-1), want_info[("next", "truncated")].reshape(-1))
        assert rb.sampler.ran_out == ref.ran_out
        assert torch.equal(got.get("obs").reshape(-1), want_index[0].float())


def test_td_estimator_modules_and_nstep_gae(emul, ref_funcs):
    """TD0Estimator / TD1Estimator / TDLambdaEstimator (advantages.py:622-1336) write value_target = the functional's
    return and advantage = value_target - value; GAE with steps_to_next_obs uses gamma ** steps per step (:1576-1578)."""
    from rl_b200.objectives.value import GAE, TD0Estimator, TD1Estimator, TDLambdaEstimator

    g = torch.Generator().manual_seed(0)
    B, T = 6, 20
    v, nv, r = (torch.randn(B, T, 1, generator=g) for _ in range(3))
    term = torch.rand(B, T, 1, generator=g) < 0.05
    done = term | (torch.rand(B, T, 1, generator=g) < 0.05)

    def make():
        return TensorDict({"state_value": v.clone(), "next": {"state_value": nv.clone(), "reward": r.clone(),
                                                              "done": done.clone(), "terminated": term.clone()}}, [B, T])

    td = TDLambdaEstimator(gamma=0.98, lmbda=0.9, value_network=None)(make())
    want = ref_funcs.td_lambda_return_estimate(0.98, 0.9, nv, r, done=done, terminated=term)
    torch.testing.assert_close(td.get("value_target"), want, rtol=1e-5, atol=1e-5)
    assert torch.equal(td.get("advantage"), td.get("value_target") - v)
    td = TD1Estimator(gamma=0.98, value_network=None)(make())
    torch.testing.assert_close(td.get("value_target"), ref_funcs.td1_return_estimate(0.98, nv, r, done=done, terminated=term),
                               rtol=1e-5, atol=1e-5)
    td = TD0Estimator(gamma=0.98, value_network=None)(make())
    torch.testing.assert_close(td.get("value_target"), ref_funcs.td0_return_estimate(0.98, nv, r, term))
    est = TDLambdaEstimator(gamma=0.98, lmbda=0.9, value_network=None, advantage_key="adv", value_target_key="ret",
                            average_rewards=True)
    td = est(make())
    assert "adv" in td.keys() and "ret" in td.keys() and est.out_keys == ["adv", "ret"]
    rn = (r - r.mean()) / r.std().clamp_min(1e-4)
    torch.testing.assert_close(td.get(("next", "reward")), rn)           # rewards are normalised in place, as upstream
    torch.testing.assert_close(td.get("ret"), ref_funcs.td_lambda_return_estimate(0.98, 0.9, nv, rn, done=done, terminated=term),
                               rtol=1e-5, atol=1e-5)
    # critic given: called on the data and on its "next"
    calls = []

    def critic(t):
        calls.append(1)
        t.set("state_value", t.get("obs") * 2)

    data = make()
    data.set("obs", v.clone())
    data.get("next").set("obs", nv.clone())
    td = TD0Estimator(gamma=0.9, value_network=critic)(data)
    assert len(calls) == 2
    torch.testing.assert_close(td.get("value_target"), r + 0.9 * (~term).int() * (nv * 2))
    # n-step transitions
    data = make()
    steps = torch.randint(1, 4, (B, T, 1), generator=g)
    data.set("steps_to_next_obs", steps)
    out = GAE(gamma=0.97, lmbda=0.9, value_network=None)(data)
    gam = torch.tensor(0.97) ** steps
    want_adv, want_tgt = ref_funcs.vec_generalized_advantage_estimate(gam, torch.tensor(0.9), v, nv, r, done=done,
                                                                      terminated=term)
    torch.testing.assert_close(out.get("advantage"), want_adv, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(out.get("value_target"), want_tgt, rtol=1e-4, atol=1e-4)


def test_prefetch_thread_pool(emul):
    """ReplayBuffer(prefetch=k) (replay_buffers.py:340-341, 1155-1164): batches come from a queue fed by worker threads;
    a without-replacement sweep still yields every item exactly once and stops at ran_out."""
    from rl_b200.data import SamplerWithoutReplacement

    n = 40
    rb = TensorDictPrioritizedReplayBuffer(alpha=0.6, beta=0.4, storage=LazyTensorStorage(n, device="cpu"), batch_size=8,
                                           prefetch=2, generator=torch.Generator().manual_seed(0))
    rb.extend(TensorDict({"obs": torch.arange(n, dtype=torch.float32).unsqueeze(-1), "td_error": torch.rand(n)}, [n]))
    for _ in range(6):
        b = rb.sample()
        assert torch.equal(b.get("obs").reshape(-1), b.get("index").reshape(-1).float())
        assert 1 <= len(rb._prefetch_queue) <= 2                       # the queue is topped up behind the consumer
    rb2 = TensorDictReplayBuffer(storage=LazyTensorStorage(n, device="cpu"), batch_size=8, prefetch=3,
                                 sampler=SamplerWithoutReplacement(), generator=torch.Generator().manual_seed(0))
    rb2.extend(TensorDict({"obs": torch.arange(n, dtype=torch.float32).unsqueeze(-1)}, [n]))
    seen = torch.cat([rb2.sample().get("index").reshape(-1) for _ in range(5)])
    assert sorted(seen.tolist()) == list(range(n))


def test_default_priority_after_skip_only_update(emul):
    """update_priority with only negative ("skip") indices leaves max_priority unset in the reference (samplers.py:1040-1052):
    the next writer batch still gets the initial default priority, through both write paths."""
    from rl_b200.data import PrioritizedSampler

    orc = po.OraclePrioritizedSampler(50, 0.6, 0.4)
    orc.update_priority(torch.tensor([-1, -1]), torch.tensor([3.0, 4.0]))
    orc.mark_update(torch.arange(10))
    for fused in (True, False):
        smp = PrioritizedSampler(50, 0.6, 0.4, device="cpu")
        smp.update_priority(torch.tensor([-1, -1]), torch.tensor([3.0, 4.0]))
        if fused:
            smp.mark_update_range(0, 10, 50)
        else:
            smp.mark_update(torch.arange(10))
        np.testing.assert_array_equal(smp._sum_tree.values.numpy()[1:], orc._sum_tree.values()[1:])
        assert float(smp._max_priority_buf[0]) == float(orc._max_priority)


def test_predraw_keeps_the_random_stream(emul):
    """PrioritizedSampler.predraw draws each sample's uniforms one call early: same torch.rand calls in the same order,
    so the sampled indices are those of the plain sampler for the same seed."""
    def run(predraw):
        rb = TensorDictPrioritizedReplayBuffer(alpha=0.6, beta=0.4, storage=LazyTensorStorage(200, device="cpu"),
                                               batch_size=16, generator=torch.Generator().manual_seed(3))
        rb.sampler.predraw = predraw
        rb.extend(TensorDict({"obs": torch.arange(200.0).unsqueeze(-1),
                              "td_error": torch.rand(200, generator=torch.Generator().manual_seed(1))}, [200]))
        out = []
        for i in range(5):
            b = rb.sample()
            out.append(b.get("index").clone())
            rb.update_priority(b.get("index"), torch.full((16,), float(i + 1)))
        return torch.stack(out)

    assert torch.equal(run(False), run(True))


@pytest.mark.parametrize("drop_last", [True, False])
@pytest.mark.parametrize("shuffle", [True, False])
def test_sampler_without_replacement_equals_live_reference(emul, ref_samplers, drop_last, shuffle):
    """SamplerWithoutReplacement against the UNMODIFIED reference class (samplers.py:221-362): same index batches, same
    ran_out sequence and _remaining_batches over three sweeps and a storage that grows in between."""
    from rl_b200.data import SamplerWithoutReplacement

    ref = ref_samplers.mod.SamplerWithoutReplacement(drop_last=drop_last, shuffle=shuffle)
    mine = SamplerWithoutReplacement(drop_last=drop_last, shuffle=shuffle)
    ref._rng = torch.Generator().manual_seed(8)
    mine._rng = torch.Generator().manual_seed(8)
    st_ref = ref_samplers.make_storage({"obs": torch.zeros(64)}, 23, 64)
    st = LazyTensorStorage(64, device="cpu")
    st.set(slice(0, 23), TensorDict({"obs": torch.zeros(23)}, [23]))
    for it in range(30):
        if it == 17:            # the storage grows: both start a new permutation
            st_ref._len = 40
            st.set(slice(23, 40), TensorDict({"obs": torch.zeros(17)}, [17]))
        a, _ = ref.sample(st_ref, 5)
        b, _ = mine.sample(st, 5)
        assert torch.equal(a, b), it
        assert ref.ran_out == mine.ran_out
        assert ref._remaining_batches == mine._remaining_batches


def _sample_quietly(rb):
    """A draw whose result is not compared (the reference could not produce it); the oracle-backed emulator may itself
    give up on degenerate batches (every slice cut to zero steps)."""
    try:
        rb.sample()
    except (RuntimeError, IndexError, ValueError):
        pass


def test_slice_sampler_randomized_buffer_flows_vs_live_reference(emul, ref_samplers):
    """Forty random buffers (ring length, several writer batches that may wrap, end density, strict / loose / padded,
    num_slices / slice_len, cache on / off): rl_b200's SliceSampler in a TensorDictReplayBuffer against the unmodified
    reference sampler on a mirror of the ring, same CPU generator seed."""
    from rl_b200.data import SliceSampler

    rng = np.random.default_rng(77)
    compared = 0
    for trial in range(80):
        L = int(rng.integers(10, 200))
        seq, S = int(rng.integers(1, 9)), int(rng.integers(1, 7))
        kwargs = dict(end_key=("next", "done"))
        kwargs.update(dict(num_slices=S) if rng.random() < 0.5 else dict(slice_len=seq))
        mode = int(rng.integers(0, 3))
        if mode == 1:
            kwargs["strict_length"] = False
        elif mode == 2:
            kwargs.update(strict_length=False, pad_output=True)
        if trial >= 40:   # span=: slices may hang out of their trajectory on either side and are cut there (:2071-2118)
            pick = lambda: [False, True, int(rng.integers(1, max(2, seq)))][int(rng.integers(0, 3))]
            sp = (pick(), pick())
            sp = tuple(v if (v is True or v is False or v < seq) else False for v in sp)
            if not any(sp):
                sp = (True, False)
            kwargs["span"] = sp
            if mode == 2:     # (the padded + span corner emits a mask only when a slice was actually cut, data-dependent
                kwargs.pop("pad_output")   # in the reference; the concatenated form is the one pinned here)
        cache = bool(rng.random() < 0.5)
        rb = TensorDictReplayBuffer(storage=LazyTensorStorage(L, device="cpu"), batch_size=S * seq,
                                    sampler=SliceSampler(cache_values=cache, **kwargs),
                                    generator=torch.Generator().manual_seed(trial))
        ref = ref_samplers.mod.SliceSampler(cache_values=False, **kwargs)
        ref._rng = torch.Generator().manual_seed(trial)
        ring_done = torch.zeros(L, 1, dtype=torch.bool)
        ring_obs = torch.zeros(L, 1)
        total = 0
        for _ in range(int(rng.integers(1, 4))):
            n = int(rng.integers(1, L + 1))
            done = torch.from_numpy(rng.random((n, 1)) < float(rng.choice([0.0, 0.05, 0.3])))
            obs = torch.arange(total, total + n, dtype=torch.float32).unsqueeze(-1)
            rb.extend(TensorDict({("next", "done"): done, "obs": obs}, [n]))
            slots = (total + torch.arange(n)) % L
            ring_done[slots], ring_obs[slots] = done, obs
            total += n
            filled = min(L, total)
            cur = rb.storage._last_cursor
            cur = range(cur.start, cur.stop) if isinstance(cur, slice) else cur
            st = ref_samplers.make_storage({("next", "done"): ring_done, "obs": ring_obs}, filled, L, cur)
            for _ in range(2):
                try:
                    want_index, want_info = ref.sample(st, S * seq)
                except RuntimeError as err:
                    if "Boolean value of Tensor" in str(err) and kwargs.get("span"):
                        # an integer span next to per-slice lengths (strict_length=False): the reference compares the int
                        # with a tensor in an `if` (samplers.py:2079 / :2091) and cannot produce this batch at all
                        _sample_quietly(rb)
                        rb._rng.set_state(ref._rng.get_state())
                        continue
                    assert "sufficient length" in str(err)
                    with pytest.raises(RuntimeError, match="sufficient length"):
                        rb.sample()
                    continue
                except ValueError as err:
                    # (with strict_length=False the reference compares the span with the CLAMPED per-slice length when
                    # there is a single slice -- a data-dependent rejection this engine does not reproduce)
                    assert "strictly lower than the sequence length" in str(err)
                    _sample_quietly(rb)
                    rb._rng.set_state(ref._rng.get_state())
                    continue
                except IndexError as err:   # a single stored step: the reference squeezes its flags to 0-d (:1913-1915)
                    # (or every slice was cut to zero steps by a span: the reference indexes an empty tensor, :2187)
                    assert "0-dim" in str(err) or "size 0" in str(err)
                    _sample_quietly(rb)
                    rb._rng.set_state(ref._rng.get_state())
                    continue
                except TypeError as err:
                    # the reference's right span calls torch.minimum(int, Tensor) when nothing made seq_length a tensor
                    # before (samplers.py:2114): it cannot produce this batch at all.  Keep the generators in step.
                    assert "minimum()" in str(err) and kwargs.get("span")
                    _sample_quietly(rb)
                    rb._rng.set_state(ref._rng.get_state())
                    continue
                got = rb.sample()
                assert torch.equal(got.get("index").reshape(-1), want_index[0]), (trial, kwargs)
                for k, v in want_info.items():
                    assert torch.equal(got.get(k).reshape(v.shape), v), (trial, k)
                assert torch.equal(got.get("obs").reshape(-1), ring_obs[want_index[0]].reshape(-1))
                compared += 1
    assert compared >= 120


def test_prioritized_slice_sampler_randomized_vs_live_reference(emul, ref_samplers):
    """Twenty-five random PrioritizedSliceSampler buffers (wrapping writer batches, TD-error write-backs with duplicates)
    against the unmodified reference class: same starts, per-step weights and flags."""
    from rl_b200.data import PrioritizedSliceSampler

    rng = np.random.default_rng(5)
    compared = 0
    for trial in range(25):
        L = int(rng.integers(30, 200))
        seq, S = int(rng.integers(2, 8)), int(rng.integers(1, 6))
        alpha, beta = float(rng.choice([0.5, 0.7, 1.0])), float(rng.choice([0.4, 1.0]))
        kw = dict(num_slices=S, end_key=("next", "done"))
        rb = TensorDictReplayBuffer(storage=LazyTensorStorage(L, device="cpu"), batch_size=S * seq,
                                    sampler=PrioritizedSliceSampler(L, alpha, beta, **kw),
                                    generator=torch.Generator().manual_seed(trial))
        ref = ref_samplers.mod.PrioritizedSliceSampler(L, alpha, beta, **kw)
        ref._rng = torch.Generator().manual_seed(trial)
        ring_done = torch.zeros(L, 1, dtype=torch.bool)
        total = 0
        for _ in range(int(rng.integers(1, 4))):
            n = int(rng.integers(1, L + 1))
            done = torch.from_numpy(rng.random((n, 1)) < float(rng.choice([0.02, 0.1])))
            rb.extend(TensorDict({("next", "done"): done, "obs": torch.zeros(n, 1)}, [n]))
            slots = (total + torch.arange(n)) % L
            ring_done[slots] = done
            total += n
            filled = min(L, total)
            cur = rb.storage._last_cursor
            cur = range(cur.start, cur.stop) if isinstance(cur, slice) else cur
            st = ref_samplers.make_storage({("next", "done"): ring_done}, filled, L, cur)
            ref.mark_update(slots, storage=st)
            k = int(rng.integers(1, 40))
            ix = torch.from_numpy(rng.integers(0, filled, k))
            pr = torch.from_numpy((rng.random(k) * 3).astype(np.float32))
            rb.update_priority(ix, pr)
            ref.update_priority(ix, pr, storage=st)
            try:
                want_index, want_info = ref.sample(st, S * seq)
            except RuntimeError as err:          # every start masked out (all trajectories shorter than the slice)
                assert "p_sum" in str(err) or "sufficient" in str(err), err
                continue
            got = rb.sample()
            assert torch.equal(got.get("index").reshape(-1), want_index[0]), trial
            assert torch.equal(got.get("priority_weight").reshape(-1), want_info["priority_weight"]), trial
            assert torch.equal(got.get(("next", "done")).reshape(-1), want_info[("next", "done")].reshape(-1))
            compared += 1
    assert compared >= 25


# ---------------------------------------------------------------------------------------------------- checkpointer
def test_tensor_storage_checkpointer_layout_and_roundtrip(emul, tmp_path):
    """TensorStorageCheckpointer (checkpointers.py:326-455): tensordict-memmap layout for TensorDict storages -- one raw
    <key>.memmap per leaf in nested directories + meta.json + storage_metadata.json -- and the reference's own pytree
    layout for tensors / pytrees; both round-trip, and only the filled rows travel."""
    import json

    import numpy as np

    from rl_b200.data import LazyTensorStorage, TensorDict, TensorStorageCheckpointer

    g = torch.Generator().manual_seed(0)
    st = LazyTensorStorage(50, device="cpu")
    assert isinstance(st.checkpointer, TensorStorageCheckpointer)
    data = TensorDict({"obs": torch.randn(30, 4, generator=g), "action": torch.randint(0, 5, (30, 1), generator=g),
                       "next": {"obs": torch.randn(30, 4, generator=g), "done": torch.rand(30, 1, generator=g) < 0.5,
                                "half": torch.randn(30, 3, generator=g).to(torch.bfloat16)}}, [30])
    st.set(slice(0, 30), data)
    st.dumps(tmp_path / "td")
    meta = json.loads((tmp_path / "td" / "storage_metadata.json").read_text())
    assert meta == {"metadata": {}, "is_pytree": False, "len": 30}
    root = json.loads((tmp_path / "td" / "meta.json").read_text())
    assert root["shape"] == [50] and root["obs"] == {"device": "cpu", "shape": [50, 4], "dtype": "torch.float32"}
    assert root["action"]["dtype"] == "torch.int64" and "_type" in root
    nxt = json.loads((tmp_path / "td" / "next" / "meta.json").read_text())
    assert nxt["done"] == {"device": "cpu", "shape": [50, 1], "dtype": "torch.bool"}
    raw = np.memmap(tmp_path / "td" / "obs.memmap", dtype=np.float32, mode="r", shape=(50, 4))   # the full-size leaf
    np.testing.assert_array_equal(raw[:30], data.get("obs").numpy())
    assert (tmp_path / "td" / "next" / "obs.memmap").stat().st_size == 50 * 4 * 4
    # into an initialised storage and into a fresh lazy one
    for fresh in (False, True):
        st2 = LazyTensorStorage(50, device="cpu")
        if not fresh:
            st2.set(slice(0, 5), data[:5])
        st2.loads(tmp_path / "td")
        assert len(st2) == 30
        got = st2.get(torch.arange(30))
        for k in data.keys(True, True):
            assert torch.equal(got.get(k), data.get(k)), k
    # pytree / bare tensor storages: the reference's _save_pytree layout (utils.py:818-873)
    tree = {"a": torch.randn(20, 3, generator=g), "b": (torch.arange(20), torch.rand(20, 2, generator=g))}
    sp = LazyTensorStorage(40, device="cpu")
    sp.set(slice(0, 20), tree)
    sp.dumps(tmp_path / "tree")
    md = json.loads((tmp_path / "tree" / "storage_metadata.json").read_text())
    assert md["is_pytree"] and md["len"] == 20
    assert md["metadata"]["a"] == {"dtype": "torch.float32", "shape": [40, 3]}
    assert md["metadata"]["b.0"] == {"dtype": "torch.int64", "shape": [40]} and "b.1" in md["metadata"]
    assert (tmp_path / "tree" / "b" / "1.memmap").exists()
    sp2 = LazyTensorStorage(40, device="cpu")
    sp2.set(slice(0, 3), {"a": tree["a"][:3], "b": (tree["b"][0][:3], tree["b"][1][:3])})
    sp2.loads(tmp_path / "tree")
    out = sp2.get(torch.arange(20))
    assert torch.equal(out["a"], tree["a"]) and torch.equal(out["b"][0], tree["b"][0]) and torch.equal(out["b"][1], tree["b"][1])
    s1 = LazyTensorStorage(10, device="cpu")
    s1.set(slice(0, 4), torch.arange(8.0).view(4, 2))
    s1.dumps(tmp_path / "single")
    assert (tmp_path / "single" / "_-single-tensor-_.memmap").exists()
    with pytest.raises(RuntimeError, match="non-initialized"):
        LazyTensorStorage(10, device="cpu").dumps(tmp_path / "empty")


@pytest.mark.parametrize("mode", ["strict", "loose", "padded", "span", "traj"])
def test_slice_sampler_2d_storage_equals_live_reference(emul, ref_samplers, mode):
    """ndim=2 storages ([T, E]: one ring per column, samplers.py:1652-1743, :1955): rl_b200's SliceSampler in a
    TensorDictReplayBuffer against the unmodified reference sampler on the same [T, E, ...] contents -- partially filled
    and full rings, same CPU generator seed: same (time, column) index pairs, same info, same rows."""
    from rl_b200.data import SliceSampler

    rng = np.random.default_rng({"strict": 1, "loose": 2, "padded": 3, "span": 4, "traj": 5}[mode])
    for trial in range(6):
        T, E = int(rng.integers(20, 90)), int(rng.integers(2, 6))
        seq, S = int(rng.integers(2, 7)), int(rng.integers(1, 6))
        kwargs = dict(num_slices=S) if rng.random() < 0.5 else dict(slice_len=seq)
        if mode == "traj":
            kwargs["traj_key"] = "episode"
        else:
            kwargs["end_key"] = ("next", "done")
        if mode == "loose":
            kwargs["strict_length"] = False
        elif mode == "padded":
            kwargs.update(strict_length=False, pad_output=True)
        elif mode == "span":
            kwargs["span"] = (True, int(rng.integers(1, seq))) if rng.random() < 0.5 else (False, True)
        # time along dim 0 of the storage: the data below is [time, env], so it is extended along dim 0
        rb = TensorDictReplayBuffer(storage=LazyTensorStorage(T * E, device="cpu", ndim=2), batch_size=S * seq,
                                    sampler=SliceSampler(**kwargs), generator=torch.Generator().manual_seed(trial),
                                    dim_extend=0)
        ref = ref_samplers.mod.SliceSampler(**kwargs)
        ref._rng = torch.Generator().manual_seed(trial)
        ring = {("next", "done"): torch.zeros(T, E, 1, dtype=torch.bool), "obs": torch.zeros(T, E, 1),
                "episode": torch.zeros(T, E, dtype=torch.long)}
        total = 0
        ep = torch.arange(E) * 1000
        for _ in range(int(rng.integers(1, 4))):
            n = int(rng.integers(1, T + 1))
            done = torch.from_numpy(rng.random((n, E, 1)) < float(rng.choice([0.03, 0.1, 0.3])))
            obs = (torch.arange(total, total + n, dtype=torch.float32).view(n, 1, 1) * 10 + torch.arange(E).view(1, E, 1)).float()
            episode = torch.empty(n, E, dtype=torch.long)
            for t in range(n):
                episode[t] = ep
                ep = ep + done[t, :, 0].long()
            rb.extend(TensorDict({("next", "done"): done, "obs": obs, "episode": episode}, [n, E]))
            rows = (total + torch.arange(n)) % T
            ring[("next", "done")][rows], ring["obs"][rows], ring["episode"][rows] = done, obs, episode
            total += n
            filled = min(T, total)
            cur = rb.storage._last_cursor
            cur = range(cur.start, cur.stop) if isinstance(cur, slice) else cur
            st = ref_samplers.make_storage(dict(ring), filled, T, cur, columns=E)
            for _ in range(2):
                try:
                    want_index, want_info = ref.sample(st, S * seq)
                except RuntimeError as err:
                    if "Boolean value of Tensor" in str(err) and kwargs.get("span"):
                        # an integer span next to per-slice lengths (strict_length=False): the reference compares the int
                        # with a tensor in an `if` (samplers.py:2079 / :2091) and cannot produce this batch at all
                        _sample_quietly(rb)
                        rb._rng.set_state(ref._rng.get_state())
                        continue
                    assert "sufficient length" in str(err)
                    with pytest.raises(RuntimeError, match="sufficient length"):
                        rb.sample()
                    continue
                except TypeError as err:   # the reference's torch.minimum(int, Tensor) bug (samplers.py:2114)
                    assert "minimum()" in str(err) and kwargs.get("span")
                    _sample_quietly(rb)
                    rb._rng.set_state(ref._rng.get_state())
                    continue
                got = rb.sample()
                gi = got.get("index")
                assert torch.equal(gi[..., 0].reshape(-1), want_index[0]) and torch.equal(gi[..., 1].reshape(-1), want_index[1]), \
                    (mode, trial, kwargs)
                for k, v in want_info.items():
                    assert torch.equal(got.get(k).reshape(v.shape), v), (mode, trial, k)
                assert torch.equal(got.get("obs").reshape(-1), ring["obs"][want_index].reshape(-1))


def test_gae_module_rereads_annealed_discount(emul):
    """GAE caches its scalar discounts for a sync-free forward, but in-place changes of the buffers (annealing,
    load_state_dict) must be seen: the cache is keyed on the buffers' version counters (ADVICE r1)."""
    from rl_b200.objectives.value import GAE, vec_generalized_advantage_estimate

    td = _gae_td(3, 12, seed=4)
    mod = GAE(gamma=0.99, lmbda=0.95, value_network=None)
    out1 = mod(td.clone()).get("advantage")
    mod.gamma.fill_(0.5)
    mod.lmbda.mul_(0.5)
    out2 = mod(td.clone()).get("advantage")
    want, _ = vec_generalized_advantage_estimate(0.5, 0.475, td.get("state_value"), td.get(("next", "state_value")),
                                                 td.get(("next", "reward")), td.get(("next", "done")),
                                                 td.get(("next", "terminated")), time_dim=-2)
    assert not torch.allclose(out1, out2)
    torch.testing.assert_close(out2, want, rtol=1e-6, atol=1e-6)
    sd = GAE(gamma=0.9, lmbda=0.8, value_network=None).state_dict()
    mod.load_state_dict(sd)
    want3, _ = vec_generalized_advantage_estimate(0.9, 0.8, td.get("state_value"), td.get(("next", "state_value")),
                                                  td.get(("next", "reward")), td.get(("next", "done")),
                                                  td.get(("next", "terminated")), time_dim=-2)
    torch.testing.assert_close(mod(td.clone()).get("advantage"), want3, rtol=1e-6, atol=1e-6)


def test_bench_group_plan_covers_every_step_count():
    """bench.py times EXACTLY K steps whatever K is: full groups of the planned size plus one shorter tail graph."""
    import bench

    for quantum in (1, 4):
        for k in range(1, 260):
            spg, rem = bench.group_plan(k, quantum)
            assert spg % quantum == 0 and 1 <= spg <= max(20, quantum)
            assert (k // spg) * spg + rem == k and 0 <= rem < spg
            if rem == 0:
                assert k % spg == 0
    assert bench.group_plan(200, 1) == (20, 0) and bench.group_plan(20, 4) == (20, 0) and bench.group_plan(50, 1) == (10, 0)
    cfg = bench.make_config(1)
    assert cfg["workload"] == bench.make_config(8)["workload"]
