"""Shared by tests/test_oracle.py and tests/golden/make_golden.py: SliceSampler scenarios, a runner for the UNMODIFIED
reference sampler that records its random draws, and the same scenario through oracle/slice_oracle.py."""
import numpy as np  # noqa: F401
import torch


def _ref_slice_run(R, sampler_kwargs, data, length, max_size, last_cursor, batch_size, seed):
    """Run the unmodified reference SliceSampler and record the two random draws it makes."""
    from _ref_tape import run

    return run(R, _live_slice_run, sampler_kwargs, data, length, max_size, last_cursor, batch_size, seed)


def _live_slice_run(R, sampler_kwargs, data, length, max_size, last_cursor, batch_size, seed):
    from unittest import mock

    m = R.mod
    smp = m.SliceSampler(**sampler_kwargs)
    smp._rng = torch.Generator().manual_seed(seed)
    st = R.make_storage(data, length, max_size, last_cursor)
    rec = {}
    real_randint, real_rand = torch.randint, torch.rand

    def randint(*a, **k):
        rec["traj"] = real_randint(*a, **k)
        rec["maxval"] = a[0]
        return rec["traj"]

    def rand(*a, **k):
        rec["u"] = real_rand(*a, **k)
        return rec["u"]

    with mock.patch.object(m.torch, "randint", randint), mock.patch.object(m.torch, "rand", rand):
        index, info = smp.sample(st, batch_size)
    return index[0], info, rec


def _slice_cases():
    g = torch.Generator().manual_seed(0)
    L = 400
    done = torch.rand(L, 1, generator=g) < 0.04
    traj = torch.cumsum(torch.rand(L, generator=g) < 0.05, 0)
    short = torch.zeros(L, 1, dtype=torch.bool)
    short[[3, 5, 40, 44, 200, 399]] = True
    nodone = torch.zeros(L, 1, dtype=torch.bool)
    return {
        "end_full": (dict(num_slices=8, end_key=("next", "done")), {("next", "done"): done}, L, L, None, 64),
        "end_partial": (dict(slice_len=10, end_key=("next", "done")), {("next", "done"): done}, 250, L, None, 50),
        "end_cursor": (dict(num_slices=5, end_key=("next", "done")), {("next", "done"): done}, L, L, 123, 40),
        "end_cursor_tensor": (dict(num_slices=5, end_key=("next", "done")), {("next", "done"): done}, L, L,
                              torch.arange(100, 131), 40),
        "traj_full": (dict(num_slices=6, traj_key="episode"), {"episode": traj, ("next", "done"): done}, L, L, None, 30),
        "traj_partial": (dict(num_slices=6, traj_key="episode"), {"episode": traj}, 300, L, None, 30),
        "strict_filter": (dict(num_slices=4, end_key=("next", "done")), {("next", "done"): short}, L, L, None, 80),
        "loose_variable": (dict(num_slices=16, end_key=("next", "done"), strict_length=False),
                           {("next", "done"): short}, L, L, None, 16 * 30),
        "loose_padded": (dict(num_slices=16, end_key=("next", "done"), strict_length=False, pad_output=True),
                         {("next", "done"): short}, L, L, None, 16 * 30),
        "no_end_full": (dict(num_slices=3, end_key=("next", "done")), {("next", "done"): nodone}, L, L, None, 60),
        "with_is_init": (dict(num_slices=8, end_key=("next", "done")),
                         {("next", "done"): done, "is_init": torch.roll(done, 1, 0)}, L, L, None, 64),
        "with_terminated": (dict(num_slices=8, end_key=("next", "done")),
                            {("next", "done"): done, ("next", "terminated"): done & (torch.rand(L, 1, generator=g) < 0.5)},
                            L, L, None, 64),
    }


def _oracle_slice(kwargs, data, length, max_size, last_cursor, batch_size, rec):
    from oracle import slice_oracle as so

    at_cap = length == max_size
    cursor = None
    if last_cursor is not None:
        cursor = int(last_cursor[-1]) if isinstance(last_cursor, torch.Tensor) else int(last_cursor)
    if kwargs.get("traj_key") is not None:
        start, stop, lens = so.traj_table(trajectory=data[kwargs["traj_key"]][:length].numpy(), at_capacity=at_cap,
                                          cursor=cursor)
    else:
        start, stop, lens = so.traj_table(end=data[("next", "done")][:length].numpy(), at_capacity=at_cap, cursor=cursor)
    if kwargs.get("num_slices") is not None:
        num_slices, seq = kwargs["num_slices"], batch_size // kwargs["num_slices"]
    else:
        seq, num_slices = kwargs["slice_len"], batch_size // kwargs["slice_len"]
    strict = kwargs.get("strict_length", True)
    start, stop, lens = so.valid_trajectories(start, stop, lens, seq, strict)
    assert rec["maxval"] == len(start)
    # storage.shape[0] is truncated to the fill level while the storage is not full (storages.py:856-863)
    return so.slice_index(start, lens, seq_length=seq, num_slices=num_slices, storage_length=length,
                          traj_draw=rec["traj"].numpy(), u=rec["u"].numpy(), strict_length=strict,
                          pad_output=kwargs.get("pad_output", False))


def _pslice_scenarios():
    """(L, filled, num_slices, seq_length, seed) for PrioritizedSliceSampler."""
    return {"full_small": (60, 60, 4, 5, 0), "full": (400, 400, 8, 10, 1), "partial": (400, 250, 8, 10, 2),
            "short_slices": (400, 400, 6, 3, 3), "long_slices": (1000, 1000, 4, 40, 4)}


def _ref_pslice_run(R, L, filled, S, T, seed, draws=3, strict=True):
    """Run the unmodified PrioritizedSliceSampler; returns done flags, the sum/min leaves it sampled from and, per draw,
    (u, index, weight, truncated)."""
    from _ref_tape import run

    return run(R, _live_pslice_run, L, filled, S, T, seed, draws=draws, strict=strict)


def _live_pslice_run(R, L, filled, S, T, seed, draws=3, strict=True):
    from unittest import mock

    m = R.mod
    g = torch.Generator().manual_seed(seed)
    done = torch.rand(L, 1, generator=g) < 0.06
    st = R.make_storage({("next", "done"): done}, filled, L, None)
    ref = m.PrioritizedSliceSampler(L, 0.7, 0.9, num_slices=S, end_key=("next", "done"), strict_length=strict)
    ref._rng = torch.Generator().manual_seed(seed + 100)
    ref.mark_update(torch.arange(filled), storage=st)
    ref.update_priority(torch.arange(filled), torch.rand(filled, generator=g) * 3, storage=st)
    sum_leaves = np.array([ref._sum_tree[i] for i in range(L)], dtype=np.float32)
    min_leaves = np.array([ref._min_tree[i] for i in range(L)], dtype=np.float32)
    out = []
    real = torch.rand
    for _ in range(draws):
        rec = {}

        def rand(*a, **k):
            rec["u"] = real(*a, **k)
            return rec["u"]

        with mock.patch.object(m.torch, "rand", rand):
            idx, info = ref.sample(st, S * T)
        out.append((rec["u"].numpy(), idx[0].numpy(), info["priority_weight"].numpy(),
                    info[("next", "truncated")].numpy().reshape(-1)))
    return done.reshape(-1).numpy(), sum_leaves, min_leaves, out
