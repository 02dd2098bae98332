"""Generates tests/golden/*.npz by importing the UNMODIFIED reference (a torchrl source checkout).

    RLB_REFERENCE_ROOT=/path/to/torchrl-checkout python tests/golden/make_golden.py

gae_golden.npz  inputs + outputs of the reference's generalized_advantage_estimate (loop) and
                vec_generalized_advantage_estimate (torchrl/objectives/value/functional.py:119-180,
                270-370) on seeded inputs, CPU fp32.
per_golden.npz  leaves, uniform draws, sampled indices and IS weights from the compiled reference
                CPU segment trees (oracle/_ref/cpu) driven by the restated sampler glue
                (samplers.py:895-956, 966-1091), including the KAT of test_prioritized.py:113-140.
"""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from oracle import per_oracle as po  # noqa: E402
from oracle.ref_loader import reference_ext, reference_functionals, reference_trees  # noqa: E402

OUT = Path(__file__).resolve().parent


def gae_cases():
    F = reference_functionals()
    out = {}
    cases = {
        "c3_small": ((64, 128, 1), 0.99, 0.95, 0.02),
        "bench_like": ((32, 512, 1), 0.99, 0.95, 0.1),
        "short": ((7, 3, 1), 0.5, 0.1, 0.3),
        "multi_f": ((5, 33, 3), 0.9, 0.99, 0.1),
        "nd_batch": ((3, 4, 50, 1), 0.99, 0.5, 0.05),
        "odd_T": ((9, 131, 1), 0.99, 0.95, 0.05),
        "long_T": ((2, 1000, 1), 0.999, 0.97, 0.01),
    }
    for i, (name, (shape, gamma, lmbda, p)) in enumerate(cases.items()):
        g = torch.Generator().manual_seed(100 + i)
        v, nv, r = (torch.randn(*shape, generator=g) for _ in range(3))
        term = torch.rand(*shape, generator=g) < p
        done = term | (torch.rand(*shape, generator=g) < p)
        gm, lm = torch.tensor(gamma), torch.tensor(lmbda)
        la, lt = F.generalized_advantage_estimate(gm, lm, v, nv, r, done=done, terminated=term)
        va, vt = F.vec_generalized_advantage_estimate(gm, lm, v, nv, r, done=done, terminated=term)
        for k, t in dict(gamma=gm, lmbda=lm, v=v, nv=nv, r=r, done=done, term=term, loop_adv=la,
                         loop_tgt=lt, vec_adv=va, vec_tgt=vt).items():
            out[f"{name}/{k}"] = t.numpy()
    np.savez_compressed(OUT / "gae_golden.npz", **out)


def td_cases():
    F = reference_functionals()
    out = {}
    cases = {"lam95": ((16, 128, 1), 0.99, 0.95, 0.05), "td1": ((8, 64, 1), 0.97, 1.0, 0.1),
             "odd": ((5, 37, 1), 0.9, 0.5, 0.2), "multi_f": ((4, 25, 3), 0.99, 0.9, 0.1)}
    for i, (name, (shape, gamma, lmbda, p)) in enumerate(cases.items()):
        g = torch.Generator().manual_seed(300 + i)
        nv, r = (torch.randn(*shape, generator=g) for _ in range(2))
        term = torch.rand(*shape, generator=g) < p
        done = term | (torch.rand(*shape, generator=g) < p)
        loop = F.td_lambda_return_estimate(gamma, lmbda, nv, r, done=done, terminated=term)
        vec = F.vec_td_lambda_return_estimate(gamma, lmbda, nv, r, done=done, terminated=term)
        for k, t in dict(gamma=torch.tensor(gamma), lmbda=torch.tensor(lmbda), nv=nv, r=r, done=done, term=term,
                         loop=loop, vec=vec).items():
            out[f"{name}/{k}"] = t.numpy()
    np.savez_compressed(OUT / "td_lambda_golden.npz", **out)


def scan_cases():
    """vtrace_golden.npz: the reference's vtrace_advantage_estimate (functional.py:1297-1382) and
    vec_generalized_advantage_estimate with per-step gamma / lmbda tensors (functional.py:317-370), and reward2go."""
    F = reference_functionals()
    out = {}
    cases = {"impala": ((16, 80, 1), 0.99, 0.05, 1.0, 1.0), "clip": ((4, 33, 1), 0.9, 0.2, 0.7, 1.3),
             "multi_f": ((3, 20, 2), 0.97, 0.1, 1.0, 0.9), "nd": ((2, 3, 40, 1), 0.99, 0.05, 1.0, 1.0)}
    for i, (name, (shape, gamma, p, rho_t, c_t)) in enumerate(cases.items()):
        g = torch.Generator().manual_seed(400 + i)
        v, nv, r = (torch.randn(*shape, generator=g) for _ in range(3))
        log_pi, log_mu = (0.5 * torch.randn(*shape, generator=g) - 1 for _ in range(2))
        term = torch.rand(*shape, generator=g) < p
        done = term | (torch.rand(*shape, generator=g) < p)
        adv, vs = F.vtrace_advantage_estimate(gamma, log_pi, log_mu, v, nv, r, done, term, rho_t, c_t)
        gammas = 0.9 + 0.1 * torch.rand(*shape, generator=g)
        lmbdas = 0.8 + 0.2 * torch.rand(*shape, generator=g)
        ga, gt = F.vec_generalized_advantage_estimate(gammas, lmbdas, v, nv, r, done=done, terminated=term)
        r2g = F.reward2go(r, done, gamma)                                     # functional.py:1385-1460
        for k, t in dict(gamma=torch.tensor(gamma), rho_thresh=torch.tensor(rho_t), c_thresh=torch.tensor(c_t), v=v,
                         nv=nv, r=r, log_pi=log_pi, log_mu=log_mu, done=done, term=term, adv=adv, vs=vs,
                         gammas=gammas, lmbdas=lmbdas, gae_adv=ga, gae_tgt=gt, r2g=r2g).items():
            out[f"{name}/{k}"] = t.numpy()
    np.savez_compressed(OUT / "vtrace_golden.npz", **out)


def slice_cases():
    """slice_golden.npz: the reference's SliceSampler (samplers.py:1207-2300, imported unmodified under stub deps) on 1-d
    storages: the trajectory table it derives, the two random draws it makes and the index / truncated / mask it returns."""
    sys.path.insert(0, str(ROOT / "tests"))
    from _slice_cases import _live_slice_run, _slice_cases
    from oracle.ref_loader import reference_samplers

    R = reference_samplers()
    out = {}
    for name, (kwargs, data, length, max_size, last_cursor, batch_size) in _slice_cases().items():
        index, info, rec = _live_slice_run(R, kwargs, data, length, max_size, last_cursor, batch_size, seed=7)
        smp = R.mod.SliceSampler(**kwargs)
        st = R.make_storage(data, length, max_size, last_cursor)
        start, stop, lens = smp._get_stop_and_length(st)
        by_traj = kwargs.get("traj_key") is not None
        sig = data[kwargs["traj_key"]] if by_traj else data[("next", "done")]
        if kwargs.get("num_slices") is not None:
            num_slices, seq = kwargs["num_slices"], batch_size // kwargs["num_slices"]
        else:
            seq, num_slices = kwargs["slice_len"], batch_size // kwargs["slice_len"]
        cursor = -1 if last_cursor is None else int(last_cursor[-1] if isinstance(last_cursor, torch.Tensor) else last_cursor)
        out[f"{name}/meta"] = np.array([length, max_size, cursor, seq, num_slices, kwargs.get("strict_length", True),
                                        kwargs.get("pad_output", False), by_traj], dtype=np.int64)
        out[f"{name}/signal"] = sig.reshape(-1).numpy()
        out[f"{name}/stored_done"] = data.get(("next", "done"), torch.zeros(max_size, 1, dtype=torch.bool)).reshape(-1).numpy()
        out[f"{name}/table"] = np.stack([start[:, 0].numpy(), stop[:, 0].numpy(), lens.numpy()])
        out[f"{name}/traj_draw"] = rec["traj"].numpy()
        out[f"{name}/u"] = rec["u"].numpy()
        out[f"{name}/index"] = index.numpy()
        out[f"{name}/truncated"] = info[("next", "truncated")].reshape(-1).numpy()
        out[f"{name}/done"] = info[("next", "done")].reshape(-1).numpy()
        if ("collector", "mask") in info:
            out[f"{name}/mask"] = info[("collector", "mask")].numpy()
    np.savez_compressed(OUT / "slice_golden.npz", **out)


def pslice_cases():
    """pslice_golden.npz: the reference's PrioritizedSliceSampler (samplers.py:2575-3028, unmodified, on the compiled
    reference trees): the leaves it drew from, its uniform draws, and the slices / per-step weights it returned."""
    sys.path.insert(0, str(ROOT / "tests"))
    from _slice_cases import _live_pslice_run, _pslice_scenarios
    from oracle.ref_loader import reference_samplers

    R = reference_samplers()
    out = {}
    for name, (L, filled, S, T, seed) in _pslice_scenarios().items():
        done, sl, ml, draws = _live_pslice_run(R, L, filled, S, T, seed)
        out[f"{name}/meta"] = np.array([L, filled, S, T], dtype=np.int64)
        out[f"{name}/done"], out[f"{name}/sum_leaves"], out[f"{name}/min_leaves"] = done, sl, ml
        out[f"{name}/u"] = np.stack([d[0] for d in draws])
        out[f"{name}/index"] = np.stack([d[1] for d in draws])
        out[f"{name}/weight"] = np.stack([d[2] for d in draws])
    np.savez_compressed(OUT / "pslice_golden.npz", **out)


def per_cases():
    assert reference_ext("cpu") is not None
    out = {}
    for i, (N, filled, B, alpha, beta) in enumerate(
            [(16, 16, 32, 0.7, 0.5), (1000, 700, 256, 0.6, 0.4), (4097, 4097, 512, 0.6, 0.4),
             (100_000, 65_000, 1024, 0.6, 0.4)]):
        smp = po.OraclePrioritizedSampler(N, alpha, beta, tree_factory=reference_trees("cpu"))
        g = torch.Generator().manual_seed(200 + i)
        smp.mark_update(torch.arange(filled))
        pr = torch.rand(filled, generator=g) * 3
        ids = torch.randint(0, filled, (filled,), generator=g)      # with duplicates
        smp.update_priority(ids, pr)
        leaves = np.array(smp._sum_tree[np.arange(N)], dtype=np.float32)
        u = torch.rand(B, generator=g)
        idx, w = smp.sample(filled, B, u=u)
        k = f"case{i}"
        out[f"{k}/meta"] = np.array([N, filled, B], dtype=np.int64)
        out[f"{k}/ab"] = np.array([alpha, beta], dtype=np.float64)
        out[f"{k}/upd_index"] = ids.numpy()
        out[f"{k}/upd_priority"] = pr.numpy()
        out[f"{k}/leaves"] = leaves
        out[f"{k}/u"] = u.numpy()
        out[f"{k}/index"] = idx.numpy()
        out[f"{k}/weight"] = w.numpy()
        out[f"{k}/p_sum"] = np.float32(smp._sum_tree.query(0, filled))
        out[f"{k}/p_min"] = np.float32(smp._min_tree.query(0, filled))
    np.savez_compressed(OUT / "per_golden.npz", **out)


if __name__ == "__main__":
    gae_cases()
    td_cases()
    scan_cases()
    slice_cases()
    pslice_cases()
    per_cases()
    for f in sorted(OUT.glob("*.npz")):
        print(f.name, f.stat().st_size)
