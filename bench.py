#!/usr/bin/env python
"""bench.py -- the replay-and-advantage hot path on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic input (BASELINE.json configs[1] + [2]):

    1. batch = rb.sample(256)            PER sample on a 1M-capacity buffer of Atari transitions (pixels and
                                         next pixels u8[4,84,84], action i64, reward f32, done, terminated):
                                         torch.rand -> rlb_per_sample -> rlb_gather of all six leaves
    2. rb.update_priority(index, |td|)   (p+eps)^alpha, last-writer-wins scatter, touched-ancestor recompute
    3. adv, tgt = GAE([4096, 128])       gamma=.99, lmbda=.95, done/terminated ~ Bernoulli(.02)

`value` = (256 sampled + 4096*128 GAE) transitions per step / device time per step, whole job.  With N > 1
the buffer is sharded by capacity (one 1M shard per rank, SURVEY 8e), every rank draws 256 from its shard
and the 256*N global minibatch is assembled on every rank by the gather kernel itself (NVLink peer stores,
split-phase: a step returns the previous draw, so the transfer overlaps the rest of the step); every rank runs its
own GAE (weak scaling: per-GPU work is fixed).  N > 1 also runs BASELINE.json configs[3] and [4] ("c4", "c5": 1.25M /
6.25M slots per shard, 128 / 512 rows per rank) and reports them as extra keys of the same JSON line.

Timing: CUDA events on the launching stream around exactly K steps after W warm-ups, barrier +
synchronize on both sides, max over ranks.  --dump-outputs DIR (one GPU) writes what the timed path returned in its
last step as DIR/<name>.npy in float32 (float64 for int64 values): the sampled batch and the advantage / value target.
Every input is drawn from fixed seeds, so two builds run with the same arguments can be compared output for output.  Inputs are larger than L2 (the storage is 56 GB; the GAE inputs
rotate through a ring of sets larger than the 126 MB L2).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

ALPHA, BETA, GAMMA, LMBDA = 0.6, 0.4, 0.99, 0.95
CAPACITY, BATCH = 1_000_000, 256
GAE_ROWS, GAE_T = 4096, 128
ROW_BYTES = 2 * 4 * 84 * 84 + 8 + 4 + 1 + 1  # 56 462 B per Atari transition
TRANSITIONS_PER_STEP = BATCH + GAE_ROWS * GAE_T
METRIC = "transitions/sec sampled+GAE at 1M buffer / Atari frames"
WORKLOAD = "C2 PER sample+update B=256 @1M Atari transitions (56462 B/row) + C3 GAE [4096,128]"
N_BUFFERS = 4                    # receive slots of the pipelined sharded exchange
NVLINK_GBPS_PER_DIR = 900.0      # NVLink 5, per GPU per direction (B200_PROFILING.md)
GAE_SHAPES = ((4096, 128), (300, 500), (32, 512), (1, 512))  # C3 + benchmarks/test_objectives_benchmarks.py:122-153


def make_config(world: int) -> dict:
    """The workload description -- identical on both arms (ours / reference)."""
    return {"workload": WORKLOAD, "capacity_per_gpu": CAPACITY, "batch_per_gpu": BATCH,
            "gae_shape": [GAE_ROWS, GAE_T, 1], "alpha": ALPHA, "beta": BETA, "gamma": GAMMA, "lmbda": LMBDA,
            "arithmetic": "fp32 priorities / trees / GAE, byte-exact u8 row moves, int64 indices",
            "transitions_per_step_per_gpu": TRANSITIONS_PER_STEP,
            "parallelism": f"capacity-sharded x{world} (one 1M shard + 256 draws per GPU, global minibatch on every rank)"
                           if world > 1 else "single GPU",
            "l2": "inputs larger than L2: 56 GB storage per GPU with random rows; GAE inputs rotate through >160 MB"}


# ------------------------------------------------------------------------------------------- helpers
def peaks() -> tuple[float, str]:
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v == "Active"})
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    return rank, world, local


def timed(fn, steps: int, warmup: int, sync_all) -> float:
    """ms per step over exactly `steps` calls of fn(i), CUDA events on the current stream."""
    for i in range(warmup):
        fn(i)
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(warmup + i)
    e1.record()
    sync_all()
    return e0.elapsed_time(e1) / steps


# ------------------------------------------------------------------------------------------- our arm
def build_buffer(dev, capacity: int, seed: int):
    """1M-capacity HBM-resident PER buffer of Atari-shaped transitions, filled with synthetic data."""
    from rl_b200.data import LazyTensorStorage, TensorDict, TensorDictPrioritizedReplayBuffer

    g = torch.Generator(device=dev).manual_seed(seed)
    rb = TensorDictPrioritizedReplayBuffer(alpha=ALPHA, beta=BETA, storage=LazyTensorStorage(capacity, device=dev),
                                           batch_size=BATCH, generator=g)
    chunk = 50_000
    for lo in range(0, capacity, chunk):
        n = min(chunk, capacity - lo)
        td = TensorDict({
            "pixels": torch.randint(0, 256, (n, 4, 84, 84), dtype=torch.uint8, device=dev, generator=g),
            "action": torch.randint(0, 18, (n, 1), device=dev, generator=g),
            "next": {"pixels": torch.randint(0, 256, (n, 4, 84, 84), dtype=torch.uint8, device=dev, generator=g),
                     "reward": torch.randn(n, device=dev, generator=g),
                     "done": torch.rand(n, 1, device=dev, generator=g) < 0.01,
                     "terminated": torch.rand(n, 1, device=dev, generator=g) < 0.01},
            "td_error": torch.rand(n, device=dev, generator=g),
        }, [n])
        rb.extend(td)
    return rb, g


def gae_ring(dev, rows: int, T: int, g, min_bytes: int = 160 << 20):
    """Input sets for GAE whose total footprint exceeds L2 so that every call reads cold data."""
    per = rows * T * 14
    n = max(2, -(-min_bytes // per))
    n = -(-n // N_BUFFERS) * N_BUFFERS  # the sharded buffer's receive slots rotate with the ring slot
    ring = []
    for _ in range(n):
        v, nv, r = (torch.randn(rows, T, 1, device=dev, generator=g) for _ in range(3))
        term = torch.rand(rows, T, 1, device=dev, generator=g) < 0.02
        done = term | (torch.rand(rows, T, 1, device=dev, generator=g) < 0.02)
        ring.append((v, nv, r, done, term))
    return ring


def kernel_roofline(dev, rb, ring, hbm_peak: float, peak_src: str) -> dict:
    """Average launch duration of the dominant kernel (the gather: 28.9 MB/launch vs 11.5 MB for GAE), timed
    with CUDA events around a CUDA-graph replay of back-to-back launches on cold rows (no host in the loop)."""
    from rl_b200 import ops

    be = ops.backend()
    st = rb.storage
    n_launch = 20
    g = torch.Generator(device=dev).manual_seed(123)
    idxs = [torch.randint(0, len(st), (BATCH,), device=dev, generator=g) for _ in range(n_launch)]
    stream = torch.cuda.Stream(dev)
    out = {}
    with torch.cuda.stream(stream):
        # warm-up outside capture
        for ix in idxs[:3]:
            be.gather(st._leaves, ix, len(st))
        stream.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            keep = [be.gather(st._leaves, ix, len(st)) for ix in idxs]
        ms = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            graph.replay()
            e1.record(stream)
            stream.synchronize()
            ms.append(e0.elapsed_time(e1) / n_launch)
        del keep
        us = sorted(ms)[len(ms) // 2] * 1e3
        row_bytes = sum(l[0].numel() * l.element_size() for l in st._leaves)  # every stored leaf, per transition
        alg = BATCH * row_bytes * 2 + BATCH * 8
        traffic = None
        tf = ROOT / "profiles" / "traffic_r1.json"
        if tf.exists():  # from the committed `ncu --set full` capture (profiles/ncu_full_r1.csv), per launch
            tj = json.loads(tf.read_text())["gather_kernel_B256"]
            traffic = tj["dram_read_bytes"] + tj["dram_write_bytes"]
        out = {"bound": "hbm", "kernel": f"gather_kernel<gather> (rlb_gather, {len(st._leaves)} leaves, B=256)",
               "row_bytes": row_bytes,
               "achieved": round(alg / us / 1e3, 1), "peak": hbm_peak, "unit": "GB/s",
               "frac": round(alg / us / 1e3 / hbm_peak, 4), "traffic": traffic, "peak_source": peak_src,
               "algorithmic_bytes": alg, "us_per_launch": round(us, 3)}
        # the same kernel over a batch sweep (graph-replayed launches on cold rows): fixed cost + streaming rate
        sweep = {}
        for bb, reps in ((1024, 8), (4096, 4), (16384, 2)):
            idx_b = [torch.randint(0, len(st), (bb,), device=dev, generator=g) for _ in range(reps)]
            be.gather(st._leaves, idx_b[0], len(st))
            stream.synchronize()
            gb = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gb, stream=stream):
                keep = [be.gather(st._leaves, ix, len(st)) for ix in idx_b]
            gb.replay()
            stream.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            gb.replay()
            e1.record(stream)
            stream.synchronize()
            del keep, gb
            us_b = e0.elapsed_time(e1) * 1e3 / reps
            alg_b = bb * row_bytes * 2 + bb * 8
            sweep[f"B{bb}"] = {"achieved": round(alg_b / us_b / 1e3, 1), "frac": round(alg_b / us_b / 1e3 / hbm_peak, 4),
                               "us_per_launch": round(us_b, 1)}
        out["batch_sweep"] = sweep
        out["steady_state_B16384"] = sweep["B16384"]
        # GAE kernel, same method
        v, nv, r, d, t = ring[0]
        graph2 = torch.cuda.CUDAGraph()
        d8 = [(x[3].view(torch.uint8), x[4].view(torch.uint8)) for x in ring]
        for i in range(2):
            be.gae(ring[i][0], ring[i][1], ring[i][2], d8[i][0], d8[i][1], GAMMA, GAMMA * LMBDA, GAE_ROWS, GAE_T, 1)
        stream.synchronize()
        with torch.cuda.graph(graph2, stream=stream):
            keep = [be.gae(x[0], x[1], x[2], dd[0], dd[1], GAMMA, GAMMA * LMBDA, GAE_ROWS, GAE_T, 1)
                    for x, dd in zip(ring, d8)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        graph2.replay()
        stream.synchronize()
        e0.record(stream)
        graph2.replay()
        e1.record(stream)
        stream.synchronize()
        us_g = e0.elapsed_time(e1) * 1e3 / len(ring)
        alg_g = GAE_ROWS * GAE_T * 22
        out["gae_kernel"] = {"achieved": round(alg_g / us_g / 1e3, 1), "frac": round(alg_g / us_g / 1e3 / hbm_peak, 4),
                             "us_per_launch": round(us_g, 3), "algorithmic_bytes": alg_g}
        del keep
    return out


def write_path_probe(dev, rb, g, hbm_peak: float) -> dict | None:
    """SURVEY 8(f)-1 beside the headline: rb.extend of 1024 Atari transitions (rows + default priorities, one rlb_extend
    launch), ten consecutive writer batches captured in one CUDA graph and replayed.  Never fatal to the bench."""
    try:
        from rl_b200.data import TensorDict

        n = 1024
        td = TensorDict({
            "pixels": torch.randint(0, 256, (n, 4, 84, 84), dtype=torch.uint8, device=dev, generator=g),
            "action": torch.randint(0, 18, (n, 1), device=dev, generator=g),
            "next": {"pixels": torch.randint(0, 256, (n, 4, 84, 84), dtype=torch.uint8, device=dev, generator=g),
                     "reward": torch.randn(n, device=dev, generator=g),
                     "done": torch.zeros(n, 1, dtype=torch.bool, device=dev),
                     "terminated": torch.zeros(n, 1, dtype=torch.bool, device=dev)},
            "td_error": torch.rand(n, device=dev, generator=g),
        }, [n])
        row = sum(l[0].numel() * l.element_size() for l in rb.storage._leaves if l is not None)
        rb.extend(td, update_priority=False)
        torch.cuda.synchronize(dev)
        side = torch.cuda.Stream(dev)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(gr, stream=side):
                for _ in range(10):
                    rb.extend(td, update_priority=False)
        torch.cuda.synchronize(dev)
        for _ in range(3):
            gr.replay()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        a.record()
        for _ in range(20):
            gr.replay()
        b.record()
        torch.cuda.synchronize(dev)
        us = a.elapsed_time(b) * 1e3 / 200
        gbs = 2 * n * row / us / 1e3
        return {"extend_n": n, "extend_us": round(us, 2), "extend_GBps": round(gbs, 1), "extend_frac_of_hbm": round(gbs / hbm_peak, 3),
                "extend_transitions_per_s": round(n / (us * 1e-6), 1), "row_bytes": row}
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:200]}


def framestack_probe(dev, g, hbm_peak: float) -> dict:
    """SURVEY 8(f)-1, second half: the de-duplicated frame-stack storage next to the materialised one.  8 environment
    streams of 84x84 frames, 4-stacks, 262144 transitions (pool 2.3 GB, far beyond L2); a B=256 tensor-index read rebuilds
    both stacks inside the gather launch.  Reports pixel bytes per stored transition and the read / write times.  Never
    fatal to the bench."""
    try:
        from rl_b200.data import FrameStackStorage, LazyTensorStorage, TensorDict

        E, T, k, cap = 8, 512, 4, 262144
        out = {}
        stores = {"dedup": FrameStackStorage(cap, n_envs=E, device=dev, min_episode_length=64),
                  "dedup_views": FrameStackStorage(cap, n_envs=E, device=dev, min_episode_length=64, materialize=False),
                  "materialised": LazyTensorStorage(cap, device=dev)}
        tail = torch.randint(0, 256, (k, E, 84, 84), dtype=torch.uint8, device=dev, generator=g)
        cursor, batch = 0, None
        for _ in range(cap // (E * T)):
            frames = torch.cat([tail, torch.randint(0, 256, (T, E, 84, 84), dtype=torch.uint8, device=dev, generator=g)])
            tail = frames[-k:]
            win = frames.unfold(0, k + 1, 1).permute(1, 0, 4, 2, 3)            # [E, T, k + 1, 84, 84] windows of the stream
            n = E * T
            batch = TensorDict({"pixels": win[:, :, :k].reshape(n, k, 84, 84), "action": torch.zeros(n, 1, dtype=torch.int64, device=dev),
                                "next": {"pixels": win[:, :, 1:].reshape(n, k, 84, 84), "reward": torch.zeros(n, device=dev),
                                         "done": torch.zeros(n, 1, dtype=torch.bool, device=dev)}}, [n])
            slots = torch.arange(cursor, cursor + n, device=dev)
            for st in stores.values():
                st.set(slots, batch)
            cursor += n
        idx = [torch.randint(0, cap, (BATCH,), device=dev, generator=g) for _ in range(20)]
        a, b = stores["dedup"].get(idx[0]), stores["materialised"].get(idx[0])
        c = stores["dedup_views"].get(idx[0])
        same = all(torch.equal(a.get(key), b.get(key)) and torch.equal(c.get(key), b.get(key))
                   for key in ("pixels", ("next", "pixels")))
        for st in stores.values():
            if hasattr(st, "check_index_status"):
                st.check_index_status()
        out["batches_equal_materialised_storage"] = bool(same)
        frame = 84 * 84
        out["pixel_bytes_per_transition"] = {"dedup": round(stores["dedup"].frame_bytes_per_transition, 1),
                                             "materialised": 2 * k * frame}
        for name, st in stores.items():
            us = graph_us([(lambda ix=ix, st=st: st.get(ix)) for ix in idx], dev)
            moved = BATCH * frame * ((k + 1) * 2 if name == "dedup_views" else (k + 1) + 2 * k if name == "dedup" else 4 * k)
            out[f"get_B{BATCH}_{name}_us"] = round(us, 2)
            out[f"get_B{BATCH}_{name}_unique_GBps"] = round(moved / us / 1e3, 1)
        writes = [(lambda st=st: st.set(torch.arange(0, E * T, device=dev), batch)) for st in (stores["dedup"],)] * 4
        out[f"set_n{E * T}_dedup_us"] = round(graph_us(writes, dev), 2)
        writes = [(lambda: stores["materialised"].set(torch.arange(0, E * T, device=dev), batch))] * 4
        out[f"set_n{E * T}_materialised_us"] = round(graph_us(writes, dev), 2)
        out["note"] = ("unique_GBps counts every distinct byte once (dedup reads k + 1 frames per transition and writes "
                       "2 k, or k + 1 as overlapping views); hbm peak %.0f GB/s" % hbm_peak)
        return out
    except Exception as e:  # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def steps_per_graph(k: int) -> int:
    """Consecutive steps captured into ONE graph.  A graph replay costs ~8 us on its own (torch refreshes the Philox
    seed / offset of the registered generator with two small fill kernels, then the launch itself), so a training loop
    that captures a few steps at a time pays it once per group; the timed region still runs EXACTLY `k` steps."""
    return group_plan(k, 1)[0]


def group_plan(k: int, quantum: int) -> tuple[int, int]:
    """(steps per graph, remainder) for a timed region of EXACTLY k steps: the largest group size <= 20 that is a multiple
    of `quantum` (the receive-slot count of the pipelined exchange; 1 on one GPU) and divides k; when only tiny groups
    divide k (a prime step count), groups of up to 20 plus ONE shorter graph holding the k % spg left-over steps."""
    top = max(quantum, min(20, k) // quantum * quantum)
    for spg in range(top, 0, -quantum):
        if k % spg == 0 and spg >= min(8, top):
            return spg, 0
    return top, k % top


def timed_groups(graphs, spg: int, steps: int, warmup: int, sync_all, tail=None) -> float:
    """ms per STEP over exactly `steps` steps, issued as steps // spg replays of graphs holding spg steps each plus, when
    spg does not divide `steps`, one replay of `tail` (a graph of the steps % spg left-over steps)."""
    n_g = len(graphs)
    launches, warm = steps // spg, -(-warmup // spg)
    rem = steps % spg
    if not rem:
        return timed(lambda i: graphs[i % n_g](), launches, warm, sync_all) / spg
    if tail is None:
        raise RuntimeError(f"{steps} steps do not divide into groups of {spg} and no tail graph was given")
    calls = launches + 1
    # (timed() numbers its calls warm, warm + 1, ...: the last one of the timed region is the tail)
    return timed(lambda i: (graphs[i % n_g]() if i - warm < launches else tail()), calls, warm, sync_all) * calls / steps


def last_timed_graph(graphs, spg: int, steps: int, warmup: int, tail=None):
    """The graph that timed_groups(graphs, spg, steps, warmup, ..., tail) replayed last (same call numbering)."""
    if steps % spg:
        return tail
    return graphs[(-(-warmup // spg) + steps // spg - 1) % len(graphs)]


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, batch, adv, target) -> dict:
    """Write one step's results as <name>.npy: float32, or float64 where an int64 value would not fit float32."""
    import numpy as np

    arrays = {"advantage": adv, "value_target": target}
    for k, v in batch.items(True, True):
        arrays["sample." + (k if isinstance(k, str) else ".".join(k))] = v
    host = {n: v.detach().cpu().numpy() for n, v in arrays.items()}
    host = {n: a.astype(np.float64 if a.dtype == np.int64 else np.float32) for n, a in host.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for n, a in host.items():
        np.save(d / f"{n}.npy", a)
    return {"dir": str(d), "arrays": sorted(host), "bytes": total}


def graph_us(fn_list, dev, reps: int = 5) -> float:
    """Median device time (us) of ONE call, measured as a CUDA-graph replay of all callables in `fn_list` back to back
    on one stream (CUDA events around the replay; no host in the loop)."""
    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        fn_list[0]()
        stream.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=stream):
            keep = [fn() for fn in fn_list]
        gr.replay()
        stream.synchronize()
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            gr.replay()
            e1.record(stream)
            stream.synchronize()
            ms.append(e0.elapsed_time(e1))
        del keep, gr
    return sorted(ms)[len(ms) // 2] * 1e3 / len(fn_list)


def component_times(dev, rb, ring8, td_err, gs, be) -> dict:
    """Graph-replayed device time of each component of the step on its own (20 calls back to back): the numbers the
    per-component CPU ratios are formed from -- the headline is dominated by GAE elements, these are not."""
    g = torch.Generator(device=dev).manual_seed(321)
    n = 20
    out = {}
    gen = rb.sampler._rng
    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        rb.sample()
        stream.synchronize()
        gr = torch.cuda.CUDAGraph()
        gr.register_generator_state(gen)
        with torch.cuda.graph(gr, stream=stream):
            keep = [rb.sample() for _ in range(n)]
        gr.replay()
        stream.synchronize()
        ms = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            gr.replay()
            e1.record(stream)
            stream.synchronize()
            ms.append(e0.elapsed_time(e1))
        del keep, gr
    out["sample_us"] = round(sorted(ms)[2] * 1e3 / n, 2)
    idx = [torch.randint(0, CAPACITY, (BATCH,), device=dev, generator=g) for _ in range(n)]
    out["update_priority_us"] = round(graph_us([(lambda ix=ix: rb.update_priority(ix, td_err)) for ix in idx], dev), 2)
    out["gae_us"] = round(graph_us([(lambda x=x: be.gae(x[0], x[1], x[2], x[3], x[4], gs[0], gs[1], GAE_ROWS, GAE_T, 1))
                                    for x in ring8[:n]], dev), 2)
    out["sample_transitions_per_s"] = round(BATCH / (out["sample_us"] * 1e-6), 1)
    out["update_transitions_per_s"] = round(BATCH / (out["update_priority_us"] * 1e-6), 1)
    out["gae_transitions_per_s"] = round(GAE_ROWS * GAE_T / (out["gae_us"] * 1e-6), 1)
    out["method"] = "CUDA-graph replay of 20 public-API calls back to back, CUDA events, median of 5"
    return out


def gae_shape_sweep(dev, be, hbm_peak: float) -> dict:
    """The GAE kernel at C3 and at the reference benchmark's own shapes (few rows / long T), graph-replayed on inputs
    that rotate through more than L2."""
    g = torch.Generator(device=dev).manual_seed(77)
    out = {}
    for rows, T, *rest in GAE_SHAPES + ((1024, 128, 4),):
        F = rest[0] if rest else 1
        per = rows * T * F * 14
        n = int(min(64, max(4, (160 << 20) // per)))
        sets = []
        for _ in range(n):
            v, nv, r = (torch.randn(rows, T, F, device=dev, generator=g) for _ in range(3))
            term = torch.rand(rows, T, F, device=dev, generator=g) < 0.02
            done = term | (torch.rand(rows, T, F, device=dev, generator=g) < 0.02)
            sets.append((v, nv, r, done.view(torch.uint8), term.view(torch.uint8)))
        us = graph_us([(lambda x=x: be.gae(x[0], x[1], x[2], x[3], x[4], GAMMA, GAMMA * LMBDA, rows, T, F)) for x in sets], dev)
        alg = rows * T * F * 22
        out[f"{rows}x{T}" + (f"x{F}" if F > 1 else "")] = {"us_per_launch": round(us, 3), "achieved": round(alg / us / 1e3, 1),
                              "frac": round(alg / us / 1e3 / hbm_peak, 4), "algorithmic_bytes": alg}
    return out


def reference_gpu_kernels(dev, rb, ring, td_err) -> dict:
    """BASELINE LEG (SURVEY 8d "kernel to beat"): the reference's OWN GPU paths timed on the same box, same inputs,
    same method (graph-replayed back-to-back calls, cold rows): aten::index per leaf (storages.py:1260-1263), the
    reference CUDA segment tree (csrc/cuda_segment_tree.cu, compiled unmodified into oracle/_ref/cuda) and its
    conv-based vec GAE on cuda (functional.py:211-267).  Never fatal to the bench."""
    out = {}
    try:
        st = rb.storage
        g = torch.Generator(device=dev).manual_seed(123)
        from rl_b200 import ops

        be = ops.backend()
        for bb, reps in ((256, 20), (1024, 8), (16384, 2)):
            idxs = [torch.randint(0, len(st), (bb,), device=dev, generator=g) for _ in range(reps)]
            ref_us = graph_us([(lambda ix=ix: [leaf[ix] for leaf in st._leaves]) for ix in idxs], dev)
            our_us = graph_us([(lambda ix=ix: be.gather(st._leaves, ix, len(st))) for ix in idxs], dev)
            out[f"gather_B{bb}"] = {"aten_index_us": round(ref_us, 2), "rlb_gather_us": round(our_us, 2),
                                    "speedup": round(ref_us / our_us, 2), "launches_ref": len(st._leaves), "launches_ours": 1}
    except Exception as e:  # noqa: BLE001
        out["gather_error"] = f"{type(e).__name__}: {e}"[:200]
    try:
        from oracle import gae_torch

        v, nv, r, d, t = ring[0]
        gm, lm = torch.tensor(GAMMA, device=dev), torch.tensor(LMBDA, device=dev)
        with torch.no_grad():
            for _ in range(3):
                gae_torch.vec_gae(gm, lm, v, nv, r, d, t)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(20):
                x = ring[i % len(ring)]
                gae_torch.vec_gae(gm, lm, x[0], x[1], x[2], x[3], x[4])
            e1.record()
            torch.cuda.synchronize(dev)
        ref_us = e0.elapsed_time(e1) * 1e3 / 20
        from rl_b200 import ops

        be = ops.backend()
        our_us = graph_us([(lambda x=x: be.gae(x[0], x[1], x[2], x[3].view(torch.uint8), x[4].view(torch.uint8), GAMMA,
                                               GAMMA * LMBDA, GAE_ROWS, GAE_T, 1)) for x in ring[:20]], dev)
        out["gae_4096x128"] = {"reference_vec_gae_cuda_us": round(ref_us, 1), "rlb_gae_us": round(our_us, 2),
                               "speedup": round(ref_us / our_us, 1),
                               "note": "reference = its conv1d path as torch ops on cuda (eager: it has host syncs and cannot be captured)"}
    except Exception as e:  # noqa: BLE001
        out["gae_error"] = f"{type(e).__name__}: {e}"[:200]
    try:
        from oracle.ref_loader import reference_ext

        ext = reference_ext("cuda")
        if ext is None or not hasattr(ext, "CudaSumSegmentTreeFp32"):
            raise RuntimeError("oracle/_ref/cuda/_torchrl.so not available")
        smp = rb.sampler
        rs, rm = ext.CudaSumSegmentTreeFp32(CAPACITY, dev), ext.CudaMinSegmentTreeFp32(CAPACITY, dev)
        leaves = smp._sum_tree.dump_leaves()
        all_idx = torch.arange(CAPACITY, device=dev)
        rs.update(all_idx, leaves)
        rm.update(all_idx, leaves)
        g = torch.Generator(device=dev).manual_seed(5)
        idx = [torch.randint(0, CAPACITY, (BATCH,), device=dev, generator=g) for _ in range(10)]
        val = torch.rand(BATCH, device=dev, generator=g)
        mass = torch.rand(BATCH, device=dev, generator=g) * rs.query(0, CAPACITY)

        def t_eager(fn, n=10):
            fn(0)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n):
                fn(i)
            e1.record()
            torch.cuda.synchronize(dev)
            return e0.elapsed_time(e1) * 1e3 / n

        def ref_update(i):
            rs.update(idx[i % 10], val)
            rm.update(idx[i % 10], val)

        ref_upd = t_eager(ref_update)
        ref_scan = t_eager(lambda i: rs.scan_lower_bound(mass))
        from rl_b200 import ops

        be = ops.backend()
        ws = smp._tree_workspace(BATCH)
        our_upd = graph_us([(lambda ix=ix: be.tree_update(smp._sum_tree.values, smp._min_tree.values, smp._sum_tree.capacity,
                                                         ix, val, ws, 1)) for ix in idx], dev)
        our_scan = graph_us([(lambda: be.tree_scan_lower_bound(smp._sum_tree.values, CAPACITY, smp._sum_tree.capacity, mass))
                             for _ in range(10)], dev)
        out["tree_B256"] = {"reference_cuda_update_us": round(ref_upd, 1), "rlb_tree_update_us": round(our_upd, 2),
                            "update_speedup": round(ref_upd / our_upd, 1),
                            "reference_cuda_scan_lower_bound_us": round(ref_scan, 1),
                            "rlb_tree_scan_lower_bound_us": round(our_scan, 2), "scan_speedup": round(ref_scan / our_scan, 1),
                            "note": "reference CUDA tree = <<<1,1>>> leaf loop + one full-level launch per level per tree (eager; device time by CUDA events)"}
        # restore our leaves' ancestors (tree_update above wrote random values into the product trees)
        smp._sum_tree.load_leaves(leaves)
        ml = leaves.clone()
        smp._min_tree.load_leaves(torch.where(all_idx < len(rb.storage), ml, torch.full_like(ml, torch.finfo(ml.dtype).max)))
    except Exception as e:  # noqa: BLE001
        out["tree_error"] = f"{type(e).__name__}: {e}"[:200]
    return out


def run_ours(args) -> dict:
    rank, world, local = dist_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
        try:
            result = run_distributed(args, dev, rank, world)
        finally:
            pass
        dist.barrier()
        dist.destroy_process_group()
        return result
    return run_single(args, dev)


def run_single(args, dev) -> dict:
    from rl_b200 import ops
    from rl_b200.graphs import CudaGraphStep

    be = ops.backend()
    rb, g = build_buffer(dev, CAPACITY, seed=0)
    ring = gae_ring(dev, GAE_ROWS, GAE_T, g)
    ring8 = [(v, nv, r, d.view(torch.uint8), t.view(torch.uint8)) for v, nv, r, d, t in ring]
    R = len(ring)
    td_err = torch.rand(BATCH, device=dev, generator=g)
    gs = (float(torch.tensor(GAMMA)), float(torch.tensor(GAMMA) * torch.tensor(LMBDA)))

    def sync_all():
        torch.cuda.synchronize()

    side_gae, side_upd = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    smp = rb.sampler
    smp.record_index_event = True
    smp.predraw = os.environ.get("RLB_BENCH_PREDRAW", "0") != "0"

    def make_step(slot: int):
        v, nv, r, d8, t8 = ring8[slot]

        def step():
            # three independent chains of the same step run on three streams (fork / join with events):
            #   main      rand -> per_sample -> gather
            #   side_upd  update_priority(index): needs the sampled indices only, overlaps the gather
            #   side_gae  GAE of this step's rollout: independent of the replay path
            main = torch.cuda.current_stream(dev)
            side_gae.wait_stream(main)
            with torch.cuda.stream(side_gae):
                a, tg = be.gae(v, nv, r, d8, t8, gs[0], gs[1], GAE_ROWS, GAE_T, 1)
            batch = rb.sample()
            index = batch.get("index")
            side_upd.wait_event(smp.index_ready)
            with torch.cuda.stream(side_upd):
                rb.update_priority(index, td_err)    # fused pow + tree write-back
            main.wait_stream(side_upd)
            main.wait_stream(side_gae)
            return batch, a, tg

        return step

    def make_eager_step(slot: int):
        v, nv, r, d8, t8 = ring8[slot]

        def step():  # the plain single-stream call sequence a Python training loop would issue
            batch = rb.sample()
            rb.update_priority(batch.get("index"), td_err)
            a, tg = be.gae(v, nv, r, d8, t8, gs[0], gs[1], GAE_ROWS, GAE_T, 1)
            return batch, a, tg

        return step

    steps = [make_step(i) for i in range(R)]
    eager_steps = [make_eager_step(i) for i in range(R)]

    # ---- (1) eager: every call goes through the Python API
    clocks = ClockSampler(dev.index or 0)
    ms_eager = timed(lambda i: eager_steps[i % R](), args.steps, args.warmup, sync_all)

    # ---- (2) the same steps captured into CUDA graphs -- `spg` consecutive steps (each with its own GAE input set) per
    # graph -- and replayed
    graphs, graph_err, ms_graph, dumped = None, None, None, None
    spg, rem = group_plan(args.steps, 1)
    try:
        gen = rb.sampler._rng
        n_groups = max(1, min(3, R // spg))
        groups = [[steps[(gi * spg + k) % R] for k in range(spg)] for gi in range(n_groups)]
        graphs = [CudaGraphStep((lambda grp=grp: [st() for st in grp]), generators=[gen], warmup=1) for grp in groups]
        tail = CudaGraphStep((lambda: [steps[k % R]() for k in range(rem)]), generators=[gen], warmup=1) if rem else None
        ms_graph = timed_groups(graphs, spg, args.steps, args.warmup, sync_all, tail)
        if args.dump_outputs:
            dumped = dump_outputs(args.dump_outputs,
                                  *last_timed_graph(graphs, spg, args.steps, args.warmup, tail).outputs[-1])
        # a longer replay run of the same graphs (the driver's --steps 20 makes the timed region < 1 ms)
        ms_graph_long = timed_groups(graphs, spg, max(args.steps, 400) // spg * spg, 8, sync_all)
        # and the one-step-per-graph figure, for comparison with round 1
        single = [CudaGraphStep(st, generators=[gen], warmup=1) for st in steps[:8]]
        ms_graph_single = timed(lambda i: single[i % 8](), 200, 8, sync_all)
        del single
    except Exception as err:
        import traceback

        graph_err = f"{type(err).__name__}: {err}"[:300]
        print(f"[bench] CUDA-graph path failed, falling back to eager: {graph_err}\n"
              + "".join(traceback.format_exc().splitlines(True)[-6:]), file=sys.stderr, flush=True)
        graphs, ms_graph, ms_graph_long, ms_graph_single = None, None, None, None
        if args.dump_outputs:
            raise RuntimeError("--dump-outputs: the CUDA-graph path failed, no outputs of the timed steps to write")
        torch.cuda.synchronize()
        fresh = torch.Generator(device=dev).manual_seed(4242)
        rb.set_rng(fresh)
        g = fresh
    clk = clocks.stop()

    # ---- sub-metrics (eager, same method)
    ms_sample = timed(lambda i: rb.sample(), args.steps, 3, sync_all)
    idx_pool = [torch.randint(0, CAPACITY, (BATCH,), device=dev, generator=g) for _ in range(8)]
    ms_update = timed(lambda i: rb.update_priority(idx_pool[i % 8], td_err), args.steps, 3, sync_all)

    def gae_only(i):
        v, nv, r, d8, t8 = ring8[i % R]
        be.gae(v, nv, r, d8, t8, gs[0], gs[1], GAE_ROWS, GAE_T, 1)

    ms_gae = timed(gae_only, args.steps, 3, sync_all)

    ms_e2e, h2d, d2h, n_lanes = e2e_run(args, dev, rb, ring, td_err, gs, be, sync_all, slice(None), 3)

    hbm_peak, peak_src = peaks()
    roof = kernel_roofline(dev, rb, ring, hbm_peak, peak_src)
    try:
        roof["gae_shapes"] = gae_shape_sweep(dev, be, hbm_peak)
    except Exception as e:  # noqa: BLE001
        roof["gae_shapes"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    try:
        comp = component_times(dev, rb, ring8, td_err, gs, be)
    except Exception as e:  # noqa: BLE001
        comp = {"error": f"{type(e).__name__}: {e}"[:200]}
    write_path = write_path_probe(dev, rb, g, hbm_peak)
    if isinstance(write_path, dict):
        write_path["framestack"] = framestack_probe(dev, g, hbm_peak)
    ref_gpu = reference_gpu_kernels(dev, rb, ring, td_err)
    cpu = cpu_baseline_run(steps=None)
    if "error" not in comp and cpu.get("phases_ms"):
        ph = cpu["phases_ms"]
        comp["vs_cpu"] = {"sample(tree+gather)": round((ph["tree_sample"] + ph["gather"]) * 1e3 / comp["sample_us"], 1),
                          "update_priority": round(ph["tree_update"] * 1e3 / comp["update_priority_us"], 1),
                          "gae": round(ph["gae"] * 1e3 / comp["gae_us"], 1)}
    ms = ms_graph if ms_graph is not None else ms_eager
    n_leaves = len(rb.storage._leaves)
    cfg = make_config(1)
    detail = {"n_leaves": n_leaves, "steps_per_graph": spg if ms_graph is not None else None,
              "launch": (f"cuda_graph replay of the public-API step, {spg} consecutive steps per graph"
                         if ms_graph is not None else "eager python API")}
    result = {
        "metric": METRIC, "value": round(TRANSITIONS_PER_STEP / (ms * 1e-3), 1), "unit": "transitions/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 5), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "impl_detail": detail,
        "e2e": {"value": round(TRANSITIONS_PER_STEP / (ms_e2e * 1e-3), 1), "unit": "transitions/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": round(ms_e2e, 5),
                "note": f"eager python API, pinned host buffers, {n_lanes} lane(s): with several lanes D2H overlaps the next steps' H2D + compute"},
        "gpu_launches": 4 * args.steps,  # ours per step: per_sample, gather, update, gae (torch.rand is torch's)
        "breakdown": {"eager_ms_per_step": round(ms_eager, 5),
                      "graph_ms_per_step": None if ms_graph is None else round(ms_graph, 5),
                      "graph_ms_per_step_long_run": None if ms_graph_long is None else round(ms_graph_long, 5),
                      "graph_ms_per_step_one_step_per_graph": None if ms_graph_single is None else round(ms_graph_single, 5),
                      "graph_error": graph_err,
                      "eager_value": round(TRANSITIONS_PER_STEP / (ms_eager * 1e-3), 1),
                      "eager_sample_us": round(ms_sample * 1e3, 2), "eager_update_priority_us": round(ms_update * 1e3, 2),
                      "eager_gae_us": round(ms_gae * 1e3, 2),
                      "components_graph_replayed": comp,
                      "write_path": write_path,
                      "reference_gpu": ref_gpu},
        "clocks": clk, "roofline": roof, "cpu_baseline": cpu,
    }
    if dumped is not None:
        result["dumped_outputs"] = dumped
    return result


def e2e_run(args, dev, rb, ring, td_err, gs, be, sync_all, own, n_lanes):
    """End to end with HOST buffers: H2D of the step's inputs and D2H of the step's results every step.  Independent
    lanes (stream + pinned buffers + device staging) rotate so that one step's D2H overlaps the next steps' H2D and
    compute (PCIe is full duplex); every step still synchronises on its own results."""
    R = len(ring)
    pin = lambda t: t.cpu().pin_memory()
    sample0 = rb.sample()
    out_keys = list(sample0.keys(True, True))
    lanes = []
    for lane in range(n_lanes):
        s = torch.cuda.Stream(dev)
        host_in = tuple(pin(x) for x in ring[lane % R])
        lanes.append({
            "stream": s, "host_in": host_in, "host_td": pin(td_err),
            "dev_in": [torch.empty_like(x) for x in ring[lane % R]], "dev_td": torch.empty_like(td_err),
            "host_out": {k: torch.empty(sample0.get(k)[own].shape, dtype=sample0.get(k).dtype).pin_memory()
                         for k in out_keys},
            "host_adv": torch.empty(GAE_ROWS, GAE_T, 1).pin_memory(), "host_tgt": torch.empty(GAE_ROWS, GAE_T, 1).pin_memory(),
            "done": torch.cuda.Event(),
        })
    h2d = sum(x.numel() * x.element_size() for x in lanes[0]["host_in"]) + td_err.numel() * 4
    d2h = sum(v.numel() * v.element_size() for v in lanes[0]["host_out"].values()) + 2 * GAE_ROWS * GAE_T * 4

    def e2e_body(L):
        for dst, src in zip(L["dev_in"], L["host_in"]):
            dst.copy_(src, non_blocking=True)
        L["dev_td"].copy_(L["host_td"], non_blocking=True)
        batch = rb.sample()
        rb.update_priority(batch.get("index"), L["dev_td"])
        di = L["dev_in"]
        a, tg = be.gae(di[0], di[1], di[2], di[3].view(torch.uint8), di[4].view(torch.uint8), gs[0], gs[1],
                       GAE_ROWS, GAE_T, 1)
        for k, hv in L["host_out"].items():
            hv.copy_(batch.get(k)[own], non_blocking=True)
        L["host_adv"].copy_(a, non_blocking=True)
        L["host_tgt"].copy_(tg, non_blocking=True)

    def e2e_step(i: int):
        L = lanes[i % n_lanes]
        L["done"].synchronize()            # the caller consumed this lane's previous results
        with torch.cuda.stream(L["stream"]):
            e2e_body(L)
            L["done"].record()

    for i in range(args.warmup):
        e2e_step(i)
    sync_all()
    cur = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(cur)
    for L in lanes:
        L["stream"].wait_event(e0)
    for i in range(args.steps):
        e2e_step(args.warmup + i)
    for L in lanes:
        cur.wait_stream(L["stream"])
    e1.record(cur)
    sync_all()
    return e0.elapsed_time(e1) / args.steps, h2d, d2h, n_lanes


# ------------------------------------------------------------------------------------------- N > 1
def make_rows(kind: str, n: int, dev, g):
    from rl_b200.data import TensorDict

    if kind == "atari":     # DQN-shaped Atari transition: 56 462 B + td_error
        return TensorDict({
            "pixels": torch.randint(0, 256, (n, 4, 84, 84), dtype=torch.uint8, device=dev, generator=g),
            "action": torch.randint(0, 18, (n, 1), device=dev, generator=g),
            "next": {"pixels": torch.randint(0, 256, (n, 4, 84, 84), dtype=torch.uint8, device=dev, generator=g),
                     "reward": torch.randn(n, device=dev, generator=g),
                     "done": torch.rand(n, 1, device=dev, generator=g) < 0.01,
                     "terminated": torch.rand(n, 1, device=dev, generator=g) < 0.01},
            "td_error": torch.rand(n, device=dev, generator=g)}, [n])
    # SAC continuous control (C5): obs / next obs f32[376], action f32[17], reward, done, terminated: 3 082 B + td_error
    return TensorDict({
        "observation": torch.randn(n, 376, device=dev, generator=g),
        "action": torch.randn(n, 17, device=dev, generator=g),
        "next": {"observation": torch.randn(n, 376, device=dev, generator=g),
                 "reward": torch.randn(n, device=dev, generator=g),
                 "done": torch.rand(n, 1, device=dev, generator=g) < 0.01,
                 "terminated": torch.rand(n, 1, device=dev, generator=g) < 0.01},
        "td_error": torch.rand(n, device=dev, generator=g)}, [n])


STREAM_ENVS, STREAM_STEPS = 8, 512


def make_stream_chunk(dev, g):
    """8 environment streams x 512 steps of 4-stacked 84x84 frames, flattened env-major like a collector batch.  The
    stream is periodic (its first stack is made of its own last frames), so writing the chunk again continues it."""
    from rl_b200.data import TensorDict

    E, T, k = STREAM_ENVS, STREAM_STEPS, 4
    frames = torch.randint(0, 256, (T, E, 84, 84), dtype=torch.uint8, device=dev, generator=g)
    win = torch.cat([frames[-k:], frames]).unfold(0, k + 1, 1).permute(1, 0, 4, 2, 3)   # [E, T, k + 1, 84, 84]
    n = E * T
    return TensorDict({
        "pixels": win[:, :, :k].reshape(n, k, 84, 84), "action": torch.randint(0, 18, (n, 1), device=dev, generator=g),
        "next": {"pixels": win[:, :, 1:].reshape(n, k, 84, 84), "reward": torch.randn(n, device=dev, generator=g),
                 "done": torch.zeros(n, 1, dtype=torch.bool, device=dev),
                 "terminated": torch.zeros(n, 1, dtype=torch.bool, device=dev)},
        "td_error": torch.rand(n, device=dev, generator=g)}, [n])


def build_sharded(dev, capacity_per_rank: int, world: int, rank: int, batch_per_rank: int = BATCH, kind: str = "atari",
                  fresh_rows: bool = True):
    """One shard per rank of a capacity-sharded buffer (weak scaling), filled with synthetic transitions.
    fresh_rows=False replicates one random chunk (new priorities per chunk): same bytes in HBM, much faster to fill."""
    from rl_b200.data.sharded import ShardedPrioritizedReplayBuffer

    g = torch.Generator(device=dev).manual_seed(1000 + rank)
    storage = None
    if kind == "atari_stream":
        from rl_b200.data import FrameStackStorage

        storage = FrameStackStorage(capacity_per_rank, n_envs=STREAM_ENVS, device=dev, min_episode_length=64)
    rb = ShardedPrioritizedReplayBuffer(alpha=ALPHA, beta=BETA, capacity=capacity_per_rank * world,
                                        batch_size=batch_per_rank * world, device=dev, generator=g, pipeline=True,
                                        n_buffers=N_BUFFERS, storage=storage)
    if kind == "atari_stream":
        td = make_stream_chunk(dev, g)
        assert capacity_per_rank % td.batch_size[0] == 0
        for _ in range(capacity_per_rank // td.batch_size[0]):
            td.set("td_error", torch.rand(td.batch_size[0], device=dev, generator=g))
            rb.extend(td)
        return rb, g
    chunk = 50_000 if kind == "atari" else 250_000
    td = None
    for lo in range(0, capacity_per_rank, chunk):
        n = min(chunk, capacity_per_rank - lo)
        if td is None or fresh_rows or n != td.batch_size[0]:
            td = make_rows(kind, n, dev, g)
        else:
            td.set("td_error", torch.rand(n, device=dev, generator=g))
        rb.extend(td)
    return rb, g


def dist_parity_check(rb, dev, rank: int, world: int) -> dict:
    """Warm-up assertion of the N > 1 run (SURVEY 8e parity row), product code only: this rank's draw must equal
    what the STAND-ALONE tree kernels (rlb_tree_query / rlb_tree_scan_lower_bound, not the fused sampler) give for the
    same uniforms; the gathered batch must equal the rank-order concatenation (NCCL all-gather) of aten::index rows of
    those draws; weights and indices must be identical on every rank.  The oracle-pinned version of the same statement
    is tests/mgpu_check.py (tests/test_mgpu.py)."""
    import torch.distributed as dist
    from rl_b200 import ops

    be = ops.backend()
    smp, st = rb.sampler, rb.storage
    smp._maybe_init_from_storage(st)
    gen = smp._rng
    state = gen.get_state()
    batch = rb.sample_now()
    torch.cuda.synchronize(dev)
    rb.check_exchange()
    g2 = torch.Generator(device=dev)
    g2.set_state(state)
    b_loc = rb._batch_size // world
    u = torch.rand(b_loc, device=dev, generator=g2)
    n = len(st)
    cap = smp._sum_tree.capacity
    zero, ln = torch.zeros(1, dtype=torch.long, device=dev), torch.full((1,), n, dtype=torch.long, device=dev)
    p_sum = be.tree_query(smp._sum_tree.values, smp._max_capacity, cap, False, zero, ln, True)
    idx = be.tree_scan_lower_bound(smp._sum_tree.values, smp._max_capacity, cap, u * p_sum).clamp_max(n - 1)
    ok = bool(torch.equal(idx, rb.local_index))
    detail = [] if ok else ["local draw != stand-alone tree kernels"]

    def gathered(x):
        out = torch.empty((world * x.shape[0], *x.shape[1:]), dtype=x.dtype, device=dev)
        dist.all_gather_into_tensor(out.view(torch.uint8) if x.dtype == torch.bool else out,
                                    x.contiguous().view(torch.uint8) if x.dtype == torch.bool else x.contiguous())
        return out

    if not torch.equal(batch.get("index"), gathered(idx + rank * rb.shard_capacity)):
        ok = False
        detail.append("index")
    keys = [k for k in batch.keys(True, True) if k not in ("index", "priority_weight")]
    if hasattr(st, "_gather_packed"):   # frame-stack shard: the rows are the storage's own (single-GPU) tensor-index read
        mine = st.get(idx)
        rows = {k: mine.get(k) for k in keys}
    else:
        data = unflatten_leaves(st)
        rows = {k: data[k][idx] for k in keys}
    for k in keys:
        if not torch.equal(batch.get(k), gathered(rows[k])):
            ok = False
            detail.append(str(k))
    w = batch.get("priority_weight")
    w0 = w.clone()
    dist.broadcast(w0, 0)
    if not torch.equal(w, w0):
        ok = False
        detail.append("weights differ between ranks")
    flag = torch.tensor([int(ok)], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return {"parity_checked": bool(flag.item()),
            "parity_detail": "gathered batch == rank-order concat of aten::index rows of each rank's draw; draw == "
                             "stand-alone tree kernels for the same uniforms; weights identical on all ranks"
                             if flag.item() else "FAILED on some rank: " + ",".join(detail)}


def unflatten_leaves(st) -> dict:
    """{key: [N, ...] storage leaf} for a TensorDict-structured storage."""
    from rl_b200.data.storages import unflatten_data

    td = unflatten_data(st._leaves, st._spec, (st._leaves[0].shape[0],))
    return {k: td.get(k) for k in td.keys(True, True)}


def exchange_probe(rb, dev, world: int) -> dict:
    """The fused gather + NVLink broadcast kernel on its own: graph of N_BUFFERS launches (rotating receive slots), all
    ranks at once.  Device time per launch and the resulting per-GPU NVLink egress / ingress rate."""
    import torch.distributed as dist
    from rl_b200 import ops

    be = ops.backend()
    st, lay = rb.storage, rb._layout
    bufs, _, _, peers = rb._symm
    b_loc = rb._batch_size // world
    g = torch.Generator(device=dev).manual_seed(17 + rb.rank)
    idxs = [torch.randint(0, len(st), (b_loc,), device=dev, generator=g) for _ in range(2 * N_BUFFERS)]
    payload = b_loc * sum(c[1] for c in lay.cols)
    out = {"payload_bytes_per_rank": payload, "multicast_available": rb._mc_delta != 0}
    for name, mc in (("unicast", 0), ("multicast", rb._mc_delta)):
        if name == "multicast" and not mc:
            continue
        fns = []
        for k, ix in enumerate(idxs):
            send = bufs[k % N_BUFFERS][rb.rank * b_loc:(rb.rank + 1) * b_loc]
            fns.append(lambda ix=ix, send=send, mc=mc: be.gather(st._leaves, ix, len(st), out=lay.leaf_views(send),
                                                                 peer_delta=peers, multicast_delta=mc))
        torch.cuda.synchronize(dev)
        dist.barrier()
        us = graph_us(fns, dev)
        t = torch.tensor([us], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        us = float(t.item())
        dist.barrier()
        out[name] = {"gather_broadcast_us": round(us, 2),
                     "nvlink_ingress_GBps": round((world - 1) * payload / us / 1e3, 1),
                     "frac_of_nvlink_per_dir": round((world - 1) * payload / us / 1e3 / NVLINK_GBPS_PER_DIR, 3)}
    return out


def run_distributed(args, dev, rank: int, world: int) -> dict:
    import torch.distributed as dist
    from rl_b200 import ops
    from rl_b200.graphs import CudaGraphStep

    be = ops.backend()
    gbatch = BATCH * world
    rb, g = build_sharded(dev, CAPACITY, world, rank)
    ring = gae_ring(dev, GAE_ROWS, GAE_T, g)
    ring8 = [(v, nv, r, d.view(torch.uint8), t.view(torch.uint8)) for v, nv, r, d, t in ring]
    R = len(ring)
    td_err = torch.rand(gbatch, device=dev, generator=g)
    td_loc = td_err[rank * BATCH:(rank + 1) * BATCH].contiguous()
    gs = (float(torch.tensor(GAMMA)), float(torch.tensor(GAMMA) * torch.tensor(LMBDA)))

    tick = torch.zeros(1, device=dev)

    def sync_all():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        # ... and a device-side barrier on the stream: the host barrier releases the ranks tens of microseconds apart,
        # which a timed region of one graph replay would count as step time of whoever waits for the late rank's rows
        dist.all_reduce(tick)

    parity = dist_parity_check(rb, dev, rank, world)
    nvlink = rb._symm not in (None, False)
    side_gae, side_upd = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    rb.record_index_event = True

    def make_step(slot: int):
        v, nv, r, d8, t8 = ring8[slot]

        def step():
            # main      rand -> per_sample -> gather + NVLink broadcast -> trailers + publish   (draw k)
            # fin       wait for the flags of draw k-1 -> importance weights                    (inside rb.sample)
            # side_upd  priority write-back of draw k's local rows: needs the sampled indices only
            # side_gae  GAE of this step's rollout
            main = torch.cuda.current_stream(dev)
            side_gae.wait_stream(main)
            with torch.cuda.stream(side_gae):
                a, tg = be.gae(v, nv, r, d8, t8, gs[0], gs[1], GAE_ROWS, GAE_T, 1)
            batch = rb.sample(slot=slot if nvlink else None)     # returns the finalised draw k-1
            side_upd.wait_event(rb.index_ready)
            with torch.cuda.stream(side_upd):
                rb.update_local_priority(td_loc)
            main.wait_stream(side_upd)
            main.wait_stream(side_gae)
            return batch, a, tg

        return step

    def make_eager_step(slot: int):
        v, nv, r, d8, t8 = ring8[slot]

        def step():
            batch = rb.sample()
            rb.update_priority(batch.get("index"), td_err)
            a, tg = be.gae(v, nv, r, d8, t8, gs[0], gs[1], GAE_ROWS, GAE_T, 1)
            return batch, a, tg

        return step

    eager_steps = [make_eager_step(i) for i in range(R)]
    clocks = ClockSampler(dev.index or 0) if rank == 0 else None
    ms_eager = timed(lambda i: eager_steps[i % R](), args.steps, args.warmup, sync_all)

    graphs, graph_err, ms_graph, ms_graph_long, spg = None, None, None, None, None
    try:
        if not nvlink:
            raise RuntimeError("NVLink transport unavailable (symmetric memory): the NCCL all-gather cannot be captured with the step")
        gen = rb.sampler._rng
        # spg consecutive steps per graph (a multiple of the receive-slot count, so graphs chain slot-continuously); the
        # exchanges run on their own stream beside the compute chain and rejoin once per graph
        spg, rem = group_plan(args.steps, N_BUFFERS)

        def make_group(g0: int, n: int | None = None):
            fns = [make_step((g0 + k) % R) for k in range(spg if n is None else n)]

            def group():
                outs = [fn() for fn in fns]
                rb.join_exchange()      # the exchange stream joins the capture once per graph, not once per step
                return outs

            return group

        graphs = [CudaGraphStep(make_group(g0), generators=[gen], warmup=1) for g0 in (0, spg)]
        # (left-over steps of a step count that is not a multiple of the slot count: one shorter graph, replayed last)
        tail = CudaGraphStep(make_group((args.steps // spg) * spg, rem), generators=[gen], warmup=1) if rem else None
        ms_graph = timed_groups(graphs, spg, args.steps, max(args.warmup, spg), sync_all, tail)
        ms_graph_long = timed_groups(graphs, spg, max(args.steps, 200) // spg * spg, spg, sync_all)
        torch.cuda.synchronize()
        rb.check_exchange()
    except Exception as err:
        import traceback

        graph_err = f"{type(err).__name__}: {err}"[:300]
        print(f"[bench rank {rank}] CUDA-graph path failed, falling back to eager: {graph_err}\n"
              + "".join(traceback.format_exc().splitlines(True)[-6:]), file=sys.stderr, flush=True)
        graphs, ms_graph, ms_graph_long = None, None, None
        torch.cuda.synchronize()
        fresh = torch.Generator(device=dev).manual_seed(4242 + rank)
        rb.local.set_rng(fresh)
        g = fresh
    clk = clocks.stop() if clocks else None

    ms_sample = timed(lambda i: rb.sample(), args.steps, 3, sync_all)
    own = slice(rank * BATCH, (rank + 1) * BATCH)
    ms_e2e, h2d, d2h, n_lanes = e2e_run(args, dev, rb, ring, td_err, gs, be, sync_all, own, 1)
    xprobe = None
    if nvlink:
        try:
            xprobe = exchange_probe(rb, dev, world)
        except Exception as e:  # noqa: BLE001
            xprobe = {"error": f"{type(e).__name__}: {e}"[:200]}

    vals = [ms_eager, ms_graph if ms_graph is not None else -1.0, ms_e2e, ms_sample,
            ms_graph_long if ms_graph_long is not None else -1.0]
    t = torch.tensor(vals, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_eager, ms_graph, ms_e2e, ms_sample, ms_graph_long = t.tolist()
    if ms_graph <= 0:
        ms_graph = None
    if ms_graph_long <= 0:
        ms_graph_long = None
    payload = BATCH * sum(c[1] for c in rb._layout.cols)
    multicast = bool(getattr(rb, "_mc_delta", 0))
    row_packed = rb._layout.row
    n_leaves = len(rb.storage._leaves)
    # free the C2 buffer before the bigger workloads
    del graphs, eager_steps, rb, ring, ring8
    import gc

    gc.collect()
    torch.cuda.empty_cache()
    extra = {}
    for name in (() if os.environ.get("RLB_BENCH_SKIP_EXTRAS") == "1" else ("c4", "c4_framestack", "c5")):
        try:
            extra[name] = sharded_workload(name, dev, rank, world, max(args.steps, 50), be)
        except Exception as e:  # noqa: BLE001
            import traceback

            extra[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
            print(f"[bench rank {rank}] workload {name} failed:\n" + "".join(traceback.format_exc().splitlines(True)[-8:]),
                  file=sys.stderr, flush=True)
        gc.collect()
        torch.cuda.empty_cache()
    if rank != 0:
        return None
    per_step = TRANSITIONS_PER_STEP * world
    ms = ms_graph if ms_graph is not None else ms_eager
    ingress = (world - 1) * BATCH * row_packed
    transport = ("gather kernel stores rows into every rank's symmetric receive buffer over NVLink peer memory; "
                 "flag release/acquire closes the exchange; sample() returns the previous draw" if nvlink
                 else "NCCL all-gather (eager)")
    cfg = make_config(world)
    detail = {"n_leaves": n_leaves, "transport": transport, "steps_per_graph": spg if ms_graph is not None else None,
              "launch": (f"cuda_graph replay of the public-API step, {spg} consecutive steps per graph; the exchange "
                         "of a draw runs on its own stream beside the next steps" if ms_graph is not None
                         else "eager python API")}
    result = {
        "metric": METRIC, "value": round(per_step / (ms * 1e-3), 1), "unit": "transitions/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 5), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "impl_detail": detail,
        "e2e": {"value": round(per_step / (ms_e2e * 1e-3), 1), "unit": "transitions/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": round(ms_e2e, 5),
                "note": "eager python API, pinned host buffers; every rank lands ITS rows of the global minibatch + its GAE outputs on the host"},
        "gpu_launches": 6 * args.steps,  # ours per step: per_sample, gather(+broadcast), pack(+publish), weights(+wait), update, gae
        **parity,
        "nvlink": {"ingress_bytes_per_step_per_gpu": ingress,
                   "egress_bytes_per_step_per_gpu": payload if multicast else ingress, "multicast": multicast,
                   "nvlink_ingress_GBps": round(ingress / (ms * 1e-3) / 1e9, 1),
                   "nvlink_egress_GBps": round((payload if multicast else ingress) / (ms * 1e-3) / 1e9, 1),
                   "wire_bound_us_per_step": round(ingress / (NVLINK_GBPS_PER_DIR * 1e9) * 1e6, 1),
                   "payload_bytes_per_rank": payload, "exchange_kernel": xprobe,
                   "note": "every rank receives the whole global minibatch (all-gather semantics): ingress = (N-1) x 256 packed rows; egress the same with unicast copies, 1 x with multicast stores (the switch replicates)"},
        "breakdown": {"eager_ms_per_step": round(ms_eager, 5),
                      "graph_ms_per_step": None if ms_graph is None else round(ms_graph, 5),
                      "graph_ms_per_step_long_run": None if ms_graph_long is None else round(ms_graph_long, 5),
                      "graph_error": graph_err, "eager_value": round(per_step / (ms_eager * 1e-3), 1),
                      "eager_sample_us": round(ms_sample * 1e3, 2)},
        "clocks": clk,
        "c4": extra.get("c4"), "c4_framestack": extra.get("c4_framestack"), "c5": extra.get("c5"),
    }
    return result


def sharded_workload(name: str, dev, rank: int, world: int, steps: int, be) -> dict:
    """BASELINE.json configs[3] / [4] at their per-shard sizes (weak-scaled below 8 GPUs):
    c4  10M-slot sharded PER of DQN-shaped Atari transitions, global batch 1024 at 8 GPUs (1.25M slots, 128 rows per rank)
    c5  50M-slot HBM-resident SAC buffer (obs 376 / act 17 f32), global batch 4096 at 8 GPUs (6.25M slots, 512 rows per
        rank) + TD-error priority write-back of the returned batch.
    A step = rb.sample() [+ write-back]; captured through the public API, replayed cyclically over the receive slots."""
    import torch.distributed as dist
    from rl_b200.graphs import CudaGraphStep

    spec = {"c4": dict(cap=1_250_000, b_loc=128, kind="atari"), "c5": dict(cap=6_250_000, b_loc=512, kind="mujoco"),
            "c4_framestack": dict(cap=305 * STREAM_ENVS * STREAM_STEPS, b_loc=128, kind="atari_stream")}[name]
    cap, b_loc, kind = spec["cap"], spec["b_loc"], spec["kind"]
    rb, g = build_sharded(dev, cap, world, rank, batch_per_rank=b_loc, kind=kind, fresh_rows=False)
    gb = b_loc * world
    td_err = torch.rand(gb, device=dev, generator=g)
    td_loc = td_err[rank * b_loc:(rank + 1) * b_loc].contiguous()
    rb.record_index_event = True
    side = torch.cuda.Stream(dev)

    tick = torch.zeros(1, device=dev)

    def sync_all():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        # ... and a device-side barrier on the stream: the host barrier releases the ranks tens of microseconds apart,
        # which a timed region of one graph replay would count as step time of whoever waits for the late rank's rows
        dist.all_reduce(tick)

    parity = dist_parity_check(rb, dev, rank, world)
    nvlink = rb._symm not in (None, False)

    def make_step(slot: int):
        def step():
            main = torch.cuda.current_stream(dev)
            batch = rb.sample(slot=slot if nvlink else None)
            if name == "c5":
                # TD-error write-back of the batch the learner just consumed (the returned draw): global indices,
                # replicated priorities; this rank rewrites the rows it owns
                rb.update_priority(batch.get("index"), td_err)
            else:
                side.wait_event(rb.index_ready)
                with torch.cuda.stream(side):
                    rb.update_local_priority(td_loc)
                main.wait_stream(side)
            return batch

        return step

    gen = rb.sampler._rng
    out = {}
    if nvlink:
        spg = 4 * N_BUFFERS

        def group():
            outs = [make_step(k)() for k in range(spg)]
            rb.join_exchange()
            return outs

        graphs = [CudaGraphStep(group, generators=[gen], warmup=1)]
        steps = max(spg, steps // spg * spg)
        ms = timed_groups(graphs, spg, steps, spg, sync_all)
        torch.cuda.synchronize()
        rb.check_exchange()
        launch = f"cuda_graph replay, {spg} steps per graph"
    else:
        eager = make_step(0)
        ms = timed(lambda i: eager(), steps, 4, sync_all)
        launch = "eager (NCCL transport)"
    ms_eager = timed(lambda i: rb.sample(), steps, 3, sync_all)
    wb = None
    if name == "c5":
        # the write-back alone, both ways: the returned index tensor (this rank's 512 rows, one launch) and an arbitrary
        # replicated global index vector of 4096 entries filtered inside the kernel (general path)
        batch = rb.sample()
        gi = batch.get("index")
        fast = graph_us([(lambda: rb.update_priority(gi, td_err)) for _ in range(10)], dev)
        gi2 = gi.clone()
        general = graph_us([(lambda: rb.update_priority(gi2, td_err)) for _ in range(10)], dev)
        wb = {"returned_batch_us": round(fast, 2), "general_global_index_us": round(general, 2), "n_global": gb}
    t = torch.tensor([ms, ms_eager], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_eager = t.tolist()
    lay = rb._layout
    row = sum(c[1] for c in lay.cols)
    ingress = (world - 1) * b_loc * lay.row
    labels = {"c4": "C4 sharded PER 10M DQN-shaped Atari transitions, batch 1024 @ 8 GPUs",
              "c5": "C5 50M HBM-resident SAC transitions (obs 376 / act 17 f32), batch 4096 @ 8 GPUs + TD-error write-back",
              "c4_framestack": "C4 on de-duplicated frame-stack shards (FrameStackStorage, 8 env streams per rank): the same "
                               "transitions, k + 1 = 5 distinct frames per exchanged row instead of 8"}
    if hasattr(rb.storage, "frame_bytes_per_transition"):
        hbm = int(rb.storage._pool.numel() + sum(l[0].numel() * l.element_size() for l in rb.storage._inner._leaves) * cap)
    else:
        hbm = cap * row
    out = {"workload": labels[name],
           "n_gpus": world, "capacity_global": cap * world, "capacity_per_gpu": cap, "global_batch": gb,
           "batch_per_gpu": b_loc, "row_bytes": row, "hbm_bytes_per_gpu": hbm,
           "ms_per_step": round(ms, 5), "transitions_per_s": round(gb / (ms * 1e-3), 1), "launch": launch,
           "eager_sample_us": round(ms_eager * 1e3, 2),
           "nvlink_bytes_per_step_per_gpu": ingress, "nvlink_ingress_GBps": round(ingress / (ms * 1e-3) / 1e9, 1),
           "wire_bound_us_per_step": round(ingress / (NVLINK_GBPS_PER_DIR * 1e9) * 1e6, 2),
           "writeback": wb, "matches_named_config": world == 8, **parity}
    del rb
    return out


# ------------------------------------------------------------------------------------------- reference arm
def cpu_baseline_run(steps: int | None, warmup: int = 2) -> dict:
    """The reference's own CPU path on the host cores: compiled reference segment trees (oracle/_ref/cpu) under
    the restated sampler glue, aten::index gather on CPU tensors, and the faster of the reference's two GAE code
    paths.  Bounded sample: a 20k-row CPU storage (gather cost is per row, not per capacity) and ~10-20 s of work; the
    timed run is repeated three times and the MEDIAN is reported (the host is shared: single runs vary 2x)."""
    from oracle import gae_torch
    from oracle import per_oracle as po
    from oracle.ref_loader import reference_trees

    cores = os.cpu_count() or 1
    factory = reference_trees("cpu")
    kind = "reference" if factory is not None else "port"
    smp = po.OraclePrioritizedSampler(CAPACITY, ALPHA, BETA, tree_factory=factory)
    g = torch.Generator().manual_seed(0)
    rows = 20_000
    smp.update_priority(torch.arange(CAPACITY), torch.rand(CAPACITY, generator=g))
    store = {"pixels": torch.randint(0, 256, (rows, 4, 84, 84), dtype=torch.uint8, generator=g),
             "next_pixels": torch.randint(0, 256, (rows, 4, 84, 84), dtype=torch.uint8, generator=g),
             "action": torch.randint(0, 18, (rows, 1), generator=g), "reward": torch.randn(rows, generator=g),
             "done": torch.rand(rows, 1, generator=g) < 0.01, "terminated": torch.rand(rows, 1, generator=g) < 0.01}
    v, nv, r = (torch.randn(GAE_ROWS, GAE_T, 1, generator=g) for _ in range(3))
    term = torch.rand(GAE_ROWS, GAE_T, 1, generator=g) < 0.02
    done = term | (torch.rand(GAE_ROWS, GAE_T, 1, generator=g) < 0.02)
    gm, lm = torch.tensor(GAMMA), torch.tensor(LMBDA)
    td = torch.rand(BATCH, generator=g)

    def t_of(fn, n):
        fn()
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        return (time.perf_counter() - t0) / n

    # give the reference the thread count it runs fastest with (many-core hosts oversubscribe the small ops of
    # the GAE code paths; aten::index parallelises over rows): tuned per phase on the bounded sample
    cands = sorted({c for c in (1, 4, 8, 16, 32, 64, cores) if c <= cores})
    ridx0 = torch.randint(0, rows, (BATCH,), generator=g)
    best_gae, best_gather = (None, None, 1e9), (None, 1e9)
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            for name, fn in (("loop", gae_torch.loop_gae), ("vec", gae_torch.vec_gae)):
                t = t_of(lambda: fn(gm, lm, v, nv, r, done, term), 2)
                if t < best_gae[2]:
                    best_gae = (name, c, t)
            t = t_of(lambda: {k: x[ridx0] for k, x in store.items()}, 3)
            if t < best_gather[1]:
                best_gather = (c, t)
    gae_fn = gae_torch.loop_gae if best_gae[0] == "loop" else gae_torch.vec_gae
    phases = {"tree_sample": 0.0, "gather": 0.0, "tree_update": 0.0, "gae": 0.0}

    def step():
        t0 = time.perf_counter()
        torch.set_num_threads(best_gather[0])
        idx, w = smp.sample(CAPACITY, BATCH, generator=g)
        t1 = time.perf_counter()
        ridx = idx % rows  # bounded storage: same number of random 28 KB rows touched
        batch = {k: x[ridx] for k, x in store.items()}
        t2 = time.perf_counter()
        smp.update_priority(idx, td)
        t3 = time.perf_counter()
        torch.set_num_threads(best_gae[1])
        with torch.no_grad():
            a, t = gae_fn(gm, lm, v, nv, r, done, term)
        t4 = time.perf_counter()
        phases["tree_sample"] += t1 - t0
        phases["gather"] += t2 - t1
        phases["tree_update"] += t3 - t2
        phases["gae"] += t4 - t3
        return batch, a, t

    for _ in range(warmup):
        step()
    if steps is None:
        t1 = t_of(step, 2)
        steps = max(5, min(400, int(4.0 / max(t1, 1e-4))))
    runs = []
    for _ in range(3):
        for k in phases:
            phases[k] = 0.0
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        runs.append(((time.perf_counter() - t0) / steps, {k: v / steps * 1e3 for k, v in phases.items()}))
    runs.sort(key=lambda x: x[0])
    dt, ph = runs[1]
    return {"value": round(TRANSITIONS_PER_STEP / dt, 1), "unit": "transitions/s",
            "cores": max(best_gather[0], best_gae[1]), "host_cores": cores, "kind": kind,
            "ms_per_step": round(dt * 1e3, 3), "steps": steps, "cpu_storage_rows": rows,
            "runs_ms_per_step": [round(x[0] * 1e3, 3) for x in runs], "phases_ms": {k: round(v, 4) for k, v in ph.items()},
            "sample": (f"median of 3 x {steps} steps of [reference C++ SumSegmentTree/MinSegmentTree sample+update B=256 @1M "
                       f"(single-threaded by construction) + aten::index gather of 256 Atari transitions from a "
                       f"{rows}-row CPU storage ({best_gather[0]} threads, {best_gather[1] * 1e3:.2f} ms) + "
                       f"{best_gae[0]} GAE [4096,128] ({best_gae[1]} threads, {best_gae[2] * 1e3:.1f} ms)]; thread "
                       f"counts are the fastest of {cands} for each phase")}


def run_reference(args) -> dict | None:
    rank, world, _ = dist_env()
    if rank != 0:
        return None
    cpu = cpu_baseline_run(steps=args.steps, warmup=args.warmup)
    cfg = make_config(world)
    return {"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "transitions/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cpu["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": cfg,
            "impl_note": "reference CPU implementation on the host cores; rank 0 only",
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "transitions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def _watchdog(seconds: float) -> None:
    """A hung collective must not hang the caller: after `seconds` the process prints what it knows and exits."""
    def fire():
        rank = int(os.environ.get("RANK", 0))
        if rank == 0:
            print(json.dumps({"metric": METRIC, "error": f"bench.py watchdog fired after {seconds:.0f} s",
                              "n_gpus": int(os.environ.get("WORLD_SIZE", 1))}), flush=True)
        os._exit(3)

    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step to DIR/<name>.npy (one GPU)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1 or dist_env()[1] != 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    if args.warmup < 3:
        args.warmup = 3
    _watchdog(float(os.environ.get("RLB_BENCH_TIMEOUT", "840")))
    if args.impl == "reference":
        res = run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; rl_b200 has no CPU fallback (use --impl reference for the CPU arm)")
        res = run_ours(args)
    if res is not None:
        print(json.dumps(res))


if __name__ == "__main__":
    main()
