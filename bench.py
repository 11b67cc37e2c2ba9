#!/usr/bin/env python
"""bench.py -- recommend() users/sec of the B200 score + top-K engine on BASELINE.json's configurations.

    python bench.py --gpus N --steps K --warmup W [--config c2|c3|c4|c5] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (score every user against the catalogue, mask viewed items, keep the K best)
over one batch of synthetic users (SURVEY.md section 8d synthetic inputs: N(0,1)/sqrt(d) factors, fixed seeds, ~100 viewed
items per user).  Named workloads (BASELINE.json `configs[1..4]`; the default is the one `metric` is quoted on):
  c2  ImplicitALS-shaped factors, users = items = 1M, d = 128, Distance.DOT, K = 10                     (default)
  c3  the same with Distance.COSINE and K = 100 (single-pass wide mode)
  c4  users = 1M, items = 10M, d = 128, DOT, K = 10 (8 GPUs: 1.25M items per shard)
  c5  SASRec-shaped id embeddings, users = 1M, items = 5M, d = 256, bf16 tensor-core candidates, K = 20

  value  : whole-job users/sec with every input already resident in HBM (device-timed, max over ranks)
  e2e    : the same metric through the public host API (`Engine.topk`; N > 1: `ShardedB200Ranker.rank_device` with host
           matrices): per step the users' factors + CSR filter are copied from pinned host memory and the K (id, score)
           pairs copied back
  N > 1  : the catalogue is item-sharded over the ranks (north_star) through `rectools_b200.sharded.ShardedB200Ranker`: every
           rank scores all users against its shard (thresholds shared over NVLink peer memory), an NCCL all-to-all by user
           slice + a certifying merge kernel + an all-gather of the merged slices; total work is fixed => "scaling": "strong"
  model_recommend : `ImplicitALSWrapperModel.recommend()` of the UNMODIFIED reference (staged in oracle/_ref) after
           `rectools_b200.install()`, users/sec incl. the host code around the ranker (N = 1, when the package is staged)
  --impl reference : the reference's CPU path (restatement of implicit.cpu.topk: BLAS sgemm + OpenMP select, all host
           threads) on a bounded sample of the same workload, rank 0 only.
  --dump-outputs DIR : after the timed steps, write what the last timed step returned (top-K ids, scores, counts; rank 0)
           as DIR/<name>.npy for output-by-output comparison of two builds: `rows` (the users), `ids` and `counts` in
           float64, `scores` in float32.  Inputs are seeded, so equal arguments give equal inputs; above DUMP_BYTES a
           fixed, seeded sample of the users is written.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ of the modules imported below is written there

BLOCK = 65536
DUMP_BYTES = 64_000_000  # --dump-outputs: the whole dump (all .npy files) stays below this


def gen_factors(n, d, seed, lo=0, hi=None):
    """Rows [lo, hi) of the seeded N(0,1)/sqrt(d) fp32 matrix; generated in blocks so shards can be made independently."""
    hi = n if hi is None else hi
    out = np.empty((hi - lo, d), dtype=np.float32)
    b0 = lo // BLOCK
    pos = 0
    for b in range(b0, (hi + BLOCK - 1) // BLOCK):
        r0, r1 = b * BLOCK, min((b + 1) * BLOCK, n)
        blk = np.random.default_rng([seed, b]).standard_normal((r1 - r0, d), dtype=np.float32)
        blk *= np.float32(1.0 / np.sqrt(d))
        a, z = max(lo, r0), min(hi, r1)
        out[pos : pos + (z - a)] = blk[a - r0 : z - r0]
        pos += z - a
    return out


def gen_viewed(n_users, n_items, per_user, seed=2):
    """CSR of ~per_user viewed items per user: int64 indptr, int32 sorted indices (rare duplicates kept)."""
    cols = np.empty((n_users, per_user), dtype=np.int32)
    for b in range((n_users + BLOCK - 1) // BLOCK):
        r0, r1 = b * BLOCK, min((b + 1) * BLOCK, n_users)
        c = np.random.default_rng([seed, b]).integers(0, n_items, size=(r1 - r0, per_user), dtype=np.int32)
        c.sort(axis=1)
        cols[r0:r1] = c
    indptr = np.arange(n_users + 1, dtype=np.int64) * per_user
    return indptr, cols.reshape(-1)


def dump_outputs(out_dir, rows, ids, scores, counts):
    """Write the top-K result of `rows` (global user indices) under `out_dir`: every user when it fits DUMP_BYTES, else a
    seeded sample of users (sorted, the same for every run with the same shapes)."""
    ids, scores, counts = np.asarray(ids).reshape(len(rows), -1), np.asarray(scores).reshape(len(rows), -1), np.asarray(counts)
    k = ids.shape[1]
    per_row = 8 + 8 * k + 4 * k + 8  # rows, ids (float64), scores (float32), counts (float64)
    n_keep = min(len(rows), (DUMP_BYTES - 4 * 128) // per_row)  # (4 * 128: the .npy headers)
    sel = np.arange(len(rows))
    if n_keep < len(rows):
        sel = np.sort(np.random.default_rng(20260).choice(len(rows), n_keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rows.npy"), np.asarray(rows)[sel].astype(np.float64))
    np.save(os.path.join(out_dir, "ids.npy"), ids[sel].astype(np.float64))
    np.save(os.path.join(out_dir, "scores.npy"), scores[sel].astype(np.float32))
    np.save(os.path.join(out_dir, "counts.npy"), counts[sel].astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = (
        "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    )

    def __init__(self, device):
        self.device, self.rows, self.proc, self.first = device, [], None, 0

    def mark(self):
        """Samples taken before this call (warm-up) are not reported.  The sampler is started BEFORE the warm-up because
        nvidia-smi's start-up (NVML initialisation over every GPU of the box) can stall CUDA calls of this process for tens
        of milliseconds -- measured as a one-off gap inside the first timed step when it was started right before it."""
        self.first = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.device)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[self.first:]:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                pw.append(float(r[2]))
            except ValueError:
                continue
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": float(np.median(sm)) if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "power_w_max": max(pw) if pw else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


CONFIGS = {
    # name: (users, items, dim, k, viewed, distance, tc, label)
    "c2": dict(users=1_000_000, items=1_000_000, dim=128, k=10, viewed=100, distance="dot", tc="auto",
               label="config2: ImplicitALSWrapperModel-shaped factors (n_factors=128)"),
    "c3": dict(users=1_000_000, items=1_000_000, dim=128, k=100, viewed=100, distance="cosine", tc="auto",
               label="config3: the config-2 factors with Distance.COSINE (fused L2-normalise)"),
    "c4": dict(users=1_000_000, items=10_000_000, dim=128, k=10, viewed=100, distance="dot", tc="auto",
               label="config4: synthetic factors, 10M items (item-sharded across the GPUs, NCCL top-K merge)"),
    "c5": dict(users=1_000_000, items=5_000_000, dim=256, k=20, viewed=100, distance="dot", tc="bf16",
               label="config5: SASRecModel-shaped id embeddings (n_factors=256), bf16 tensor-core path"),
}


def resolve_config(a):
    cfg = CONFIGS[a.config]
    for key in ("users", "items", "dim", "k", "viewed", "distance", "tc"):
        if getattr(a, key) is None:
            setattr(a, key, cfg[key])
    return cfg


def workload_name(a):
    return (
        f"{CONFIGS[a.config]['label']}: users={a.users} items={a.items} d={a.dim} Distance.{a.distance.upper()} "
        f"K={a.k} filter_viewed=True (~{a.viewed} viewed/user)"
    )


def rounded(x, tc):
    """bf16 runs: the factors are rounded to bf16 FIRST and the same rounded values go to the engine and the oracle (SURVEY 8d)."""
    if tc != "bf16":
        return x
    import torch

    return torch.from_numpy(x).to(torch.bfloat16).float().numpy()


# --------------------------------------------------------------------------------------------------------------
def run_reference(a):
    """CPU arm: restatement of the reference's implicit.cpu.topk path on the host cores (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import cpu_baseline
    from oracle.topk_oracle import calc_norms

    threads = cpu_baseline.use_all_threads()  # (torchrun exports OMP_NUM_THREADS=1)
    n_s = a.ref_users
    # bound the sample: the sgemm of one step is n_s x items x d; keep ~3e11 FLOP per step whatever the catalogue size
    n_s = max(64, min(n_s, int(n_s * (1_000_000 * 128) / (a.items * a.dim))))
    items = rounded(gen_factors(a.items, a.dim, 1), a.tc)
    users = rounded(gen_factors(a.users, a.dim, 0, 0, min(a.users, n_s * (a.steps + a.warmup))), a.tc)
    indptr, indices = gen_viewed(len(users), a.items, a.viewed)
    from scipy import sparse

    csr = sparse.csr_matrix((np.ones(len(indices), np.float32), indices, indptr), shape=(len(users), a.items))
    norms = calc_norms(items) if a.distance == "cosine" else None
    times = []
    for s in range(a.warmup + a.steps):
        lo = (s * n_s) % max(1, len(users) - n_s + 1)
        t0 = time.perf_counter()
        last = cpu_baseline.topk_cpu(items, users[lo : lo + n_s], a.k, norms, csr[lo : lo + n_s], num_threads=threads)
        dt = time.perf_counter() - t0
        if s >= a.warmup:
            times.append(dt)
    if a.dump_outputs:
        ids, scores = last
        # (like implicit's topk, topk_cpu leaves filtered items in the rows with score -FLT_MAX; they are not results)
        dump_outputs(a.dump_outputs, np.arange(lo, lo + ids.shape[0]), ids, scores, (scores > -np.finfo(np.float32).max).sum(axis=1))
    total = sum(times)
    value = n_s * len(times) / total
    line = {
        "impl": "reference",
        "metric": "recommend() users/sec",
        "value": value,
        "unit": "users/s",
        "n_gpus": a.gpus,
        "steps": a.steps,
        "warmup": a.warmup,
        "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(a), "name": a.config, "sample": f"{n_s} users per step against all {a.items} items"},
        "cpu_baseline": {
            "value": value, "unit": "users/s", "cores": threads, "kind": "port",
            "sample": f"{n_s} users x {a.items} items per step; numpy/OpenBLAS sgemm + C/OpenMP per-row select, {threads} threads each "
                      "(oracle/cpu_baseline.py, restating implicit.cpu.topk.topk as called at rank_implicit.py:264-272)",
        },
        "e2e": {"value": value, "unit": "users/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def model_recommend_leg(a, items, users, indptr, indices, dev_index):
    """`ImplicitALSWrapperModel.recommend()` of the unmodified reference with the engine installed under it (SURVEY 8d:
    reported next to e2e; includes the host code around the ranker: CSR provider, id maps, the result DataFrame)."""
    from oracle import stage_reference

    if not stage_reference.available():
        return {"unavailable": "reference package not staged (oracle/_ref is made by __graft_entry__.build() in the build container)"}
    added = stage_reference.add_to_path()
    try:
        import pandas as pd
        from rectools import Columns
        from rectools.dataset import Dataset, IdMap, Interactions

        import rectools_b200
        from tests.ref_models import injected_als

        n_users, n_items = users.shape[0], items.shape[0]
        t0 = time.perf_counter()
        rows = np.repeat(np.arange(n_users, dtype=np.int64), np.diff(indptr))
        keep = np.ones(len(indices), dtype=bool)  # the rows are sorted: duplicated (user, item) pairs are neighbours
        keep[1:] = (indices[1:] != indices[:-1]) | (rows[1:] != rows[:-1])
        df = pd.DataFrame({Columns.User: rows[keep], Columns.Item: indices[keep].astype(np.int64)})
        del rows, keep
        df[Columns.Weight] = np.float64(1.0)
        df[Columns.Datetime] = pd.Timestamp("2024-01-01")
        dataset = Dataset(IdMap(np.arange(n_users, dtype=np.int64)), IdMap(np.arange(n_items, dtype=np.int64)), Interactions(df))
        model = injected_als(users, items)  # the injection of tests/models/test_implicit_als.py:193-197
        t_setup = time.perf_counter() - t0
        rectools_b200.install(device=dev_index, tc_mode=a.tc)
        try:
            all_users = dataset.user_id_map.external_ids
            t0 = time.perf_counter()
            reco = model.recommend(all_users, dataset, k=a.k, filter_viewed=True)  # first call: builds + caches the viewed CSR
            t_first = time.perf_counter() - t0
            times = []
            for _ in range(2):
                t0 = time.perf_counter()
                reco = model.recommend(all_users, dataset, k=a.k, filter_viewed=True)
                times.append(time.perf_counter() - t0)
        finally:
            rectools_b200.uninstall()
        best = min(times)
        return {
            "value": n_users / best, "unit": "users/s", "seconds": best, "first_call_seconds": t_first, "setup_seconds": t_setup,
            "rows": int(len(reco)), "interactions": int(len(df)),
            "api": "rectools.models.ImplicitALSWrapperModel.recommend(users, dataset, k, filter_viewed=True) after rectools_b200.install() "
                   "(unmodified reference from oracle/_ref; pre-fitted factors injected as in tests/models/test_implicit_als.py:193-197)",
        }
    except Exception as exc:  # pylint: disable=broad-except
        return {"unavailable": f"{type(exc).__name__}: {exc}"}
    finally:
        stage_reference.remove_from_path(added)


# --------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="named BASELINE.json workload (default: c2, the headline)")
    ap.add_argument("--users", type=int, default=None)
    ap.add_argument("--items", type=int, default=None)
    ap.add_argument("--dim", type=int, default=None)
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--viewed", type=int, default=None)
    ap.add_argument("--distance", default=None, choices=["dot", "cosine"])
    ap.add_argument("--tc", default=None, choices=["auto", "fp16", "bf16", "off"])
    ap.add_argument("--ref-users", type=int, default=1024, help="users per step of the CPU arms (bounded sample)")
    ap.add_argument("--parity-users", type=int, default=1024, help="users of the in-run parity sample (N > 1: at most 256)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-model", action="store_true", help="skip the model.recommend() leg")
    ap.add_argument("--no-share", action="store_true", help="N > 1: no threshold sharing between the item shards")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's top-K result as DIR/<name>.npy (see the module docstring)")
    ap.add_argument("--item-shards", type=int, default=0,
                    help="N > 1: item shards I (a divisor of N); the ranks form I item shards x N/I user groups.  0 = N (the north-star "
                         "scheme: every rank ranks all users against 1/N of the catalogue); 1 = plain user sharding")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(a.warmup, 0)
    resolve_config(a)

    if a.impl == "reference":
        run_reference(a)
        return

    import torch

    from rectools_b200 import Engine, _lib
    from rectools_b200.sharded import ShardedB200Ranker, shard_bounds

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)

    # ---------------- partitioning: I item shards x Ug user groups (default I = world: item sharding, north star)
    n_ishards = a.item_shards if a.item_shards > 0 else world
    if world % n_ishards:
        raise SystemExit("--item-shards must divide the number of GPUs")
    n_ugroups = world // n_ishards
    shard_idx, group_idx = rank % n_ishards, rank // n_ishards
    n_users_all = a.users
    wl_name = workload_name(a)
    u0, u1 = shard_bounds(n_users_all, n_ugroups)[group_idx]

    # ---------------- synthetic inputs (this rank's item range and user slice)
    lo, hi = shard_bounds(a.items, n_ishards)[shard_idx]
    items_local = rounded(gen_factors(a.items, a.dim, 1, lo, hi), a.tc)
    users = rounded(gen_factors(n_users_all, a.dim, 0, u0, u1), a.tc)
    indptr, indices = gen_viewed(n_users_all, a.items, a.viewed)
    if n_ugroups > 1:
        indices = indices[indptr[u0] : indptr[u1]].copy()
        indptr = (indptr[u0 : u1 + 1] - indptr[u0]).copy()
    n_loc_users = u1 - u0  # rows this rank ranks; n_users_all is the whole job
    k = min(a.k, a.items)

    if world == 1:
        eng = Engine(items_local, cosine=a.distance == "cosine", device=local_rank, tc_mode=a.tc)
        sharded = None
    else:
        # the repo's own multi-GPU API: item shards (x user groups), thresholds shared over NVLink peer memory, one packed
        # all-gather + certifying merge (rectools_b200/sharded.py)
        sharded = ShardedB200Ranker(a.distance, None, items_local, device=local_rank, tc_mode=a.tc, objects_are_local=True,
                                    n_objects_total=a.items, item_shards=n_ishards, share_thresholds=not a.no_share, max_rows=n_users_all)
        eng = sharded.local.engine
    info = eng.info()

    # device-resident copies for the `value` measurement
    d_users = torch.from_numpy(users).to(dev)
    d_indptr = torch.from_numpy(indptr).to(dev)
    d_indices = torch.from_numpy(indices).to(dev)
    if world == 1:
        o_ids = torch.empty((n_loc_users, k), dtype=torch.int32, device=dev)
        o_sc = torch.empty((n_loc_users, k), dtype=torch.float32, device=dev)
        o_cnt = torch.empty((n_loc_users,), dtype=torch.int32, device=dev)
    launches = [0]
    stats_log = []
    result = {}

    def step_resident():
        if world == 1:
            st = eng.topk_ptrs(
                n_loc_users, k, o_ids.data_ptr(), o_sc.data_ptr(), o_cnt.data_ptr(),
                _lib.Q_INPUTS_ON_DEVICE | _lib.Q_OUTPUTS_ON_DEVICE,
                subjects=d_users.data_ptr(), indptr=d_indptr.data_ptr(), indices=d_indices.data_ptr(),
                stream=torch.cuda.current_stream().cuda_stream,
            )
            result["ids"], result["sc"] = o_ids, o_sc
        else:
            result["ids"], result["sc"], result["cnt"] = sharded.rank_device(d_users, k, d_indptr, d_indices)
            st = dict(sharded.last_stats)
            launches[0] += 2  # the merge kernels (init + select)
        launches[0] += st.get("n_launches", 0)
        stats_log.append(st)

    # pinned host buffers for the end-to-end measurement
    if not a.no_e2e:
        h_users = torch.from_numpy(users).pin_memory()
        h_indptr = torch.from_numpy(indptr).pin_memory()
        h_indices = torch.from_numpy(indices).pin_memory()
        if world == 1:
            h_ids = torch.empty((n_loc_users, k), dtype=torch.int32).pin_memory()
            h_sc = torch.empty((n_loc_users, k), dtype=torch.float32).pin_memory()
            h_cnt = torch.empty((n_loc_users,), dtype=torch.int32).pin_memory()
        else:
            hm_ids = torch.empty((n_users_all, k), dtype=torch.int32).pin_memory()
            hm_sc = torch.empty((n_users_all, k), dtype=torch.float32).pin_memory()
    e2e_bytes = [0, 0]
    e2e_stats = {}

    def step_e2e():
        if world == 1:
            eng.topk(k, subjects=h_users.numpy(), indptr=h_indptr.numpy(), indices=h_indices.numpy(),
                     out=(h_ids.numpy(), h_sc.numpy(), h_cnt.numpy()))
            st = eng.last_stats
        else:
            ids, sc, _ = sharded.rank_device(h_users, k, h_indptr, h_indices)  # host matrices in, merged device tensors out
            st = dict(sharded.last_stats)
            if rank == 0:
                hm_ids.copy_(ids, non_blocking=True)
                hm_sc.copy_(sc, non_blocking=True)
                st["d2h_bytes"] = int(ids.shape[0]) * k * 8
            torch.cuda.current_stream().synchronize()
        e2e_bytes[0], e2e_bytes[1] = st.get("h2d_bytes", 0), st.get("d2h_bytes", 0)
        e2e_stats.clear()
        e2e_stats.update({kk: st.get(kk) for kk in ("ms_total", "ms_main", "ms_select", "ms_h2d", "ms_d2h")})

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_ms_log = []

    def timed(fn, warmup, steps):
        for _ in range(warmup):
            fn()
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record()
        for i in range(steps):
            fn()
            ev[i + 1].record()
        barrier()
        ms = torch.tensor([ev[0].elapsed_time(ev[steps])], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        step_ms_log.append([round(ev[i].elapsed_time(ev[i + 1]), 3) for i in range(steps)])  # this rank's per-step times
        return float(ms.item())

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(a.warmup, 3) if a.steps > 0 else 0):
        step_resident()
    launches[0] = 0
    stats_log.clear()
    sampler.mark()
    total_ms = timed(step_resident, 0, a.steps)
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        if world == 1:
            dump_outputs(a.dump_outputs, np.arange(u0, u1), o_ids.cpu().numpy(), o_sc.cpu().numpy(), o_cnt.cpu().numpy())
        else:  # rank 0 holds the merged result of the whole job
            ids = result["ids"].cpu().numpy()
            dump_outputs(a.dump_outputs, np.arange(ids.shape[0]), ids, result["sc"].cpu().numpy(), result["cnt"].cpu().numpy())
    timed_launches = launches[0]
    timed_stats = list(stats_log)
    value = n_users_all * a.steps / (total_ms / 1e3)  # whole job: all user groups

    e2e = None
    if not a.no_e2e:
        e2e_steps = max(1, min(a.steps, 3))
        e2e_ms = timed(step_e2e, 1, e2e_steps)
        e2e = {
            "value": n_users_all * e2e_steps / (e2e_ms / 1e3), "unit": "users/s", "steps": e2e_steps,
            "h2d_bytes_per_step": int(e2e_bytes[0]), "d2h_bytes_per_step": int(e2e_bytes[1]),
            "api": ("rectools_b200.Engine.topk (C ABI b200_rank_topk) with pinned host buffers" if world == 1 else
                    "rectools_b200.sharded.ShardedB200Ranker.rank_device with pinned host matrices (per rank: C ABI b200_rank_topk, NCCL "
                    "all-to-all + b200_rank_merge_certified + all-gather), merged result copied to the host on rank 0"),
            "engine_ms_last_step": dict(e2e_stats),
        }
        step_resident()  # leave the resident result in `result` for the parity sample

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (the fused tensor-core pass), timed by CUDA events in the engine:
    # ms_main sums EVERY launch of the fused kernel in a step (main pass, re-rank passes)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    ms_main = float(np.mean([s["ms_main"] for s in timed_stats])) if timed_stats else float("nan")
    ms_select = float(np.mean([s.get("ms_select", 0.0) for s in timed_stats])) if timed_stats else float("nan")
    path = timed_stats[0]["path"] if timed_stats else -1
    n_loc = hi - lo
    flops = 2.0 * n_loc_users * n_loc * a.dim
    st0 = timed_stats[0] if timed_stats else {}
    if path == 1:
        peak = peaks.get("bf16_tflops_sustained")
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (the kernel runs ~all of a long step)"
        if peak is None:
            peak, peak_src = 1400.0, "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md; MEASURED_PEAKS.json absent)"
        achieved = flops / (ms_main * 1e-3) / 1e12
        # dram__bytes_read + write of one launch of this kernel from the committed `ncu --set full` capture, when that
        # capture was taken on exactly this workload; otherwise null
        traffic = None
        for cap_name in ("r02_ncu_fused_kernel.json", "r01_ncu_tc_kernel.json"):
            try:
                cap = json.load(open(os.path.join(ROOT, "profiles", cap_name)))
                if world == 1 and (cap["users"], cap["items"], cap["dim"]) == (n_loc_users, a.items, a.dim) and cap.get("k", 10) == k:
                    traffic = cap["dram_bytes_per_launch"]
                    break
            except (OSError, ValueError, KeyError):
                pass
        shard_bytes = int(n_loc * info["d_pad"] * 2)
        n_waves = -(-(-(-n_loc_users // 256)) // (info["sm_count"] // 2))  # waves of subject tiles = HBM passes over the shard
        roof = {
            "kernel": f"fused_topk_kernel<{st0.get('epi_warps', 8)}> (TMA -> tcgen05.mma.cta_group::2 256x256x16 -> TMEM -> fused streaming "
                      "top-K' selection" + (", wide mode: frozen threshold + global append" if st0.get("wide") else "") + ")",
            "bound": "tensor",
            "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
            "frac": achieved / peak, "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram read+write)", "peak_source": peak_src,
            "algorithmic": f"2*U*N_g*d = 2*{n_loc_users}*{n_loc}*{a.dim} FLOP per step",
            "ms_per_launch": ms_main, "launches_per_step": st0.get("n_tc_launches"),
            "ms_select_per_step": ms_select,
            "peak_burst": peaks.get("bf16_tflops"),
            "frac_of_burst": achieved / peaks["bf16_tflops"] if peaks.get("bf16_tflops") else None,
            "item_stream": {
                "note": "item-factor HBM stream: the carousel keeps the CTA pairs on the same object tiles, so the 16-bit shard is read "
                        "from HBM about once per wave of subject tiles (the other 73 of 74 reads are L2 hits); the path is tensor-bound",
                "shard_bytes": shard_bytes, "hbm_passes_per_step": n_waves,
                "achieved_gbs": shard_bytes * n_waves / (ms_main * 1e-3) / 1e9,
                "hbm_gbs_peak": peaks.get("hbm_gbs"),
                "frac_of_hbm_peak": (shard_bytes * n_waves / (ms_main * 1e-3) / 1e9) / peaks["hbm_gbs"] if peaks.get("hbm_gbs") else None,
            },
        }
    else:
        achieved = flops / (ms_main * 1e-3) / 1e12
        roof = {"kernel": "exact_topk_kernel", "bound": "fp64", "achieved": achieved, "peak": None, "unit": "TFLOP/s",
                "frac": None, "traffic": None, "ms_per_launch": ms_main}

    # ---------------- parity sample against the fp64 oracle, same run
    parity = None
    if a.parity_users > 0:
        from oracle.topk_oracle import rank_oracle
        from scipy import sparse

        # N > 1: rank 0 checks the merged result of (a sample of) its own user slice against the WHOLE catalogue
        n_par = min(a.parity_users, n_loc_users) if world == 1 else min(a.parity_users, 256, n_loc_users)
        sel = np.unique(np.linspace(0, n_loc_users - 1, n_par).astype(np.int64))
        csr = sparse.csr_matrix((np.ones(len(indices), np.float32), indices, indptr), shape=(n_loc_users, a.items))[sel]
        items_all = items_local if world == 1 else rounded(gen_factors(a.items, a.dim, 1), a.tc)
        got_ids = result["ids"].cpu().numpy()[sel].reshape(-1)
        got_sc = result["sc"].cpu().numpy()[sel].reshape(-1)
        # (score blocks of the oracle bounded to ~2 GB of fp64: 250 users at 1M items, 25 at 10M)
        _, oid, osc = rank_oracle(a.distance, users[sel], items_all, np.arange(len(sel)), k, csr, accum="f64",
                                  batch=max(8, min(512, int(2.5e8 / a.items))))
        if a.distance == "cosine":
            un = np.sqrt(np.einsum("ij,ij->i", users[sel], users[sel], dtype=np.float64)).astype(np.float32)
            osc = osc * np.repeat(un, k)
        mism = int((got_ids != oid).sum())
        max_rel = float(np.max(np.abs(got_sc - osc) / np.maximum(np.abs(osc), 1e-30)))
        parity = {"users_checked": int(len(sel)), "id_mismatches": mism, "max_rel_score_err": max_rel,
                  "oracle": "oracle/topk_oracle.py rank_oracle(accum='f64')"}

    cpu = None
    if not a.no_cpu_baseline and world == 1:
        from oracle import cpu_baseline
        from oracle.topk_oracle import calc_norms
        from scipy import sparse

        threads = cpu_baseline.use_all_threads()
        n_s = max(64, min(a.ref_users, n_loc_users, int(a.ref_users * (1_000_000 * 128) / (a.items * a.dim))))
        csr = sparse.csr_matrix((np.ones(int(indptr[n_s]), np.float32), indices[: int(indptr[n_s])], indptr[: n_s + 1]), shape=(n_s, a.items))
        norms = calc_norms(items_local) if a.distance == "cosine" else None
        cpu_baseline.topk_cpu(items_local, users[: min(64, n_s)], k, norms, csr[: min(64, n_s)], num_threads=threads)  # warm-up
        t0 = time.perf_counter()
        reps = 0
        while reps < 1 or (time.perf_counter() - t0 < 10 and reps < 8):
            cpu_baseline.topk_cpu(items_local, users[:n_s], k, norms, csr, num_threads=threads)
            reps += 1
        dt = (time.perf_counter() - t0) / reps
        cpu = {"value": n_s / dt, "unit": "users/s", "cores": threads, "kind": "port",
               "sample": f"{n_s} users x {a.items} items, {reps} repetitions; numpy/OpenBLAS sgemm + C/OpenMP select, {threads} threads each, "
                         "restating implicit.cpu.topk.topk (rank_implicit.py:264-272)"}

    model_reco = None
    if not a.no_model and world == 1 and a.distance == "dot" and a.tc != "bf16":
        # (ImplicitALSWrapperModel's u2i distance is hard-wired to DOT, implicit_als.py:136)
        del d_users, d_indptr, d_indices
        model_reco = model_recommend_leg(a, items_local, users, indptr, indices, local_rank)

    line = {
        "metric": "recommend() users/sec",
        "value": value,
        "unit": "users/s",
        "n_gpus": world,
        "steps": a.steps,
        "warmup": max(a.warmup, 3),
        "ms_per_step": total_ms / max(a.steps, 1),
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": ("f16" if info["tc_dtype"] == 1 else "bf16" if info["tc_dtype"] == 2 else "f64")
        + " tensor-core candidates + f64-accumulated f32 re-score",
        "data": "synthetic",
        "config": {
            "workload": wl_name,
            "name": a.config,
            "parallelism": (
                "single GPU" if world == 1 else
                f"items sharded over {world} GPU(s) (ShardedB200Ranker), thresholds {'shared over NVLink peer memory' if sharded.local.sharing else 'not shared'}, "
                "NCCL all-to-all by user slice + certifying merge of the slice + all-gather of the merged slices" if n_ugroups == 1 else
                f"users sharded over {world} GPU(s), NCCL all-gather of the results" if n_ishards == 1 else
                f"grid: {n_ishards} item shards x {n_ugroups} user groups, NCCL all-gather + merge per user group, all-gather of the results"
            ),
            "l2": "inputs larger than L2 (16-bit item shard %.0f MB + users %.0f MB per step)"
            % (n_loc * info["d_pad"] * 2 / 1e6, n_loc_users * info["d_pad"] * 2 / 1e6),
            "engine": {kk: st0.get(kk) for kk in ("path", "k_cand", "n_splits", "epi_warps", "wide", "n_tc_launches", "n_fallback_rows",
                                                   "n_exact_rows", "n_uncertified_rows")},
            "engine_ms_last_step": {kk: timed_stats[-1].get(kk) for kk in ("ms_total", "ms_main", "ms_select", "ms_h2d", "ms_d2h")} if timed_stats else {},
            "device": info["device_name"],
        },
        "e2e": e2e,
        "model_recommend": model_reco,
        "gpu_launches": int(timed_launches),
        "ms_steps_rank0": step_ms_log[0] if step_ms_log else None,
        "clocks": clocks,
        "roofline": roof,
        "cpu_baseline": cpu,
        "parity": parity,
    }
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
