#!/usr/bin/env python
"""bench.py — recommend_user users/sec (all-items top-K) on synthetic C2:
TwoTower-style retrieval, 10 M users x 1 M items, embed 64, top-100, consumed filter on.

    python bench.py --gpus 1 --steps 20 --warmup 3            # this repo's CUDA path
    python bench.py --impl reference --steps 3 --warmup 1     # reference algorithm on host cores
    python bench.py --steps 5 --dump-outputs DIR              # + the last timed step's ids as DIR/*.npy
    torchrun --nproc-per-node N ... bench.py --gpus N ...     # one rank per GPU (users sharded)

One JSON line on rank 0 (see the driver contract).  A "step" = one recommend call for a batch of
`--batch` distinct users per rank (device leg: launches of <= 32768 users; host seam: <= 16384, so that the
D2H of a chunk and the id conversion of the next overlap kernels).  `value` is device-resident
(user ids already in HBM, result left in HBM); `e2e` goes through the reference-facing seam
`recommend_from_embedding(model, <python list of user ids>, n_rec, ...)` with HOST ids in and a
fresh HOST int64[B, n_rec] array out.  For N > 1 the same run also times the two paths that DO have
a collective (sharded LightGCN propagation, row-sharded embedding lookup) under `secondary`.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED_U, SEED_I, SEED_C, SEED_Q = 1, 2, 3, 4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--users", type=int, default=10_000_000)
    ap.add_argument("--items", type=int, default=1_000_000)
    ap.add_argument("--dim", type=int, default=64)
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--topk", type=int, default=100)
    ap.add_argument("--mean-consumed", type=float, default=50.0)
    ap.add_argument("--cpu-users", type=int, default=64, help="users per CPU-baseline call")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--path", default="auto", choices=["auto", "exact"])
    ap.add_argument("--no-secondary", action="store_true", help="skip the collective legs at N > 1")
    ap.add_argument("--config", default="c2", choices=["c1", "c2", "c3", "c4", "c5"],
                    help="BASELINE.json configuration: c2 (default, the headline line); c1/c3/c4/c5 = the other "
                         "configurations on one GPU (librecommender_b200/bench_configs.py)")
    ap.add_argument("--epi-warps", type=int, default=0, help="tuning: epilogue warps per TMEM quadrant (2|3)")
    ap.add_argument("--pre-coef", type=float, default=0.0, help="tuning: speculative rank coefficient")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last timed step of rank 0 (device leg "
                         "and end-to-end leg) as DIR/<name>.npy in float64, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config != "c2"):
        ap.error("--dump-outputs writes the results of the CUDA path of --config c2 (--impl b200)")
    return args


# --------------------------------------------------------------------------------------------
# synthetic catalogue (SURVEY.md §8d, C2) — generated on the device, seeds fixed
# --------------------------------------------------------------------------------------------
def make_tables(args, device):
    import torch

    def table(rows, seed):
        g = torch.Generator(device=device)
        g.manual_seed(seed)
        t = torch.empty((rows, args.dim), dtype=torch.float32, device=device)
        step = 1 << 20
        for r0 in range(0, rows, step):
            r1 = min(rows, r0 + step)
            x = torch.randn((r1 - r0, args.dim), generator=g, device=device, dtype=torch.float32)
            t[r0:r1] = x / x.norm(dim=1, keepdim=True)       # TwoTower norm_embed=True
        return t

    U = table(args.users + 1, SEED_U)
    I = table(args.items + 1, SEED_I)
    return U, I


def make_consumed_csr(args, device):
    """c_u ~ min(Poisson(mean), 500) items per user, Zipf(1.0) over a fixed random permutation of
    the items, duplicates inside a user removed (=> sorted unique lists)."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(SEED_C)
    n_users, N = args.users, args.items
    counts = torch.poisson(torch.full((n_users,), float(args.mean_consumed), device=device), generator=g)
    counts = counts.clamp_(max=min(500, N // 4)).to(torch.int64)
    w = 1.0 / torch.arange(1, N + 1, device=device, dtype=torch.float64)
    cdf = torch.cumsum(w, 0)
    cdf = (cdf / cdf[-1]).to(torch.float32)
    perm = torch.randperm(N, generator=g, device=device)
    shift = max(1, (N - 1).bit_length())
    keys = []
    chunk_users = 1 << 20
    for u0 in range(0, n_users, chunk_users):
        u1 = min(n_users, u0 + chunk_users)
        c = counts[u0:u1]
        tot = int(c.sum())
        owner = torch.repeat_interleave(torch.arange(u0, u1, device=device), c)
        r = torch.rand(tot, generator=g, device=device)
        rank = torch.searchsorted(cdf, r).clamp_(max=N - 1)
        item = perm[rank]
        keys.append(torch.unique((owner << shift) | item))    # sorted, de-duplicated
    key = torch.cat(keys)
    owner = key >> shift
    idx = (key & ((1 << shift) - 1)).to(torch.int32)
    cnt = torch.bincount(owner, minlength=n_users)
    indptr = torch.zeros(n_users + 1, dtype=torch.int64, device=device)
    indptr[1:] = torch.cumsum(cnt, 0)
    return indptr, idx


def make_batches(args, rank, n):
    rng = np.random.default_rng(SEED_Q + 1000 * rank)
    return [rng.choice(args.users, size=args.batch, replace=False).astype(np.int64) for _ in range(n)]


DUMP_BYTES = 64 * 10**6


def dump_outputs(dirname, arrays):
    """Write each [B, ...] result as <dirname>/<name>.npy in float64 (item ids are exact there).  Above
    DUMP_BYTES in all, every array keeps the same fixed, seeded sample of rows (rows.npy lists them)."""
    host = {k: np.asarray(v.cpu().numpy() if hasattr(v, "cpu") else v, dtype=np.float64) for k, v in arrays.items()}
    if sum(a.nbytes for a in host.values()) > DUMP_BYTES:
        n = next(iter(host.values())).shape[0]
        row_bytes = sum(a[0].nbytes for a in host.values()) + 8          # + its entry in rows.npy
        keep = (DUMP_BYTES - 4096) // row_bytes                          # 4096: room for the .npy headers
        rows = np.sort(np.random.default_rng(SEED_Q + 2000).choice(n, keep, replace=False))
        host = {k: a[rows] for k, a in host.items()}
        host["rows"] = rows.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(dirname, f"{k}.npy"), a)


# --------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi fields through NVML)
# --------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {
        0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
        0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
        0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting",
    }

    def __init__(self, index):
        self.samples, self.reasons, self.stop_flag, self.ok = [], set(), False, False
        self.sm_max = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            pass
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop_flag:
            try:
                self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
                mask = int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        if self.ok:
            self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.ok:
            self.th.join(timeout=1.0)
        med = int(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------
# CPU baseline: the reference's algorithm (oracle port, same numpy primitives) on host cores
# --------------------------------------------------------------------------------------------
def _reference_fn():
    """The reference's OWN recommend_from_embedding (mounted /root/reference or the byte-identical
    staged copy oracle/_ref) when present -> kind "reference"; else the oracle port -> kind "port"."""
    try:
        from oracle.ref_loader import load_reference, reference_available, reference_kind

        if reference_available():
            load_reference()
            from libreco.recommendation import recommend_from_embedding as ref_fn

            return ref_fn, "reference", reference_kind()
    except Exception as e:   # pragma: no cover
        print(f"[bench] reference import failed ({e!r}); timing the oracle port", file=sys.stderr)
    return None, "port", "absent"


def cpu_baseline_run(args, U_rows_fn, I_host, consumed_fn, seconds, users_per_call, max_calls=None,
                     keep_first=None):
    """Time the reference algorithm on host cores.  Users are renumbered 0..n-1 for the call (the
    reference indexes ``user_embeddings[user_ids]`` and ``model.user_consumed[user]``)."""
    import types

    from oracle.ranking import recommend_from_embedding_numpy_path

    ref_fn, kind, _ = _reference_fn()
    rng = np.random.default_rng(SEED_Q + 77)
    done_users, t_total, calls = 0, 0.0, 0
    per_call = []
    while True:
        users = rng.choice(args.users, size=users_per_call, replace=False).astype(np.int64)
        rows = U_rows_fn(users)
        consumed = consumed_fn(users)
        local = list(range(users_per_call))
        consumed_local = {j: consumed[int(u)] for j, u in enumerate(users.tolist()) if int(u) in consumed}
        model = types.SimpleNamespace(task="ranking", n_items=args.items, n_users=users_per_call,
                                      user_consumed=consumed_local)
        t0 = time.perf_counter()
        if ref_fn is not None:
            ids = ref_fn(model, local, args.topk, rows, I_host, True, False)
        else:
            ids = recommend_from_embedding_numpy_path(local, args.topk, rows, I_host, args.items,
                                                      consumed_local, True)
        dt = time.perf_counter() - t0
        assert ids.shape == (users_per_call, args.topk)
        if keep_first is not None and not keep_first:
            keep_first.update(users=users, ids=np.asarray(ids), rows=rows, consumed=consumed)
        calls += 1
        if calls > 1 or max_calls == 1:   # first call is the warm-up unless only one is allowed
            t_total += dt
            done_users += users_per_call
            per_call.append(dt)
        if (max_calls and calls >= max_calls + (0 if max_calls == 1 else 1)) or t_total >= seconds:
            break
    return done_users / max(t_total, 1e-9), per_call, kind


def host_views(U, I, indptr, idx):
    """Callables that fetch the host-side data the CPU arm needs for a user sample."""
    import torch

    I_host = I.cpu().numpy()

    def rows(users):
        return U[torch.as_tensor(users, device=U.device)].cpu().numpy()

    def consumed(users):
        ut = torch.as_tensor(users, device=indptr.device)
        b, e = indptr[ut].cpu().numpy(), indptr[ut + 1].cpu().numpy()
        out = {}
        for u, bb, ee in zip(users.tolist(), b.tolist(), e.tolist()):
            if ee > bb:
                out[u] = idx[bb:ee].cpu().numpy().tolist()
        return out

    return I_host, rows, consumed


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    import torch

    distributed = world > 1
    if args.impl == "reference" and rank != 0:
        return 0                                   # rank 0 alone runs the CPU arm
    if args.impl == "reference" and not torch.cuda.is_available():
        device = torch.device("cpu")               # the CPU arm does not need a GPU (synthetic tables made on the host)
    else:
        torch.cuda.set_device(local_rank)
        device = torch.device("cuda", local_rank)
    if args.config != "c2":
        if rank != 0 or args.impl != "b200":
            return 0
        from librecommender_b200 import bench_configs

        print(json.dumps(bench_configs.CONFIGS[args.config](args, ROOT, ClockSampler(local_rank))))
        return 0
    if distributed and args.impl == "b200":
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=device)

    workload = (f"C2 TwoTower retrieval: {args.users} users x {args.items} items, embed {args.dim}, "
                f"top-{args.topk}, filter_consumed, batch {args.batch} users/step/GPU")
    config = {"workload": workload, "users": args.users, "items": args.items, "embed": args.dim,
              "n_rec": args.topk, "batch_per_gpu": args.batch, "global_batch": args.batch * world,
              "users_per_launch": {"device_leg": min(args.batch, 32768), "e2e_leg": min(args.batch, 16384)},
              "parallelism": f"users sharded x{world}, item table replicated, no data-path collective",
              "l2": "inputs larger than L2 (item table 256 MB fp32 + 128 MB fp16, user table 2.56 GB)",
              "device_leg": "2 steps in flight on one stream (async handle, check of step i after enqueue of i+1)",
              "e2e_leg": "synchronous reference-facing seam recommend_from_embedding(model, python list of ids, ...): "
                         "list -> H2D ids, kernels, D2H ids + status (side stream, chunk-pipelined), one sync, "
                         "fresh host int64 array",
              "cpu_arm": f"{args.cpu_users} users per call (np.tile in the reference needs 8*B*N bytes: "
                         f"B = {args.batch} would need {8 * args.batch * args.items / 1e9:.0f} GB), same catalogue"}

    U, I = make_tables(args, device)
    indptr, idx = make_consumed_csr(args, device)
    if device.type == "cuda":
        torch.cuda.synchronize()

    if args.impl == "reference":
        try:   # torchrun exports OMP_NUM_THREADS=1: the CPU arm must still use every host thread
            from threadpoolctl import threadpool_limits

            threadpool_limits(limits=os.cpu_count())
        except Exception:
            pass
        I_host, rows_fn, cons_fn = host_views(U, I, indptr, idx)
        ncalls = max(1, args.steps)
        for _ in range(max(0, min(args.warmup, 2))):
            cpu_baseline_run(args, rows_fn, I_host, cons_fn, 0.0, args.cpu_users, max_calls=1)
        ups, per_call, kind = cpu_baseline_run(args, rows_fn, I_host, cons_fn, 1e9, args.cpu_users,
                                               max_calls=ncalls if ncalls > 1 else 1)
        ms = 1e3 * float(np.mean(per_call))
        cores = os.cpu_count()
        what = ("the reference's own libreco.recommendation.recommend_from_embedding (unmodified, "
                "oracle/_ref or /root/reference)" if kind == "reference" else
                "oracle port of recommend.py:57-78 + ranking.py:10-78")
        line = {
            "impl": "reference", "metric": "recommend_user users/sec (all-items top-K)", "value": ups,
            "unit": "users/s", "n_gpus": args.gpus, "steps": len(per_call), "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": ups, "unit": "users/s", "cores": cores, "kind": kind,
                             "sample": f"{args.cpu_users} users per call x {len(per_call)} calls, full "
                                       f"{args.items}-item catalogue ({what}, numpy/OpenBLAS on all host threads)"},
            "e2e": {"value": ups, "unit": "users/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ this repo's CUDA path
    import types

    from librecommender_b200 import _lib
    from librecommender_b200 import recommend_from_embedding
    from librecommender_b200.consumed import ConsumedCSR
    from librecommender_b200.engine import scorer_for

    if args.epi_warps or args.pre_coef:
        _lib.check(_lib.lib.b200_recommend_embed_tune(args.epi_warps, args.pre_coef))
    csr = ConsumedCSR.from_device_tensors(indptr, idx)
    # the object the reference's seam receives: `model` with n_items / n_users / task / user_consumed,
    # and the two embedding tables (device-resident here, as TwoTower.set_embeddings leaves them)
    model = types.SimpleNamespace(task="ranking", n_items=args.items, n_users=args.users, user_consumed=csr)
    scorer = scorer_for(model, U, I)
    plan = scorer.fused_plan(args.batch, args.topk)
    n_batches = args.warmup + args.steps
    batches_np = make_batches(args, rank, n_batches)
    batches_list = [b.tolist() for b in batches_np]            # what the reference passes: a python list
    batches_d = [torch.from_numpy(b).to(device) for b in batches_np]
    torch.cuda.synchronize()

    def barrier():
        if distributed:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if not distributed:
            return ms
        import torch.distributed as dist

        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident leg ------------------------------------------------------------
    for i in range(args.warmup):
        scorer.recommend_device(batches_d[i], args.topk, True, False, args.path)
    barrier()
    scorer.events = []
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    # two steps in flight: step i+1 is enqueued before step i is checked (rows the fused path
    # could not prove are repaired in .result(); every check happens inside the timed region)
    out, pending, fallback_dev = None, None, 0
    for i in range(args.warmup, n_batches):
        nxt = scorer.recommend_device_async(batches_d[i], args.topk, True, False, args.path)
        if pending is not None:
            out = pending.result()
            fallback_dev += scorer.last_fallback_rows
        pending = nxt
    out = pending.result()
    fallback_dev += scorer.last_fallback_rows
    e1.record()
    barrier()
    launches = _lib.launch_count() - launches0
    dev_ms = max_over_ranks(e0.elapsed_time(e1))
    sweep_ms = [a.elapsed_time(b) for a, b in scorer.events]
    scorer.events = None
    value = world * args.batch * args.steps / (dev_ms * 1e-3)

    # ---- end-to-end leg: python list of host ids in, fresh host ids out ---------------------
    for i in range(min(args.warmup, 2)):
        recommend_from_embedding(model, batches_list[i], args.topk, U, I, True, False)
    barrier()
    e0.record()
    res, fallback_e2e = None, 0
    for i in range(args.warmup, n_batches):
        res = recommend_from_embedding(model, batches_list[i], args.topk, U, I, True, False)
        fallback_e2e += scorer.last_fallback_rows
    e1.record()
    barrier()
    clocks = sampler.stop()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = world * args.batch * args.steps / (e2e_ms * 1e-3)
    assert res.shape == (args.batch, args.topk) and res.dtype == np.int64 and (res >= 0).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"device_ids": out, "e2e_ids": res})

    # ---- parity of one TIMED batch, outside the timed region: fused result vs the exact path ----
    last = batches_d[n_batches - 1]
    n_chk = min(args.batch, 8192)
    exact_ids = scorer.recommend_exact(last[:n_chk], args.topk, True, False).cpu().numpy()
    parity = {"checked_rows": int(n_chk),
              "e2e_ids_equal_exact_path": float((res[:n_chk] == exact_ids).all(axis=1).mean()),
              "device_ids_equal_exact_path": float((out[:n_chk].cpu().numpy() == exact_ids).all(axis=1).mean())}

    run_secondary = distributed and not args.no_secondary
    if distributed and not run_secondary:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if rank != 0 and not run_secondary:
        return 0

    if rank != 0:            # other ranks only take part in the collective legs
        finish_with_secondary({}, run_secondary, rank, world, device, max_over_ranks, barrier)
        return 0

    # ---- roofline of the dominant kernel (tcgen05 sweep) ----------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    roofline = None
    if sweep_ms:
        import librecommender_b200.engine as _eng

        rows_per_launch = min(args.batch, _eng.FUSED_ROWS_PER_CALL)      # device leg: users per b200_recommend_embed launch
        flops = 2.0 * args.dim * args.items * rows_per_launch          # per launch (SURVEY §8d: 2*d*N per user)
        avg_ms = float(np.mean(sweep_ms))
        achieved = flops / (avg_ms * 1e-3) / 1e12
        peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "sweep_traffic.json")))
            # the capture is of a 16 384-user launch: scale to this run's users per launch (records and item-table
            # passes both grow linearly with the user tiles)
            traffic = tr["dram_bytes_per_launch"] * rows_per_launch / float(tr.get("users_per_launch", 16384))
        except Exception:
            pass
        roofline = {"bound": "tensor", "kernel": "b200::tc::sweep_kernel (PRE + guess + MAIN)", "achieved": achieved,
                    "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured; fp16 runs at the bf16 rate)"
                    if peaks else "fallback 1400 (of fallback)",
                    "traffic": traffic, "avg_launch_ms": avg_ms, "launches_timed": len(sweep_ms),
                    "rows_per_launch": rows_per_launch,
                    "share_of_step": avg_ms * len(sweep_ms) / max(dev_ms, 1e-9) if not distributed else None}

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        I_host, rows_fn, cons_fn = host_views(U, I, indptr, idx)
        first = {}
        ups, per_call, kind = cpu_baseline_run(args, rows_fn, I_host, cons_fn, args.cpu_seconds, args.cpu_users,
                                               keep_first=first)
        what = ("the reference's own recommend_from_embedding, unmodified" if kind == "reference"
                else "oracle port of the reference's numpy path")
        cpu = {"value": ups, "unit": "users/s", "cores": os.cpu_count(), "kind": kind,
               "sample": f"{args.cpu_users} users per call x {len(per_call)} calls against the full "
                         f"{args.items}-item catalogue ({what})"}
        # the CPU arm's answer for its first call doubles as the checker of the CUDA path on those users
        from oracle.ranking import near_tie_mask

        got = recommend_from_embedding(model, first["users"].tolist(), args.topk, U, I, True, False)
        full = first["rows"] @ I_host[:args.items].T
        parity["cpu_reference_rows"] = int(len(first["users"]))
        parity["ids_equal_cpu_reference"] = float((got == first["ids"]).mean())
        parity["ids_equal_cpu_reference_outside_near_ties"] = bool(
            near_tie_mask(first["ids"], got, full, 1e-6).all())

    line = {
        "metric": "recommend_user users/sec (all-items top-K)", "value": value, "unit": "users/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 scores (fp16 tensor-core candidate pass + exact fp32 re-score)",
        "data": "synthetic", "config": config, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "users/s", "h2d_bytes_per_step": args.batch * 8,
                "d2h_bytes_per_step": args.batch * args.topk * 8 + args.batch * 4,
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
        "path": args.path, "plan": plan,
        "fallback_rows": {"device_leg": int(fallback_dev), "e2e_leg": int(fallback_e2e),
                          "rows_per_leg": int(args.batch * args.steps)},
        "parity": parity,
    }
    finish_with_secondary(line, run_secondary, rank, world, device, max_over_ranks, barrier)
    return 0


def finish_with_secondary(line, run_secondary, rank, world, device, max_over_ranks, barrier):
    """Print the ONE JSON line (rank 0).  At N > 1 the collective legs run first, under a watchdog: if
    they do not finish in time (a hung exchange must not cost the primary measurement) the line is
    printed with the time-out recorded and every rank exits."""
    if not run_secondary:
        print(json.dumps(line))
        return
    import torch.distributed as dist

    done = threading.Event()
    deadline_s = float(os.environ.get("B200_SECONDARY_DEADLINE_S", "420"))

    def watchdog():
        if not done.wait(deadline_s):
            if rank == 0:
                line["secondary"] = {"error": f"collective legs exceeded {deadline_s:.0f} s"}
                print(json.dumps(line), flush=True)
            os._exit(0)

    threading.Thread(target=watchdog, daemon=True).start()
    try:
        from librecommender_b200 import bench_collectives

        secondary = bench_collectives.run(rank, world, device, max_over_ranks, barrier)
    except Exception as e:   # the primary line must survive
        secondary = {"error": repr(e)[:400]}
    done.set()
    if rank == 0:
        line["secondary"] = secondary
        print(json.dumps(line), flush=True)
    try:
        dist.barrier()
        dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    sys.exit(main())
