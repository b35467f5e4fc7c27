#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path: filter -> hash-aggregate.

Workload (BASELINE.json configs[1], SURVEY.md 8d row 2):
    SELECT k, sum(v), count(v), avg(x) FROM t WHERE v % 3 = 0 GROUP BY k
    t = 1e9 rows, k Int64 uniform [0,1e6), v Int64 uniform [-2^31,2^31), x Float64 integer-valued [0,2^20)
    synthetic, counter-based generator (dbx_synth_fill / orc_synth_fill, seeds 42/43/44).

One "step" = one full query over the 1e9-row batch: table reset, fused filter+partial
aggregation, final merge, result materialisation.

  value  rows/s with the three columns already resident in HBM (CUDA events on the operator's
         stream; includes table re-initialisation and result finalisation, excludes nothing)
  e2e    the same query through the public operator API with HOST (pinned) columns pushed in
         blocks: host->device copies and the device->host copy of the result are inside the
         timed region
  roofline  the fused kernel alone: 24 algorithmic bytes per row / its CUDA-event duration
            against the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline  the CPU oracle (reference-algorithm restatement, OpenMP) on a bounded sample

`--impl reference` times the CPU oracle on the host cores (the Rust reference cannot be
built in this image: no cargo/rustc).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rows/sec filter->hash-agg (sum,count,avg GROUP BY 1e6 int64 keys) over int64/float64 columns"
SEEDS = (42, 43, 44)
N_KEYS = 1_000_000
BYTES_PER_ROW = 24.0  # three 8-byte columns, each read exactly once (SURVEY.md 8d)
KERNEL_NAME = "filter_group_agg_kernel<3,FAST=1,INDIRECT=0,BULK=0>"
KERNEL_NAME_JIT = "dbx_jit_agg_fast (filter_group_agg_body<3,FAST=1> compiled for this plan by NVRTC at operator creation)"


def ncu_traffic():
    """dram read+write bytes of ONE 2^28-row launch of the fused kernel, from the committed ncu --set full capture."""
    p = os.path.join(ROOT, "profiles", "r02_agg_kernel_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d["dram_bytes_per_launch"], d["note"]
    return None, "no ncu capture of this kernel committed yet"



def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi during the timed region."""

    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index
        self.marks = []

    def mark(self):
        """Remember how many samples had arrived (called at the start and end of the timed region)."""
        self.marks.append(len(self.rows))

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows, window = self.rows, "warm-up + timed region (no sample fell inside the timed region alone)"
        if len(self.marks) >= 2 and self.marks[1] > self.marks[0]:
            rows, window = self.rows[self.marks[0]:self.marks[1]], "timed region"
        self.window = window
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for nm, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


DUMP_BYTES = 63 << 20  # array data of --dump-outputs; the rest of 64 MB is left for the .npy headers


def download_block(L, dev, blk):
    """Host copies (numpy) of the columns of a library-owned DEVICE result block; NULLs become NaN."""
    import numpy as np
    from databend_b200 import lib
    from databend_b200.block import np_dtype
    cols = []
    for i in range(blk.num_cols):
        c = blk.cols[i]
        a = np.empty(c.len, dtype=np_dtype(c.dtype))
        if c.len:
            lib.check(L.dbx_memcpy_d2h(dev, a.ctypes.data, c.data, a.nbytes))
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        if c.validity and c.len:
            vb = np.empty((c.validity_bit_offset + c.len + 7) // 8, dtype=np.uint8)
            lib.check(L.dbx_memcpy_d2h(dev, vb.ctypes.data, c.validity, vb.nbytes))
            valid = np.unpackbits(vb, bitorder="little")[c.validity_bit_offset:c.validity_bit_offset + c.len]
            a[valid == 0] = np.nan
        cols.append(a)
    return cols


def write_outputs(out_dir, tables):
    """--dump-outputs: `tables` maps a table to {name: array}; the arrays of one table share their
    first dimension.  Written as <out_dir>/<name>.npy in float32/float64.  When everything together
    exceeds DUMP_BYTES, every table keeps the same fraction of its rows, chosen by a fixed seed, so
    two builds run with the same arguments write the same rows."""
    import numpy as np
    total = sum(a.nbytes for t in tables.values() for a in t.values())
    frac = min(1.0, DUMP_BYTES / total) if total else 1.0
    os.makedirs(out_dir, exist_ok=True)
    for cols in tables.values():
        n = len(next(iter(cols.values())))
        m = int(n * frac)
        keep = np.sort(np.random.default_rng(0).choice(n, m, replace=False)) if m < n else slice(None)
        for name, a in cols.items():
            np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a[keep]))


def make_query():
    from databend_b200 import expr as E
    from databend_b200.transforms import AggregatorParams
    params = AggregatorParams([0], [("sum", 1), ("count", 1), ("avg", 2)])
    filt = E.eq(E.col(1) % E.lit(3), E.lit(0))
    return params, filt


# ---------------------------------------------------------------------------------- reference arm
def run_reference(args):
    """CPU arm: the oracle port on all host threads, each step a bounded sample of the workload."""
    import numpy as np
    from databend_b200.block import Column, DataBlock
    from oracle import oracle as orc
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = len(os.sched_getaffinity(0))  # torchrun pins OMP_NUM_THREADS=1: ask for every host core explicitly
    n = args.cpu_rows
    params, filt = make_query()
    k = orc.synth_fill(0, SEEDS[0], N_KEYS, 0, n)
    v = orc.synth_fill(1, SEEDS[1], 0, 0, n)
    x = orc.synth_fill(2, SEEDS[2], 20, 0, n)
    blk = DataBlock([Column.from_data(k), Column.from_data(v), Column.from_data(x)])
    cp = params.to_c(filt)
    for _ in range(args.warmup):
        orc.filter_group_agg(blk, cp, threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        orc.filter_group_agg(blk, cp, threads=threads)
    dt = (time.perf_counter() - t0) / args.steps
    val = n / dt
    sample = f"{n} rows of the same synthetic columns per step (reference-algorithm CPU restatement in C/OpenMP; the Rust reference cannot be built here)"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": "filter+hash-agg sum/count/avg GROUP BY 1e6 int64 keys, WHERE v%3=0", "rows": n},
        "cpu_baseline": {"value": val, "unit": "rows/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if not args.no_knn:  # second half of the metric, on the same host cores: row-wise cosine_distance + top-k
        from databend_b200 import abi
        sn, sq, dim, kk = min(args.knn_rows, args.knn_cpu_rows), 8, args.knn_dim, args.knn_k
        rng = np.random.default_rng(0)
        c = rng.standard_normal((sn, dim)).astype(np.float32)
        qs = rng.standard_normal((sq, dim)).astype(np.float32)
        orc.distance_rows(abi.DIST_COSINE, c, qs[0], threads=threads)
        t0 = time.perf_counter()
        for i in range(sq):
            d = orc.distance_rows(abi.DIST_COSINE, c, qs[i], threads=threads)
            np.argpartition(d, min(kk, sn - 1))[:kk]
        dt_k = time.perf_counter() - t0
        line["knn"] = {"metric": "kNN QPS @768d (cosine_distance, brute force, exact top-k)", "impl": "reference",
                       "value": sq / dt_k * sn / args.knn_rows, "unit": "queries/s",
                       "cpu_baseline": {"value": sq / dt_k * sn / args.knn_rows, "unit": "queries/s", "cores": threads, "kind": "port",
                                        "sample": f"{sq} queries x {sn} rows x {dim} dims, row-wise cosine_distance (oracle, OpenMP) + top-{kk}, scaled by {sn}/{args.knn_rows} rows"}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------- kNN leg
def run_knn(args, L, dev, rank, world, barrier):
    """configs[4]: cosine_distance brute-force kNN, corpus sharded by rows across ranks, queries
    replicated; per-rank top-k all-gathered and merged.  Returns the "knn" object of the JSON line
    and the (row ids, distances) of the last timed batch; (None, None) on ranks other than 0."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from databend_b200 import abi, lib
    from databend_b200.block import Column
    from databend_b200.transforms import DeviceBuffer
    from databend_b200.vector import VectorTopN

    n_total, dim, nq, k = args.knn_rows, args.knn_dim, args.knn_queries, args.knn_k
    r0, r1 = n_total * rank // world, n_total * (rank + 1) // world
    n = r1 - r0
    cbuf = DeviceBuffer(n * dim * 4, dev)
    lib.check(L.dbx_synth_fill(dev, 4, 42, 0, r0 * dim, n * dim, cbuf.ptr))
    qbuf = DeviceBuffer(nq * dim * 4, dev)
    lib.check(L.dbx_synth_fill(dev, 4, 43, 0, 0, nq * dim, qbuf.ptr))
    t0 = time.perf_counter()
    op = VectorTopN("cosine_distance", Column.device(abi.VEC_F32, n, cbuf.ptr, vec_dim=dim), dev)
    create_s = time.perf_counter() - t0
    q_dev = Column.device(abi.VEC_F32, nq, qbuf.ptr, vec_dim=dim)
    q_host = Column.vector(qbuf.download(np.float32, nq * dim).reshape(nq, dim))

    def search(q):
        if world == 1:
            return op.search(q, k)
        # per-rank top-k stays in HBM; ONE collective over [nq, k] global row ids and distance bits
        idx_t = torch.empty((nq, k), dtype=torch.int64, device=f"cuda:{dev}")
        d_t = torch.empty((nq, k), dtype=torch.float32, device=f"cuda:{dev}")
        op.search_into(q, k, idx_t.data_ptr(), d_t.data_ptr())
        t = torch.stack([idx_t + r0, d_t.view(torch.int32).to(torch.int64)])
        g = torch.empty((world,) + tuple(t.shape), dtype=torch.int64, device=f"cuda:{dev}")
        dist.all_gather_into_tensor(g, t)
        ai = g[:, 0].permute(1, 0, 2).reshape(nq, world * k)
        ad = g[:, 1].permute(1, 0, 2).reshape(nq, world * k).to(torch.int32).view(torch.float32)
        # merge: ascending (distance, row id); NaN last like OrderedFloat.  Ranks hold ascending row
        # ranges and every rank's list is ordered by (distance, row id), so ONE stable sort by
        # distance over the rank-major concatenation keeps ascending global row ids inside ties.
        key = torch.where(torch.isnan(ad), torch.full_like(ad, float("inf")), ad)
        o2 = torch.argsort(key, dim=1, stable=True)[:, :k]
        return ai.gather(1, o2).cpu().numpy(), ad.gather(1, o2).cpu().numpy()

    def timed(q, steps, warmup):
        for _ in range(warmup):
            search(q)
        barrier()
        gemm = []
        t0 = time.perf_counter()
        for _ in range(steps):
            res = search(q)
            gemm.append(op.last_gemm_ms()[0])
        barrier()
        ms = (time.perf_counter() - t0) * 1e3 / steps
        t = torch.tensor([ms, sum(gemm) / len(gemm)], dtype=torch.float64, device=f"cuda:{dev}")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist(), res

    launches0 = L.dbx_kernel_launch_count()
    (ms_dev, gemm_ms), res = timed(q_dev, args.steps, args.warmup)
    launches = L.dbx_kernel_launch_count() - launches0
    (ms_host, _), _ = timed(q_host, max(1, min(args.steps, 3)), 1)
    stats = op.stats()
    op.close()
    if rank != 0:
        return None, None
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, src = 1400.0, "fallback (B200_PROFILING.md sustained)"
    if os.path.exists(p):
        with open(p) as f:
            peak, src = json.load(f).get("bf16_tflops_sustained", 1400.0), "measured sustained cuBLAS bf16 (MEASURED_PEAKS.json)"
    flop = 2.0 * nq * n * dim  # per rank and batch: the similarity GEMM (SURVEY 8d row 5)
    achieved = flop / (gemm_ms * 1e-3) / 1e12
    out = {
        "metric": "kNN QPS @768d (cosine_distance, brute force, exact top-k)", "value": nq / (ms_dev * 1e-3), "unit": "queries/s",
        "ms_per_batch": ms_dev, "n_gpus": world, "scaling": "strong", "dtype": "bf16 candidate GEMM (f32 accumulate) + exact f32 re-rank",
        "config": {"workload": "configs[4]", "corpus_rows": n_total, "rows_per_gpu": n, "dim": dim, "queries": nq, "k": k,
                   "data": "synthetic N(0,1), device-generated", "create_s": create_s,
                   "parallelism": f"corpus rows x{world}" + ("" if world == 1 else " + all-gather of per-GPU top-k")},
        "gpu_launches_per_batch": int(launches // max(1, args.steps)),
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "traffic": None, "kernel": f"knn_gemm_filter_kernel<{stats['cluster']}>", "kernel_ms": gemm_ms,
                     "flop_per_launch_set": flop, "peak_source": src},
        "certified_queries": stats["certified"], "exact_fallback_queries": stats["exact_fallback"],
        "e2e": {"value": nq / (ms_host * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": nq * dim * 4,
                "d2h_bytes_per_step": nq * k * 12, "ms_per_batch": ms_host,
                "timing": "host wall clock around VectorTopN.search() with HOST query vectors, max over ranks"},
    }
    if world == 1 and not args.no_cpu:
        from oracle import oracle as orc
        threads = len(os.sched_getaffinity(0))
        sn, sq = min(n_total, 1_000_000), 8
        rng = np.random.default_rng(0)
        c = rng.standard_normal((sn, dim)).astype(np.float32)
        qs = rng.standard_normal((sq, dim)).astype(np.float32)
        orc.distance_rows(abi.DIST_COSINE, c, qs[0], threads=threads)
        t0 = time.perf_counter()
        for i in range(sq):
            d = orc.distance_rows(abi.DIST_COSINE, c, qs[i], threads=threads)
            np.argpartition(d, k)[:k]
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": sq / dt * sn / n_total, "unit": "queries/s", "cores": threads, "kind": "port",
                               "sample": f"{sq} queries x {sn} rows, row-wise cosine_distance (oracle, OpenMP) + top-k, scaled by {sn}/{n_total} rows"}
    return out, res

# ---------------------------------------------------------------------------------- GPU arm
def verify_result(out_block, dev, rank, world, cols, n, keys_total, torch, dist):
    """Full-scale check OUTSIDE the timed region: every group of this rank's result block
    (host columns [sum(v), count(v), avg(x), k]) against an independent recomputation of the whole
    query with torch index ops on the same device columns (bincount / index_add_ per key, all-reduced
    across ranks), plus — rank 0 — the CPU oracle on every row of a key subsample.  Returns a dict."""
    import numpy as np
    from databend_b200 import abi
    kd, vd, xd = cols

    def dev_tensor(ptr, dtype):
        # wrap the library-owned device column without copying (torch only as the checker)
        class _Holder:
            pass
        h = _Holder()
        h.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i8" if dtype == torch.int64 else "<f8", "data": (ptr, False), "version": 2}
        return torch.as_tensor(h, device=f"cuda:{dev}")

    k_t, v_t, x_t = dev_tensor(kd, torch.int64), dev_tensor(vd, torch.int64), dev_tensor(xd, torch.float64)
    cnt = torch.zeros(keys_total, dtype=torch.int64, device=f"cuda:{dev}")
    sv = torch.zeros(keys_total, dtype=torch.int64, device=f"cuda:{dev}")
    sx = torch.zeros(keys_total, dtype=torch.float64, device=f"cuda:{dev}")
    step = 1 << 27
    sub_keys = 997  # oracle subsample: every row whose key is < sub_keys
    sub_rows = []
    for lo in range(0, n, step):
        hi = min(n, lo + step)
        kk, vv, xx = k_t[lo:hi], v_t[lo:hi], x_t[lo:hi]
        m = torch.remainder(vv, 3) == 0  # v % 3 = 0 does not depend on the sign convention of %
        ks = kk[m]
        cnt += torch.bincount(ks, minlength=keys_total)
        sv.index_add_(0, ks, vv[m])  # int64 wrapping add
        sx.index_add_(0, ks, xx[m])  # integer-valued < 2^20: exact in any order
        sm = kk < sub_keys
        sub_rows.append(torch.stack([kk[sm], vv[sm], xx[sm].view(torch.int64)]).cpu())
    if world > 1:
        dist.all_reduce(cnt)
        dist.all_reduce(sv)
        dist.all_reduce(sx)
    # this rank's groups against the expectation
    g_k = torch.from_numpy(out_block.columns[3].values().astype(np.int64)).to(f"cuda:{dev}")
    g_sv = torch.from_numpy(out_block.columns[0].values().view(np.int64).copy()).to(f"cuda:{dev}")
    g_cnt = torch.from_numpy(out_block.columns[1].values().astype(np.int64)).to(f"cuda:{dev}")
    g_avg = torch.from_numpy(out_block.columns[2].values().copy()).to(f"cuda:{dev}")
    bad = int((g_cnt != cnt[g_k]).sum() + (g_sv != sv[g_k]).sum() + (g_avg != sx[g_k] / cnt[g_k].to(torch.float64)).sum())
    dup = int(g_k.numel() - torch.unique(g_k).numel())
    t = torch.tensor([g_k.numel(), bad, dup, int(g_cnt.sum())], dtype=torch.int64, device=f"cuda:{dev}")
    if world > 1:
        dist.all_reduce(t)
    groups_total, bad_total, dup_total, rows_selected = [int(v) for v in t.tolist()]
    expected_groups = int((cnt > 0).sum())
    res = {"groups": groups_total, "expected_groups": expected_groups, "mismatching_values": bad_total, "duplicate_keys": dup_total,
           "selected_rows": rows_selected, "expected_selected_rows": int(cnt.sum()),
           "how": "every group vs torch bincount/index_add_ over all rows (all-reduced across ranks)"}
    ok = groups_total == expected_groups and bad_total == 0 and dup_total == 0 and rows_selected == int(cnt.sum())
    # oracle on the key subsample (rank 0 gathers the subsample rows of every rank)
    sub = torch.cat(sub_rows, dim=1)
    if world > 1:
        sizes = [None] * world
        dist.all_gather_object(sizes, int(sub.shape[1]))
        pad = torch.zeros((3, max(sizes)), dtype=torch.int64, device=f"cuda:{dev}")
        pad[:, : sub.shape[1]] = sub.to(f"cuda:{dev}")
        gp = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(gp, pad)
        sub = torch.cat([g[:, :s_].cpu() for g, s_ in zip(gp, sizes)], dim=1)
        # every rank's owned subsample groups -> all ranks (rank 0 checks)
        mine = (g_k < sub_keys)
        loc = torch.stack([g_k[mine], g_sv[mine], g_cnt[mine], g_avg[mine].view(torch.int64)]).cpu()
        parts = [None] * world
        dist.all_gather_object(parts, loc.numpy())
        got = np.concatenate(parts, axis=1)
    else:
        mine = (g_k < sub_keys)
        got = torch.stack([g_k[mine], g_sv[mine], g_cnt[mine], g_avg[mine].view(torch.int64)]).cpu().numpy()
    if rank == 0:
        from databend_b200.block import Column, DataBlock
        from oracle import oracle as orc
        sn = sub.numpy()
        sblk = DataBlock([Column.from_data(np.ascontiguousarray(sn[0])), Column.from_data(np.ascontiguousarray(sn[1])),
                          Column.from_data(np.ascontiguousarray(sn[2]).view(np.float64))])
        params, filt = make_query()
        okeys, _, oaggs, _, _ = orc.filter_group_agg(sblk, params.to_c(filt), threads=len(os.sched_getaffinity(0)))
        oo = np.argsort(okeys[0].view(np.int64))
        go = np.argsort(got[0])
        same = (len(oo) == len(go) and np.array_equal(okeys[0].view(np.int64)[oo], got[0][go])
                and np.array_equal(oaggs[0].view(np.int64)[oo], got[1][go]) and np.array_equal(oaggs[1].view(np.int64)[oo], got[2][go])
                and np.array_equal(oaggs[2].view(np.int64)[oo], got[3][go]))
        res["oracle_subsample"] = {"keys_below": sub_keys, "rows": int(sn.shape[1]), "groups": int(len(oo)), "bit_exact": bool(same)}
        ok = ok and same
    res["ok"] = bool(ok)
    return res


def run_dbx(args):
    import gc
    import numpy as np
    import torch
    import torch.distributed as dist
    from databend_b200 import abi, build, lib
    from databend_b200.block import Column, DataBlock
    from databend_b200.exchange import all_to_all_rows
    from databend_b200.transforms import (DeviceBuffer, TransformFinalAggregate, TransformPartialAggregate, _block_from_c)

    build.build()
    L = lib.load()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    lib.require_device()
    dev = local_rank
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))

    total_rows = args.rows
    # strong scaling: the 1e9-row table is split into `world` contiguous row ranges
    r_begin = total_rows * rank // world
    r_end = total_rows * (rank + 1) // world
    n = r_end - r_begin
    params, filt = make_query()
    types = [abi.I64, abi.I64, abi.F64]

    bufs = [DeviceBuffer(n * 8, dev) for _ in range(3)]
    lib.check(L.dbx_synth_fill(dev, 0, SEEDS[0], args.keys, r_begin, n, bufs[0].ptr))
    lib.check(L.dbx_synth_fill(dev, 1, SEEDS[1], 0, r_begin, n, bufs[1].ptr))
    lib.check(L.dbx_synth_fill(dev, 2, SEEDS[2], 20, r_begin, n, bufs[2].ptr))
    dblock = DataBlock([Column.device(abi.I64, n, bufs[0].ptr), Column.device(abi.I64, n, bufs[1].ptr),
                        Column.device(abi.F64, n, bufs[2].ptr)], n)

    part = TransformPartialAggregate(params, types, filt, dev)
    fin = TransformFinalAggregate(params, types, dev)
    sp = C.c_void_p()
    lib.check(L.dbx_op_stream(part.handle, C.byref(sp)))
    part_stream = torch.cuda.ExternalStream(sp.value, device=dev)
    lib.check(L.dbx_op_stream(fin.handle, C.byref(sp)))
    fin_stream = torch.cuda.ExternalStream(sp.value, device=dev)

    use_peer = world > 1 and os.environ.get("DBX_EXCHANGE", "peer") == "peer"
    xchg = None
    if use_peer:
        from databend_b200.exchange import PeerExchange
        ok = 1
        try:
            xchg = PeerExchange(part, rank, world)
            xchg.connect()
        except Exception as e:  # e.g. no peer access between these GPUs: all ranks fall back together
            ok = 0
            print(f"[bench] rank {rank}: peer-memory exchange unavailable ({e}); using the NCCL all-to-all", file=sys.stderr)
        t_ok = torch.tensor([ok], dtype=torch.int32, device=f"cuda:{dev}")
        dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
        if int(t_ok.item()) == 0:
            if xchg is not None:
                xchg.close()
            xchg = None
            use_peer = False
    # Software pipelining across the two operators (they are different Processors in the reference
    # too): the partial operator starts scanning the next query's input while the final operator
    # still merges / materialises the current one.  Every query's full work stays inside the timed
    # region: the first timed step enqueues its own scan, the last one enqueues none.
    pipeline = use_peer and os.environ.get("DBX_BENCH_PIPELINE", "1") != "0"

    def exchange(out_mem):
        """partial -> (N>1: hash-partition + exchange) -> final merge (no host sync on the peer path)"""
        part.on_finish()
        if world == 1:
            fin.transform(part)
        elif use_peer:
            # rows go straight into the owners' HBM over NVLink (the same pass re-arms the partial's
            # table); a one-warp kernel waits for the sources' flags on the device, then the merge
            xchg.scatter(part)
            part.reset()
            xchg.merge(fin)
        else:
            rows_ptr = C.c_void_p()
            offs = (C.c_int64 * (world + 1))()
            rb = C.c_int32(0)
            lib.check(L.dbx_agg_partial_partition(part.handle, world, C.byref(rows_ptr), offs, C.byref(rb)), part.handle)
            row_bytes = rb.value
            send_counts = [offs[i + 1] - offs[i] for i in range(world)]
            total_send = offs[world]
            send = torch.empty(max(total_send, 1) * row_bytes, dtype=torch.uint8, device=f"cuda:{dev}")
            if total_send:
                lib.check(L.dbx_memcpy_d2d(dev, send.data_ptr(), rows_ptr.value, total_send * row_bytes))
            lib.check(L.dbx_device_free(dev, rows_ptr))
            recv, recv_counts = all_to_all_rows(send, send_counts, row_bytes)
            torch.cuda.current_stream().synchronize()
            fin.merge_rows(recv.data_ptr(), sum(recv_counts))

    state = {"queued": False}
    kernel_ms, phases, step_walls = [], [], []
    variant = part.kernel_variant()

    def step_device(input_blocks, out_mem, prefetch_next):
        """one query: scan (+filter+partial agg) -> exchange -> final -> result block"""
        if not state["queued"]:
            if not use_peer:
                part.reset()
            for b in input_blocks:
                part.transform(b)
        state["queued"] = False
        exchange(out_mem)
        if pipeline and prefetch_next:  # the next query's scan runs while this one is merged and materialised
            for b in input_blocks:
                part.transform(b)
            state["queued"] = True
        out = fin.on_finish(out_mem)
        # read the kernel's event pair only now: asking earlier blocks the host until the kernel
        # has finished and exposes the launch latency of everything behind it
        kernel_ms.append(part.kernel_ms(1 if state["queued"] else 0))
        if xchg is not None:
            phases.append(xchg.phase_ms())
        fin.reset()
        return out[0]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(blocks, steps, out_mem, timed, keep_last=False):
        """keep_last: return the last step's device result block itself (the caller releases it)."""
        res = None
        for i in range(steps):
            res = step_device(blocks, out_mem, prefetch_next=(i + 1 < steps))
            if timed:
                step_walls.append(time.perf_counter())
            if out_mem == abi.MEM_DEVICE and not (keep_last and i + 1 == steps):
                rows_out = res.num_rows
                L.dbx_block_release(C.byref(res))
                res = rows_out
        return res

    sampler = ClockSampler(dev)
    if rank == 0:
        sampler.start()  # before the warm-up: nvidia-smi's start-up must not fall into the timed region
    groups = run_steps([dblock], args.warmup, abi.MEM_DEVICE, False)
    kernel_ms.clear()
    phases.clear()
    barrier()
    gc.disable()
    sampler.mark()
    launches0 = L.dbx_kernel_launch_count()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record(part_stream)
    t0 = time.perf_counter()
    groups = run_steps([dblock], args.steps, abi.MEM_DEVICE, True, keep_last=bool(args.dump_outputs))
    ev1.record(fin_stream)
    barrier()
    wall = time.perf_counter() - t0
    sampler.mark()
    gc.enable()
    agg_out = None
    if args.dump_outputs:  # the last timed step's result, as the caller of the operator receives it
        last = groups
        groups = last.num_rows
        agg_out = download_block(L, dev, last)
        L.dbx_block_release(C.byref(last))
        if world > 1:  # every rank owns a disjoint set of groups
            parts = [None] * world
            dist.all_gather_object(parts, agg_out)
            agg_out = [np.concatenate(c) for c in zip(*parts)]
    dev_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    launches = L.dbx_kernel_launch_count() - launches0
    step_ms = max(dev_ms, 0.0) / args.steps
    t = torch.tensor([step_ms, wall * 1e3 / args.steps], dtype=torch.float64, device=f"cuda:{dev}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    step_ms, wall_ms = t.tolist()
    k_ms = sum(kernel_ms) / max(1, len(kernel_ms))
    per_step = np.diff(np.array([t0] + step_walls)) * 1e3
    phase_avg = None
    if phases:
        phase_avg = {k: float(np.mean([p_[k] for p_ in phases])) for k in phases[0]}
        phase_avg["partial_kernel"] = k_ms
        pt = torch.tensor([phase_avg[k] for k in sorted(phase_avg)], dtype=torch.float64, device=f"cuda:{dev}")
        dist.all_reduce(pt, op=dist.ReduceOp.MAX)
        phase_avg = {k: v for k, v in zip(sorted(phase_avg), pt.tolist())}
        phase_avg["note"] = "device ms per query, mean over the timed steps, max over ranks (CUDA events; wait_spin = the wait kernel's own globaltimer measure)"

    # ---- verification (outside the timed region): the whole result, at full size
    verify = None
    if not args.no_verify:
        res_host = step_device([dblock], abi.MEM_HOST, prefetch_next=False)
        try:
            verify = verify_result(res_host, dev, rank, world, [b_.ptr for b_ in bufs], n, args.keys, torch, dist)
        except Exception as e:  # the checker itself failed: say so, never claim a verified result
            verify = {"ok": False, "groups": None, "error": f"{type(e).__name__}: {e}"}
        if rank == 0 and not verify["ok"]:
            print(f"[bench] VERIFICATION FAILED: {verify}", file=sys.stderr)

    # ---- e2e: host (pinned) columns pushed through the operator API, result pulled to the host
    e2e = None
    if not args.no_e2e:
        e_rows = min(n, args.e2e_rows // world if args.e2e_rows else n)
        try:
            import psutil
            avail = psutil.virtual_memory().available
            while e_rows * 24 * world > 0.5 * avail and e_rows > 1_000_000:
                e_rows //= 2
        except Exception:
            pass
        hp = []
        for i in range(3):
            p = C.c_void_p()
            lib.check(L.dbx_host_alloc(e_rows * 8, C.byref(p)))
            lib.check(L.dbx_memcpy_d2h(dev, p, bufs[i].ptr, e_rows * 8))
            hp.append(p)
        harr = [np.ctypeslib.as_array(C.cast(hp[i], C.POINTER(C.c_int64 if i < 2 else C.c_double)), shape=(e_rows,)) for i in range(3)]
        hblock = DataBlock([Column.from_data(harr[0]), Column.from_data(harr[1]), Column.from_data(harr[2])], e_rows)

        def e2e_leg(block_rows, steps):
            hblocks = [b.freeze() for b in hblock.split_by_rows(block_rows)]  # descriptors built once, as a compiled caller would
            res = None
            for _ in range(max(1, min(2, args.warmup - 1))):
                res = run_steps(hblocks, 1, abi.MEM_HOST, False)
            barrier()
            t0 = time.perf_counter()
            res = run_steps(hblocks, steps, abi.MEM_HOST, False)
            barrier()
            ms = (time.perf_counter() - t0) * 1e3 / steps
            te = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{dev}")
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return te.item(), res

        e_steps = max(1, min(args.steps, 3))
        e_wall_ms, res = e2e_leg(args.block_rows, e_steps)
        d2h = sum(c.data.nbytes for c in res.columns)
        e2e = {"value": (e_rows * world) / (e_wall_ms * 1e-3), "unit": "rows/s", "h2d_bytes_per_step": int(e_rows * 24),
               "d2h_bytes_per_step": int(d2h), "rows": int(e_rows * world), "block_rows": args.block_rows,
               "ms_per_step": e_wall_ms, "timing": "host wall clock around push..pull incl. stream sync, max over ranks"}
        if args.small_block_rows:
            s_ms, _ = e2e_leg(args.small_block_rows, 1)
            e2e["small_blocks"] = {"block_rows": args.small_block_rows, "value": (e_rows * world) / (s_ms * 1e-3), "unit": "rows/s",
                                   "ms_per_step": s_ms, "note": "the reference's max_block_size (settings_default.rs:142)"}
        for p in hp:
            L.dbx_host_free(p)

    knn = None
    if xchg is not None:
        barrier()
        xchg.close()
    part.close()
    fin.close()
    for b_ in bufs:
        b_.free()
    knn_out = None
    if not args.no_knn:
        knn, knn_out = run_knn(args, L, dev, rank, world, barrier)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- CPU baseline on a bounded sample (rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu:
        from oracle import oracle as orc
        threads = len(os.sched_getaffinity(0))
        cn = args.cpu_rows
        k = orc.synth_fill(0, SEEDS[0], N_KEYS, 0, cn)
        v = orc.synth_fill(1, SEEDS[1], 0, 0, cn)
        x = orc.synth_fill(2, SEEDS[2], 20, 0, cn)
        cblk = DataBlock([Column.from_data(k), Column.from_data(v), Column.from_data(x)])
        cp = params.to_c(filt)
        orc.filter_group_agg(cblk, cp, threads=threads)
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            orc.filter_group_agg(cblk, cp, threads=threads)
        cdt = (time.perf_counter() - t0) / reps
        cpu = {"value": cn / cdt, "unit": "rows/s", "cores": threads, "kind": "port",
               "sample": f"first {cn} rows of the same columns, reference-algorithm C/OpenMP restatement (oracle), {reps} reps",
               "note": "a restatement, not Databend's executor: reported baseline only (its per-bucket final merge is not tuned)"}

    peak, peak_src = peaks()
    achieved = BYTES_PER_ROW * n / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
    traffic, traffic_note = ncu_traffic()
    line = {
        "metric": METRIC, "value": total_rows / (step_ms * 1e-3), "unit": "rows/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": {"workload": "configs[1]: filter(v%3=0) + hash-agg sum(v),count(v),avg(x) GROUP BY k; 1e6 int64 keys",
                   "rows": total_rows, "rows_per_gpu": n, "groups_out": verify["groups"] if verify else None,
                   "groups_out_rank0": int(groups),
                   "columns": "k:int64 v:int64 x:float64", "l2": "inputs (24 B/row x rows) far larger than the 126 MB L2",
                   "timing": "CUDA events on the operators' streams around the K steps, max over ranks; wall_ms_per_step alongside",
                   "pipelining": ("partial operator scans query i+1 while the final operator merges/materialises query i (every query's work inside the timed region)" if pipeline else "none"),
                   "per_step_wall_ms": {"min": float(per_step.min()), "median": float(np.median(per_step)), "max": float(per_step.max())},
                   "parallelism": f"row-range x{world}" + ("" if world == 1 else (" + peer-memory (NVLink) scatter of partial groups" if use_peer else " + NCCL all-to-all of partial groups"))},
        "wall_ms_per_step": wall_ms, "gpu_launches": int(launches), "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_note": traffic_note,
                     "achieved_per_launch_bytes": BYTES_PER_ROW * min(n, 1 << 28), "kernel": (KERNEL_NAME_JIT if variant == "specialised" else KERNEL_NAME), "kernel_variant": variant, "kernel_ms": k_ms,
                     "algorithmic_bytes_per_row": BYTES_PER_ROW, "peak_source": peak_src},
        "phases": phase_avg, "verify": verify,
        "cpu_baseline": cpu, "e2e": e2e, "knn": knn,
    }
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        # group order out of the hash table is unspecified: rows are written in ascending key order
        o = np.argsort(agg_out[3], kind="stable")
        tables = {"agg": {name: agg_out[i][o] for i, name in enumerate(["agg_sum_v", "agg_count_v", "agg_avg_x", "agg_k"])}}
        if knn_out is not None:
            tables["knn"] = {"knn_row_id": knn_out[0].astype(np.float64), "knn_distance": knn_out[1].astype(np.float32)}
        write_outputs(args.dump_outputs, tables)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="dbx", choices=["dbx", "reference"])
    ap.add_argument("--rows", type=int, default=1_000_000_000)
    ap.add_argument("--e2e-rows", type=int, default=0, help="0 = same as --rows")
    ap.add_argument("--block-rows", type=int, default=1 << 22, help="rows per pushed host block in the e2e leg (max_block_size)")
    ap.add_argument("--cpu-rows", type=int, default=50_000_000)
    ap.add_argument("--keys", type=int, default=N_KEYS, help="distinct group keys (the named config uses 1e6)")
    ap.add_argument("--small-block-rows", type=int, default=65536, help="also time the e2e leg with blocks of this many rows (65536 = the reference's max_block_size)")
    ap.add_argument("--no-verify", action="store_true", help="skip the full-size result verification (outside the timed region)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-knn", action="store_true", help="skip the kNN leg (second half of BASELINE.json's metric)")
    ap.add_argument("--knn-rows", type=int, default=10_000_000)
    ap.add_argument("--knn-dim", type=int, default=768)
    ap.add_argument("--knn-queries", type=int, default=1024)
    ap.add_argument("--knn-k", type=int, default=10)
    ap.add_argument("--knn-cpu-rows", type=int, default=1_000_000, help="corpus rows of the CPU sample in the reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32/float64, "
                         "at most 64 MB in all: a fixed, seeded sample of the rows when larger): the query result in "
                         "ascending key order (agg_sum_v, agg_count_v, agg_avg_x, agg_k; integers converted to float64) "
                         "and the kNN leg's top-k per query (knn_row_id, knn_distance)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "dbx":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl dbx")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_dbx(args)


if __name__ == "__main__":
    main()
