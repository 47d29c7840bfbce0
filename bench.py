#!/usr/bin/env python
"""bench.py — events/sec of the segmented event fold (BASELINE.json metric) on N B200s of one node.

A "step" is one full pass of the hot path over one batch of synthetic input: rebuilding every aggregate's state from its
CSR event log (configs[1]: 1,048,576 aggregates x 32 fixed 64-byte events = 2 GiB of events per GPU; the log is far larger
than the 126 MB L2, so no flush is needed between timed iterations).

  value   whole-job events/s with the log resident in HBM, K pipelined folds, CUDA events on the engine's stream, max over
          ranks (weak scaling of the fold itself: every rank folds its own shard of aggregates)
  e2e     the same metric through the C ABI with HOST buffers in the format the reference's topic holds: every step hands the
          step's events as lz4 Kafka RecordBatch bytes in pinned host memory to sgr_dingest_submit / sgr_dingest_fold (decode on the
          device) and reads the state table back (sgr_export_states). e2e_packed_records: round 1's variant, 64-byte records
          over PCIe (sgr_load_events + sgr_fold + sgr_export_states)
  roofline   algorithmic bytes / device time of the fold kernel against the measured HBM peak
  cpu_baseline   the CPU oracle (port of the reference's fold) on this box's host cores, NUMA-placed log, pinned threads
  routed  configs[2], the configuration north_star names for N GPUs: the FULL problem (10 M aggregates x 100 events = 64 GB,
          arrival order, pre-distributed by source partition) strong-scaled over the N ranks: hash-partition by aggregate, ONE
          exchange over NVLink, fold — pipelined (surge_b200/csrc/route_push.cu): `exchange_pipelined` moves whole 64-byte
          records' sectors, `exchange_projected_16B` only the words the fold program reads, `nccl_all_to_all` is the
          count + pack + grouped ncclSend/ncclRecv path for comparison. Every mode prints a 64-bit hash of the
          whole state table (sum over ranks; identical at N = 1, 2, 4, 8 by construction of the log), the same hash from an
          independent vectorised torch restatement of the Counter fold over the full table, and a 4096-aggregate sample
          checked against the CPU oracle.
  configs every other BASELINE.json config (N = 1 only): configs[0] BankAccount, configs[3] Zipf / variable records at full
          size, configs[4] streaming micro-batches — each with its own parity check.

`--impl reference` times the reference's CPU implementation of the path instead (the oracle port: the reference is Scala/JVM
and cannot be built in this image), rank 0 only.

`--dump-outputs DIR` writes, after the timed steps, the state table the last timed step left (rank 0's shard) as DIR/states.npy,
so that two builds run with the same arguments (same seeded inputs) can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_AGG = 1 << 20
EVENTS_PER_AGG = 32
STATE_BYTES = 16
METRIC = "events/sec replayed (segmented per-aggregate event fold)"
WORKLOAD = "configs[1]: 1,048,576 aggregates x 32 fixed-width 64-B events, single B200 segmented fold (per GPU)"
ROUTED_N_GLOBAL = 10_000_000     # configs[2]: 10 M aggregates x 100 events, hash-partitioned, one exchange
ROUTED_EPA = 100
ROUTED_SEED = 3
NVLINK_PEAK_GBS = 770.0          # measured peer copy per direction per GPU on this pool (B200_PROFILING.md)
M64 = (1 << 64) - 1
DUMP_MAX_BYTES = 64_000_000      # --dump-outputs: all arrays together


def algorithmic_bytes(n_agg: int, epa: int) -> int:
    """B_alg = stored event bytes + 8*(nAgg+1) CSR offsets + S*nAgg states written (SURVEY.md 8d)."""
    return n_agg * epa * 64 + 8 * (n_agg + 1) + STATE_BYTES * n_agg


def state_columns(table):
    """A Counter state table (u8 [n, 16], include/sgr.h) as float64 [n, 4]: count and version (the program's i32 words), then
    the engine's u32 flags and err_idx. float64 holds every 32-bit value exactly."""
    import numpy as np

    table = np.ascontiguousarray(table)
    cols = table.view(np.int32).astype(np.float64)
    cols[:, 2:] = table.view(np.uint32)[:, 2:]
    return cols


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes every array as out_dir/<name>.npy."""
    import numpy as np

    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peak_gbs() -> tuple[float, str]:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Polls NVML for SM clock and throttle reasons while the timed regions run."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:  # noqa: BLE001
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
        }
        while not self._stop.is_set():
            try:
                mhz = int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                self.samples.append((mhz, util))
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self) -> dict:
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        mhz = [m for m, _ in self.samples]
        return {"sm_mhz": int(statistics.median(mhz)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(mhz)}


# ---------------------------------------------------------------------------------------------------- CPU legs
def host_config2_log(n_agg: int, epa: int, seed: int):
    """The configs[1] Counter log built on the host (numpy), for the CPU legs."""
    import numpy as np

    from surge_b200 import formats as F

    rng = np.random.Generator(np.random.Philox(seed))
    n = n_agg * epa
    rec = np.zeros((n, 16), dtype=np.int32)
    u = rng.random(n, dtype=np.float32)
    rec[:, 0] = np.where(u < 0.45, F.COUNT_INCREMENTED, np.where(u < 0.9, F.COUNT_DECREMENTED, F.NO_OP_EVENT))
    idx = np.arange(n, dtype=np.int64)
    rec[:, 1] = (idx % epa + 1).astype(np.int32)
    rec[:, 2] = (idx // epa).astype(np.int32)
    rec[:, 4] = rng.integers(0, 1 << 31, size=n, dtype=np.int64).astype(np.int32)
    off = (np.arange(n_agg + 1, dtype=np.uint64) * np.uint64(epa * 64))
    return rec, off


def cpu_fold_setup(rec, off, threads: int):
    """NUMA-sane CPU arm: the log is copied once into fresh memory by the pinned workers that will fold it (first touch puts
    every worker's byte range on its own node); every timed pass then runs with worker t on CPU t."""
    from oracle import oracle as O

    O.fold_packed(O.MODEL_COUNTER, O.REC_FIXED64, rec[: 64 * 16], off[:33], threads=1)  # load the library
    return O.place_log(rec, off, threads)


def time_cpu_oracle(rec, off, threads: int, min_seconds: float, max_reps: int):
    from oracle import oracle as O

    placed = cpu_fold_setup(rec, off, threads)
    O.fold_packed(O.MODEL_COUNTER, O.REC_FIXED64, placed, off, threads=threads, pinned=True)   # warm-up pass
    reps, t_total, nev = 0, 0.0, 0
    while reps < max_reps and (reps == 0 or t_total < min_seconds):
        t0 = time.perf_counter()
        _, n, _ = O.fold_packed(O.MODEL_COUNTER, O.REC_FIXED64, placed, off, threads=threads, pinned=True)
        t_total += time.perf_counter() - t0
        nev += n
        reps += 1
    return nev / t_total, reps, t_total


def run_reference(args) -> None:
    """The reference's CPU implementation of the path (oracle port, all host threads), rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # one step = one pass over the full configs[1] log (33.5 M events, 2 GiB, far larger than any CPU cache, like the GPU arm's
    # step); a cache-resident sample would overstate what the CPU path does on this workload
    rec, off = host_config2_log(N_AGG, EVENTS_PER_AGG, seed=2)
    from oracle import oracle as O

    placed = cpu_fold_setup(rec, off, cores)
    del rec
    for _ in range(max(args.warmup, 1)):
        O.fold_packed(O.MODEL_COUNTER, O.REC_FIXED64, placed, off, threads=cores, pinned=True)
    t0 = time.perf_counter()
    nev = 0
    for _ in range(args.steps):
        states, n, _ = O.fold_packed(O.MODEL_COUNTER, O.REC_FIXED64, placed, off, threads=cores, pinned=True)
        nev += n
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"states": state_columns(states)})
    value = nev / dt
    sample = (f"{N_AGG} aggregates x {EVENTS_PER_AGG} events per step (the full configs[1] log, host memory first-touched by the "
              f"pinned worker that folds it), {args.steps} steps")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "events/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "i32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample, "impl_note": "CPU port of the reference's fold (oracle/sgr_oracle.c), one pinned thread per "
                   "hardware thread; the Scala/JVM reference cannot be built in this image"},
        "cpu_baseline": {"value": value, "unit": "events/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------------- parity helpers (torch)
def _s64(c: int) -> int:
    return c - (1 << 64) if c >= (1 << 63) else c


def _lsr(x, k: int):
    return (x >> k) & ((1 << (64 - k)) - 1)


def _splitmix64_t(x):
    x = x + _s64(0x9E3779B97F4A7C15)
    x = (x ^ _lsr(x, 30)) * _s64(0xBF58476D1CE4E5B9)
    x = (x ^ _lsr(x, 27)) * _s64(0x94D049BB133111EB)
    return x ^ _lsr(x, 31)


def torch_states_hash(words64, gids) -> int:
    """torch twin of sgr_states_hash (csrc/bulk_fold.cu): words64 = the state table viewed as int64 [n, state_bytes / 8]."""
    h = _splitmix64_t(gids)
    for k in range(words64.shape[1]):
        h = _splitmix64_t(h ^ words64[:, k])
    return int(h.sum().item()) & M64


def routed_expected_hash(gids, epa: int, seed: int) -> int:
    """Independent vectorised restatement of the Counter fold (scaladsl TestBoundedContext.scala:77-89) over the deterministic
    configs[2] log, for the aggregates `gids` (int64 CUDA tensor), from None: count = wrapped sum of +-by, version = seq of the
    last counting event, every aggregate exists and changed. Returns the state hash of that table."""
    import torch

    from surge_b200 import synth as S

    count = torch.zeros_like(gids, dtype=torch.int32)
    version = torch.zeros_like(gids, dtype=torch.int32)
    for k in range(epa):
        typ, by = S.routed_round(gids, k, seed)
        count = count + torch.where(typ == 0, by, torch.where(typ == 1, -by, torch.zeros_like(by)))
        version = torch.where(typ < 2, torch.full_like(version, k + 1), version)
    w0 = (count.to(torch.int64) & 0xFFFFFFFF) | (version.to(torch.int64) << 32)
    w1 = torch.full_like(w0, 3)   # EXISTS | CHANGED, err_idx 0
    return torch_states_hash(torch.stack([w0, w1], 1), gids)


# ---------------------------------------------------------------------------------------------------- configs[2]
def config2_routed(rank, world, local_rank, dev, barrier, note, scale: float, iters: int):
    import numpy as np
    import torch
    import torch.distributed as dist

    from oracle import oracle as O
    from surge_b200 import ReplayEngine
    from surge_b200 import dist as D
    from surge_b200 import programs as P
    from surge_b200 import synth as S

    n_global = max(int(ROUTED_N_GLOBAL * scale) // 64 * 64, 64)
    epa = ROUTED_EPA
    rec = S.routed_log_device(rank, world, n_global, epa, ROUTED_SEED, dev)
    n = rec.shape[0]
    flat = rec.view(torch.uint8).view(-1)
    part = S.routed_partitions(n_global, 64)
    total_events = n_global * epa
    res = {"workload": f"configs[2]{'' if scale == 1.0 else f' x {scale}'}: {n_global} aggregates x {epa} events x 64 B = {total_events * 64 / 1e9:.1f} GB, "
                       f"arrival order, pre-distributed by source partition over {world} rank(s); owner = partition(hash(id)) % nranks; strong scaling",
           "events_total": total_events, "n_ranks": world}
    # the oracle's word on a sample of aggregates (the same sample at every N)
    sample = np.random.default_rng(2024).choice(n_global, size=min(4096, n_global), replace=False).astype(np.int64)
    sample.sort()
    srec, soff = S.routed_events_host(sample, epa, ROUTED_SEED)
    want_sample, _, _ = O.fold_packed(O.MODEL_COUNTER, O.REC_FIXED64, srec, soff, threads=min(os.cpu_count() or 1, 16))

    eng = ReplayEngine(local_rank)
    eng.register_program(P.counter_program())
    if world > 1:
        cap = int(n * 1.12) + 64 * 1024 * world
        D.exchange_ids(eng, rank, world, cap, fused=True)
        eng.dist_set_partitions(part)
        modes = [("exchange_pipelined", 2), ("exchange_projected_16B", 3), ("nccl_all_to_all", 0)]
    else:
        modes = [("single_gpu_sort_free", None)]
    expected_hash = None
    for name, fused in modes:
        times = []
        its = iters if fused != 0 else min(iters, 2)
        for it in range(its + 1):   # first iteration is the warm-up (allocations, NCCL connections)
            barrier()
            t0 = time.perf_counter()
            if fused is None:
                eng.fold_unsorted(flat, n_global)
            else:
                eng.dist_route_and_fold(flat, fused)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            ds = eng.dist_stats() if fused is not None else None
            v = [dt, eng.stats().ms_fold, ds.ms_pipeline if ds else 0.0, ds.ms_scatter if ds else 0.0, ds.ms_exchange if ds else 0.0,
                 ds.ms_count if ds else 0.0, ds.ms_group if ds else 0.0]
            t = torch.tensor(v, dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            if it > 0:
                times.append([float(x) for x in t])
        best = min(times, key=lambda r: r[0])
        # ---- parity: hash of the whole table (sum over ranks), the torch restatement's hash, the oracle on the sample
        h = torch.tensor([np.int64(np.uint64(eng.states_hash()))], dtype=torch.int64, device=dev)
        gl = torch.from_numpy(eng.dist_local_aggregates().astype(np.int64)).to(dev) if fused is not None else torch.arange(n_global, device=dev, dtype=torch.int64)
        if expected_hash is None:
            eh = torch.tensor([np.int64(np.uint64(routed_expected_hash(gl, epa, ROUTED_SEED)))], dtype=torch.int64, device=dev)
            if world > 1:
                dist.all_reduce(eh)
            expected_hash = int(eh.item()) & M64
        states = eng.states_tensor()
        pos = torch.searchsorted(gl, torch.from_numpy(sample).to(dev))
        pos_c = pos.clamp(max=gl.numel() - 1)
        mine = gl[pos_c] == torch.from_numpy(sample).to(dev)
        got = states[pos_c[mine]].cpu().numpy()
        bad = torch.tensor([int((got != want_sample[mine.cpu().numpy()]).any(axis=1).sum()), int(mine.sum())], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(h)
            dist.all_reduce(bad)
        state_hash = int(h.item()) & M64
        ev = int(eng.stats().n_events)
        tot = torch.tensor([ev], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(tot)
        wire = (ds.exchange_record_bytes if ds and ds.exchange_record_bytes else 64)
        remote = (ds.n_sent_remote if ds else 0)
        xfer_ms = best[2] if fused in (2, 3) else best[4]
        res[name] = {
            "events_per_s": total_events / best[0], "ms_wall": best[0] * 1e3, "ms_wall_all": [round(r[0] * 1e3, 3) for r in times],
            "ms_device_pipeline": best[2] if fused in (2, 3) else None, "ms_partition": best[3] if fused in (2, 3) else None,
            "ms_route_count": best[5] if fused == 0 else None, "ms_route_scatter": best[3] if fused == 0 else None, "ms_exchange": best[4] if fused == 0 else None,
            "ms_fold": best[1], "ms_group": best[6],
            "exchange_bytes_per_record": wire,
            "nvlink_out_gb_per_s_per_gpu": (remote * wire / (xfer_ms * 1e-3) / 1e9) if (world > 1 and xfer_ms) else None,
            "parity": {"state_hash": f"{state_hash:016x}", "torch_restatement_hash": f"{expected_hash:016x}",
                       "full_table_equals_restatement": state_hash == expected_hash,
                       "oracle_sample_aggregates": int(bad[1]), "oracle_sample_mismatches": int(bad[0]),
                       "events_folded": int(tot.item()), "events_expected": total_events},
        }
        note(f"routed {name}: {res[name]['ms_wall']:.2f} ms, hash ok {state_hash == expected_hash}")
    if world > 1:
        res["nvlink_peak_gb_per_s"] = NVLINK_PEAK_GBS
        res["exchange_lower_bound_ms"] = (total_events / world) * (world - 1) / world * 64 / (NVLINK_PEAK_GBS * 1e9) * 1e3
    eng.close()
    del eng, rec, flat
    torch.cuda.empty_cache()
    return res


# ---------------------------------------------------------------------------------------------------- configs[0], [3], [4] (N = 1)
def config0_bank(dev, peak):
    """configs[0]: BankAccount, 1k aggregates x 10 events (the reference's CPU-runnable case) bit-exact vs the oracle, and the
    same model on the configs[1] shape for the wide-state kernel's rate."""
    import uuid

    import numpy as np
    import torch

    from oracle import oracle as O
    from surge_b200 import ReplayEngine
    from surge_b200 import formats as F
    from surge_b200 import programs as P

    recs = []
    for a in range(1000):
        acct = str(uuid.UUID(int=(a * 0x9E3779B97F4A7C15 + 1) & ((1 << 128) - 1)))
        recs.append(F.bank_created_record(a, 1, acct, f"owner-{a}", "c0de", 1000.0))
        for k in range(9):
            recs.append(F.bank_updated_record(a, k + 2, acct, 1000.0 + (k + 1) * 0.25))
    log = np.frombuffer(b"".join(recs), dtype=np.uint8)
    off = np.arange(1001, dtype=np.uint64) * np.uint64(640)
    want, nev, _ = O.fold_packed(O.MODEL_BANK_ACCOUNT, O.REC_FIXED64, log, off)
    with ReplayEngine(0) as e:
        e.register_program(P.bank_account_program())
        e.load_events(log, off)
        e.fold()
        small_ok = bool(np.array_equal(e.export_states(), want))
    n_agg, epa = 1 << 20, 32
    n = n_agg * epa
    gen = torch.Generator(device=dev)
    gen.manual_seed(9)
    r = torch.randint(-(1 << 31), 1 << 31, (n, 16), generator=gen, device=dev, dtype=torch.int64).to(torch.int32)
    idx = torch.arange(n, device=dev, dtype=torch.int64)
    r[:, 0] = (idx % epa != 0).to(torch.int32)   # first event of every account creates it, the rest update the balance
    r[:, 1] = (idx % epa + 1).to(torch.int32)
    r[:, 2] = (idx // epa).to(torch.int32)
    r[:, 3] = 0
    offd = torch.arange(n_agg + 1, device=dev, dtype=torch.int64) * (epa * 64)
    b_alg = n * 64 + 8 * (n_agg + 1) + 64 * n_agg
    out = {"workload": "configs[0]: BankAccount sample aggregate (64-byte state, IF_EXISTS rule, JVM Double balance)",
           "small_1k_x_10": {"events": int(nev), "bit_exact_vs_oracle": small_ok}}
    tabs = []
    for label, kernel in (("auto", 0), ("lane_sequential_tma", 1)):
        with ReplayEngine(0) as e:
            e.register_program(P.bank_account_program())
            e.set_option("kernel", kernel)
            e.load_events(r.view(torch.uint8), offd)
            ms = []
            for _ in range(4):
                e.set_initial_states(None)
                e.fold()
                ms.append(e.stats().ms_fold)
            tabs.append(e.states_tensor().clone())
            # a 2048-aggregate sample against the oracle
            if kernel == 0:
                sel = torch.arange(0, n_agg, n_agg // 2048, device=dev)
                seg = r.view(n_agg, epa * 16)[sel].cpu().numpy().view(np.uint8).reshape(-1)
                soff = np.arange(len(sel) + 1, dtype=np.uint64) * np.uint64(epa * 64)
                w, _, _ = O.fold_packed(O.MODEL_BANK_ACCOUNT, O.REC_FIXED64, seg, soff)
                sample_ok = bool(np.array_equal(e.states_tensor()[sel].cpu().numpy(), w))
        best = min(ms[1:])
        out[f"configs1_shape_{label}"] = {"ms_fold": best, "events_per_s": n / best * 1e3, "achieved_gb_per_s": b_alg / best / 1e6, "frac_of_hbm_peak": b_alg / best / 1e6 / peak}
    out["configs1_shape_kernels_agree"] = bool(torch.equal(tabs[0], tabs[1]))
    out["configs1_shape_oracle_sample_ok"] = sample_ok
    return out


def config3_zipf(dev, peak, scale: float):
    """configs[3]: Zipf(1.1) keys, 10 M aggregates, 3.2e8 events, payloads 32-512 B (variable records, ~95 GB) on one B200."""
    import numpy as np
    import torch

    from oracle import oracle as O
    from surge_b200 import ReplayEngine
    from surge_b200 import native as N
    from surge_b200 import programs as P

    n_keys, n_events = int(10_000_000 * scale), int(320_000_000 * scale)
    gen = torch.Generator(device=dev)
    gen.manual_seed(4)
    w = 1.0 / torch.pow(torch.arange(1, n_keys + 1, device=dev, dtype=torch.float64), 1.1)
    cdf = torch.cumsum(w, 0)
    cdf /= cdf[-1].clone()
    counts = torch.zeros(n_keys, dtype=torch.int64, device=dev)
    step = 40_000_000
    for lo in range(0, n_events, step):   # inverse-CDF sampling, in slices (temporaries stay small)
        k = torch.searchsorted(cdf, torch.rand(min(step, n_events - lo), generator=gen, device=dev, dtype=torch.float64)).clamp_(max=n_keys - 1)
        counts += torch.bincount(k, minlength=n_keys)
    del w, cdf, k
    plen = torch.randint(32, 513, (n_events,), generator=gen, device=dev, dtype=torch.int64)
    rlen = 16 + ((plen + 15) // 16) * 16
    rec_off = torch.zeros(n_events + 1, dtype=torch.int64, device=dev)
    rec_off[1:] = torch.cumsum(rlen, 0)
    del rlen
    total = int(rec_off[-1])
    starts = torch.zeros(n_keys + 1, dtype=torch.int64, device=dev)
    starts[1:] = torch.cumsum(counts, 0)
    seg = rec_off[starts]
    buf = torch.empty(total, dtype=torch.uint8, device=dev)
    chunk = 1 << 32
    for lo in range(0, total, chunk):     # filler the fold must still read
        hi = min(total, lo + chunk)
        buf[lo:hi] = torch.randint(0, 256, (hi - lo,), generator=gen, device=dev, dtype=torch.uint8)
    w32 = buf.view(torch.int32)
    agg = torch.repeat_interleave(torch.arange(n_keys, device=dev, dtype=torch.int64), counts)
    pos = rec_off[:-1] // 4
    w32[pos + 3] = agg.to(torch.int32)
    w32[pos + 1] = (torch.arange(n_events, device=dev, dtype=torch.int64) - starts[agg] + 1).to(torch.int32)
    del agg
    w32[pos + 2] = plen.to(torch.int32)
    del plen
    u = torch.rand(n_events, generator=gen, device=dev)
    w32[pos] = torch.where(u < 0.45, 0, torch.where(u < 0.9, 1, 2)).to(torch.int32)
    # the Counter's `by` (first 4 payload bytes) stays random filler: any i32 is a legal increment
    del u, pos
    torch.cuda.synchronize()
    hot = int(counts.max())
    b_alg = total + 8 * (n_keys + 1) + 16 * n_keys + 8 * (n_events + 1)
    out = {"workload": f"configs[3]{'' if scale == 1.0 else f' x {scale}'}: Zipf(1.1) keys, {n_keys} aggregates, {n_events} events, payloads 32-512 B, {total / 1e9:.1f} GB log, one B200",
           "hottest_key_share": hot / n_events, "algorithmic_bytes": b_alg}
    with ReplayEngine(0) as e:
        e.register_program(P.counter_program(N.REC_VAR16))
        e.load_events_indexed(buf, seg, rec_off)
        ms = []
        for _ in range(3):
            e.set_initial_states(None)
            e.fold()
            ms.append(e.stats().ms_fold)
        st = e.stats()
        best = min(ms[1:])
        out.update({"ms_fold": best, "events_per_s": n_events / best * 1e3, "achieved_gb_per_s": b_alg / best / 1e6, "frac_of_hbm_peak": b_alg / best / 1e6 / peak,
                    "events_folded": int(st.n_events), "launches": int(st.fold_launches), "kernel": "fold_vruns_kernel"})
        # oracle on a sample of aggregates: 4096 random ones with segments of at most 8 MiB, plus the 8 largest below that bound
        seg_h = seg.cpu().numpy()
        seg_len = np.diff(seg_h)
        ok_idx = np.nonzero(seg_len <= (8 << 20))[0]
        rng = np.random.default_rng(31)
        pick = np.unique(np.concatenate([rng.choice(ok_idx, size=min(4096, len(ok_idx)), replace=False), ok_idx[np.argsort(seg_len[ok_idx])[-8:]]]))
        parts = [buf[int(seg_h[i]):int(seg_h[i + 1])].cpu().numpy() for i in pick]
        soff = np.zeros(len(pick) + 1, dtype=np.uint64)
        np.cumsum([len(p) for p in parts], out=soff[1:])
        want, _, _ = O.fold_packed(O.MODEL_COUNTER, O.REC_VAR16, np.concatenate(parts) if parts else np.zeros(0, np.uint8), soff, threads=min(os.cpu_count() or 1, 16))
        got = e.states_tensor()[torch.from_numpy(pick).to(dev)].cpu().numpy()
        out["parity"] = {"oracle_sample_aggregates": int(len(pick)), "oracle_sample_mismatches": int((got != want).any(axis=1).sum()),
                         "events_folded_equals_events": int(st.n_events) == n_events, "state_hash": f"{e.states_hash():016x}"}
    del buf, w32, rec_off, seg, starts, counts
    torch.cuda.empty_cache()
    return out


def config4_microbatch(dev, n_batches: int):
    """configs[4]: 100k-event batches appended to 1,048,576 live aggregates (incremental fold), sustained rate and latency."""
    import numpy as np
    import torch

    from oracle import oracle as O
    from surge_b200 import ReplayEngine
    from surge_b200 import programs as P
    from surge_b200 import synth as S

    n_agg, batch = 1 << 20, 100_000
    rec, off = S.counter_csr_device(n_agg, 4, seed=5, device=dev)
    out = {"workload": f"configs[4]: {n_batches} batches of {batch} events onto {n_agg} live aggregates, incremental fold"}
    with ReplayEngine(0) as e:
        e.register_program(P.counter_program())
        e.load_events(rec.view(torch.uint8), off)
        e.fold()
        gen = torch.Generator(device=dev)
        gen.manual_seed(55)
        nb_pool = min(n_batches, 200)   # 200 distinct batches (1.28 GB), cycled
        pool = torch.zeros((nb_pool, batch, 16), dtype=torch.int32, device=dev)
        u = torch.rand((nb_pool, batch), generator=gen, device=dev)
        pool[:, :, 0] = torch.where(u < 0.45, 0, torch.where(u < 0.9, 1, 2)).to(torch.int32)
        pool[:, :, 1] = torch.arange(batch, device=dev, dtype=torch.int32)[None, :]
        pool[:, :, 2] = torch.randint(0, n_agg, (nb_pool, batch), generator=gen, device=dev, dtype=torch.int64).to(torch.int32)
        pool[:, :, 4] = torch.randint(0, 1 << 31, (nb_pool, batch), generator=gen, device=dev, dtype=torch.int64).to(torch.int32)
        torch.cuda.synchronize()
        want = e.export_states()
        for b in range(3):
            want = O.fold_incremental(O.MODEL_COUNTER, pool[b].cpu().numpy().view(np.uint8).reshape(-1), want)
            e.fold_incremental(pool[b].view(torch.uint8))
        out["bit_exact_vs_oracle_after_3_batches"] = bool(np.array_equal(e.export_states(), want))
        for b in range(10):
            e.fold_incremental(pool[b % nb_pool].view(torch.uint8))
        lat = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for b in range(n_batches):
            t1 = time.perf_counter()
            e.fold_incremental(pool[b % nb_pool].view(torch.uint8))
            lat.append(time.perf_counter() - t1)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        st = e.stats()
        lat = np.array(lat) * 1e6
        out.update({"events_per_s": n_batches * batch / dt, "batch_latency_us": {"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99))},
                    "device_ms_last_batch": float(st.ms_fold), "note": "launch-bound: one persistent launch per batch (6.4 MB of records), far below the HBM roofline by design"})
    return out


# ---------------------------------------------------------------------------------------------------- main
def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer region (default min(steps, 20))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--verbose", action="store_true", help="progress markers on stderr")
    ap.add_argument("--no-routed", action="store_true", help="skip configs[2] (the routed 10 M x 100 problem)")
    ap.add_argument("--no-configs", action="store_true", help="skip configs[0], [3], [4] (N = 1)")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink configs[2] and configs[3] (debugging on a busy box); 1.0 = the BASELINE sizes")
    ap.add_argument("--routed-iters", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the state table of the last one as "
                    "DIR/states.npy: float64 [aggregates, 4] = count, version, flags, err_idx (rank 0's shard)")
    args = ap.parse_args()
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)   # an unusable DIR fails here, not after the run
    if args.impl == "reference":
        run_reference(args)
        return

    def note(msg):
        if args.verbose:
            print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)

    note("importing torch")
    import numpy as np
    import torch
    import torch.distributed as dist

    from surge_b200 import ReplayEngine
    from surge_b200 import programs as P
    from surge_b200 import synth as S

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the replay engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peak, peak_src = measured_peak_gbs()
    # ---- this rank's shard: its own 2^20 aggregates (hash-partitioned aggregates are independent units)
    note("generating the log on the device")
    rec, off = S.counter_csr_device(N_AGG, EVENTS_PER_AGG, seed=2 + rank, device=dev)
    n_events = N_AGG * EVENTS_PER_AGG
    log_bytes = int(rec.numel() * 4)
    b_alg = algorithmic_bytes(N_AGG, EVENTS_PER_AGG)
    eng = ReplayEngine(local_rank)
    eng.register_program(P.counter_program())
    eng.load_events(rec.view(torch.uint8), off)
    stream = torch.cuda.ExternalStream(eng.stream_ptr(), device=dev)

    W = max(args.warmup, 3)
    K = args.steps
    note("warm-up folds")
    for _ in range(W):
        eng.set_initial_states(None)
        eng.fold()
    kernel_ms = eng.stats().ms_fold  # one fold alone, CUDA events around the kernel

    note("timed region 1")
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    # ---- timed region 1 (value): K pipelined folds, inputs resident in HBM
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(K):
        eng.set_initial_states(None)   # every step is a full rebuild from None
        eng.fold_async()
    ev1.record(stream)
    eng.wait()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = K * int(eng.stats().fold_launches)
    folded_events = int(eng.stats().n_events)
    assert folded_events == n_events, (folded_events, n_events)

    # ---- timed region 2 (e2e): host buffers through the C ABI, H2D + fold + D2H every step
    ke = args.e2e_steps or min(K, 20)
    note("pinned host buffers")
    host_log = torch.empty(rec.numel() * 4, dtype=torch.uint8, pin_memory=True)
    host_log.copy_(rec.view(torch.uint8).view(-1))
    host_off = off.cpu().numpy().astype(np.uint64)
    host_states = torch.empty(N_AGG * STATE_BYTES, dtype=torch.uint8, pin_memory=True)
    host_log_np, host_states_np = host_log.numpy(), host_states.numpy().reshape(N_AGG, STATE_BYTES)
    e2 = ReplayEngine(local_rank)
    e2.register_program(P.counter_program())
    for _ in range(2):
        e2.load_events(host_log_np, host_off)
        e2.set_initial_states(None)
        e2.fold()
        e2.export_states(host_states_np)
    barrier()
    note("timed region 2 (e2e)")
    t0 = time.perf_counter()
    for _ in range(ke):
        e2.load_events(host_log_np, host_off)      # H2D of the step's input from pinned host memory
        e2.set_initial_states(None)
        e2.fold()
        e2.export_states(host_states_np)           # D2H of the step's result
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    st2 = e2.stats()
    # the e2e result must be the same table the resident fold produced
    same = bool(torch.equal(torch.from_numpy(host_states_np.reshape(-1)).to(dev), eng.states_tensor().reshape(-1)))
    assert same, "e2e state table differs from the HBM-resident fold"
    # ---- configs[2]: the routed problem north_star names, strong-scaled, parity-hashed. Runs after the wire-format section;
    #      SGR_BENCH_ROUTED_FIRST=1 runs it before (an A/B kept from checking that the order does not change its time: it does not).
    routed = None
    routed_first = os.environ.get("SGR_BENCH_ROUTED_FIRST", "0") == "1"

    def run_routed():
        nonlocal routed
        if args.no_routed:
            return
        try:
            note("configs[2] routed")
            routed = config2_routed(rank, world, local_rank, dev, barrier, note, args.scale, args.routed_iters)
        except Exception as ex:  # noqa: BLE001 - the headline line must survive a failure of the extra measurement
            routed = {"error": f"{type(ex).__name__}: {ex}"}
        torch.cuda.empty_cache()

    if routed_first:
        run_routed()

    # ---- timed region 3 (e2e over the WIRE format): what the topic holds — lz4 RecordBatch bytes — goes to the device as it is;
    #      CRC, lz4, record parse, id interning and the fold run there (surge_b200/csrc/dingest_kernels.cu). Every step: submit
    #      the 32 partitions' bytes from pinned host memory, decode + fold into a fresh table, read the table back.
    wire_res = None
    wire = {}          # what the set-up leaves for the timed part
    try:
        if os.environ.get("SGR_BENCH_SKIP_WIRE"):
            raise RuntimeError("skipped (SGR_BENCH_SKIP_WIRE)")
        note("encoding the topic (32 partitions, lz4 batches of 512 records)")
        from concurrent.futures import ThreadPoolExecutor

        from oracle import oracle as O   # INPUT construction only: the producer-side encoder of the test infrastructure
        from surge_b200.dingest import DeviceIngest

        n_part = 32
        cols = rec.view(N_AGG, EVENTS_PER_AGG, 16)[:, :, [0, 1, 2, 4]].cpu().numpy()     # type, seq, agg, by
        def encode(p):
            sel = cols[p::n_part].reshape(-1, 4)
            return O.kafka_encode_counter(sel[:, 2].astype(np.uint32), sel[:, 0].astype(np.uint32), sel[:, 1].astype(np.uint32), sel[:, 3].astype(np.int32),
                                          recs_per_batch=512, lz4=True)
        with ThreadPoolExecutor(max_workers=max(1, min(n_part, (os.cpu_count() or 1) // world))) as ex:
            wires = list(ex.map(encode, range(n_part)))
        wire_bytes = int(sum(len(w) for w in wires))
        pinned = []
        for w in wires:
            t = torch.empty(len(w), dtype=torch.uint8, pin_memory=True)
            t.numpy()[:] = w
            pinned.append(t)
        del wires, cols
        e3 = ReplayEngine(local_rank)
        wire["e3"] = e3
        e3.register_program(P.counter_program())
        dg = DeviceIngest(e3, 1 << 21)
        wire["dg"] = dg

        phase = [0.0, 0.0, 0.0]

        def wire_step():
            ta = time.perf_counter()
            e3.set_initial_states(None)      # every step is a full rebuild: empty table, empty dictionary, offsets 0
            dg.reset()
            for p, t in enumerate(pinned):
                dg.submit(p, t)              # H2D of the step's input from pinned host memory
            tb = time.perf_counter()
            st = dg.fold()                   # decode + intern + fold on the device, ids back to the host key table
            tc = time.perf_counter()
            e3.export_states(host_states_np) # D2H of the step's result
            td = time.perf_counter()
            phase[0] += tb - ta; phase[1] += tc - tb; phase[2] += td - tc
            return st
        for _ in range(2):
            stw = wire_step()
        assert stw["n_records"] == n_events and stw["n_new_keys"] == N_AGG, stw
        torch.cuda.synchronize()
        wire["ready"] = True
    except Exception as ex:  # noqa: BLE001 - the headline line must survive
        wire_res = {"error": f"{type(ex).__name__}: {ex}"}
    # Every rank reports whether its set-up worked; the all-reduce is also the barrier in front of the timed region. (No barrier may
    # sit inside a try block: a rank that failed would never reach it and the others would wait for it forever.)
    all_ready = bool(wire.get("ready"))
    if world > 1:
        flag = torch.tensor([1 if all_ready else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        all_ready = bool(int(flag.item()))
    if all_ready:
        try:
            note("timed region 3 (e2e, wire format)")
            phase[:] = [0.0, 0.0, 0.0]
            t0 = time.perf_counter()
            for _ in range(ke):
                wire_step()
            torch.cuda.synchronize()
            wire_s = time.perf_counter() - t0
            # parity of the wire path: a sample of aggregates by id against the HBM-resident fold's table
            ref_tab = eng.states_tensor().cpu().numpy()
            bad = 0
            for g in range(0, N_AGG, N_AGG // 4096):
                got = e3.get(f"agg-{g}")
                bad += int(got != ref_tab[g, :8].tobytes())
            wire_res = {"seconds": wire_s, "wire_bytes": wire_bytes, "last_step_ms": dg.last_timing(), "host_ms_per_step": {"submit": phase[0] / ke * 1e3, "fold": phase[1] / ke * 1e3, "export": phase[2] / ke * 1e3}, "bytes_per_event": wire_bytes / n_events, "sample_mismatches": bad,
                        "decompressed_bytes": int(stw["n_decompressed_bytes"]), "batches": int(stw["n_batches"])}
            assert bad == 0, "wire-format e2e differs from the resident fold"
        except Exception as ex:  # noqa: BLE001 - the headline line must survive
            wire_res = {"error": f"{type(ex).__name__}: {ex}"}
    elif wire_res is None:
        wire_res = {"error": "another rank could not set up the wire-format run"}
    try:
        if "dg" in wire:
            wire["dg"].close()
        if "e3" in wire:
            wire["e3"].close()
    except Exception:  # noqa: BLE001
        pass
    wire.clear()
    pinned = None
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # timed region 1's table: nothing has folded on `eng` since its last step
        dump_outputs(args.dump_outputs, {"states": state_columns(eng.states_tensor().cpu().numpy())})
    e2.close(); eng.close()
    cpu_rec = np.array(host_log_np, copy=True) if (world == 1 and not args.no_cpu_baseline) else None
    del rec, host_log, host_log_np
    torch.cuda.empty_cache()

    if not routed_first:
        run_routed()
    configs = None
    if world == 1 and not args.no_configs:
        configs = {}
        for key, fn in (("configs[0]", lambda: config0_bank(dev, peak)), ("configs[3]", lambda: config3_zipf(dev, peak, args.scale)),
                        ("configs[4]", lambda: config4_microbatch(dev, 1000))):
            try:
                note(key)
                configs[key] = fn()
            except Exception as ex:  # noqa: BLE001
                configs[key] = {"error": f"{type(ex).__name__}: {ex}"}
            torch.cuda.empty_cache()

    # ---- max over ranks
    wire_ok = wire_res is not None and "seconds" in wire_res
    wire_s = wire_res["seconds"] if wire_ok else float("inf")
    if world > 1:
        t = torch.tensor([ms_total, e2e_s, wire_s if wire_ok else 1e30], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_s, wire_s = float(t[0]), float(t[1]), float(t[2])
        wire_ok = wire_s < 1e29
    value = world * n_events * K / (ms_total * 1e-3)
    e2e_packed_value = world * n_events * ke / e2e_s
    e2e_wire_value = world * n_events * ke / wire_s if wire_ok else None

    if rank == 0:
        achieved = b_alg / (kernel_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        for name in ("r02_fold_runs_traffic.json", "r01_fold_runs_traffic.json"):
            tp = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tp):
                try:
                    traffic = json.load(open(tp))["dram_bytes_per_launch"]
                    traffic_src = f"profiles/{name} (ncu --set full capture of the same kernel and shape; not re-measured in this run)"
                    break
                except Exception:  # noqa: BLE001
                    traffic = None
        out = {
            "metric": METRIC, "value": value, "unit": "events/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "aggregates_per_gpu": N_AGG, "events_per_aggregate": EVENTS_PER_AGG,
                       "record_bytes": 64, "state_bytes": STATE_BYTES, "model": "Counter (scaladsl TestBoundedContext)",
                       "l2": "inputs (2 GiB log per GPU) are 16x the 126 MB L2; no flush between iterations",
                       "sharding": "value: aggregates sharded across ranks, no data-path collective; the hash-partitioned configuration with "
                                   "its exchange (configs[2]) is the `routed` block (see DESIGN.md multi-GPU)"},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": b_alg, "kernel": "fold_runs_kernel",
                         "kernel_ms": kernel_ms, "peak_source": peak_src,
                         "pipelined_frac": (b_alg / (ms_total / K * 1e-3) / 1e9) / peak},
            # e2e: the events of the step enter as HOST bytes in the format the reference's topic holds (lz4 RecordBatch v2, what its
            # read_committed consumer is handed) through the public API a restore uses: sgr_dingest_submit* -> sgr_dingest_fold ->
            # sgr_export_states. e2e_packed_records is round 1's variant (pre-decoded 64-byte records over PCIe), kept for comparison.
            "e2e": ({"value": e2e_wire_value, "unit": "events/s", "h2d_bytes_per_step": int(wire_res["wire_bytes"]),
                     "d2h_bytes_per_step": int(N_AGG * STATE_BYTES + N_AGG * 24), "steps": ke, "ms_per_step": wire_s / ke * 1e3,
                     "input": "Kafka RecordBatch v2 bytes, lz4, 32 partitions x batches of 512 records, pinned host memory",
                     "wire_bytes_per_event": wire_res["bytes_per_event"], "pcie_gb_per_s_at_this_rate": wire_res["wire_bytes"] / (wire_s / ke) / 1e9,
                     "last_step_host_ms": wire_res.get("last_step_ms"), "host_ms_per_step": wire_res.get("host_ms_per_step"),
                     "parity": {"sample_aggregates": 4096, "sample_mismatches": wire_res["sample_mismatches"], "checked_against": "the HBM-resident fold's table, by aggregate id (sgr_get)"},
                     "api": "sgr_dingest_submit x 32 -> sgr_dingest_fold -> sgr_export_states (decode on the device: csrc/dingest_kernels.cu)"}
                    if wire_ok else
                    {"value": e2e_packed_value, "unit": "events/s", "h2d_bytes_per_step": int(log_bytes + host_off.nbytes), "d2h_bytes_per_step": int(N_AGG * STATE_BYTES),
                     "note": "wire-format leg failed: " + str((wire_res or {}).get("error")) + "; this is the packed-record path"}),
            "e2e_packed_records": {"value": e2e_packed_value, "unit": "events/s", "h2d_bytes_per_step": int(log_bytes + host_off.nbytes),
                    "d2h_bytes_per_step": int(N_AGG * STATE_BYTES), "steps": ke, "ms_per_step": e2e_s / ke * 1e3,
                    "ms_h2d": float(st2.ms_h2d), "ms_fold": float(st2.ms_fold), "ms_d2h": float(st2.ms_d2h),
                    # this variant's step is the PCIe copy of the 64-byte records: its rate is the bound of the number, not the kernel
                    "h2d_gb_per_s": (float(log_bytes + host_off.nbytes) / (float(st2.ms_h2d) * 1e-3) / 1e9) if st2.ms_h2d > 0 else None,
                    "h2d_share_of_step": (float(st2.ms_h2d) / (e2e_s / ke * 1e3)) if e2e_s > 0 else None},
            "clocks": clocks,
        }
        if routed is not None:
            out["routed"] = routed
        if configs is not None:
            out["configs"] = configs
        if cpu_rec is not None:
            cores = os.cpu_count() or 1
            v, reps, secs = time_cpu_oracle(cpu_rec, host_off, cores, min_seconds=8.0, max_reps=40)
            out["cpu_baseline"] = {"value": v, "unit": "events/s", "cores": cores, "kind": "port",
                                   "sample": f"full configs[1] log ({n_events} events, host memory first-touched by the pinned worker that folds it) x {reps} passes, "
                                             f"{secs:.1f} s, oracle/sgr_oracle.c with {cores} pinned threads"}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
