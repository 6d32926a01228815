#!/usr/bin/env python
"""bench.py -- the headline measurement and, as extra keys on the same JSON line, every other BASELINE.json
config at its BASELINE size (10 M rows per GPU), at every N.

  python bench.py --gpus N --steps K --warmup W          (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                   (the reference's CPU path, oracle port)

Headline (`value`, `roofline`, `e2e`): FP64 HOFM degree-3 (rank 32, explicit lower orders) predict + gradient
over a synthetic Criteo-shaped CSR (39 nnz/row, 1M hashed features) -- BASELINE.json config 4 / SURVEY 8d "C4" --
in samples/s.  A "step" is one predict+grad pass (zero grads -> fused forward + dloss + gradient scatter ->
loss/gb reduction [-> NCCL all-reduce of grad P/w when N>1]) over this rank's resident shard of `--rows` rows
(weak scaling: every rank holds its own 10M-row shard).

Extra keys (each measured in the same process, device time on the library's stream, MAX over ranks):
  parity_check   N>1 only, BEFORE any timing: the sharded MBPSGD / AdaGrad / minibatch-SGD / FFM paths on small
                 uneven shards against the CPU oracle (tests/sharded_parity.py); a failure exits non-zero
  c4_decision_function, c4_adagrad   the other two C4 paths (batched prediction; AdaGrad synchronous minibatch)
  c3_mbpsgd      FM degree 2 rank 16, MBPSGD logistic, epochs at three minibatch sizes
  c5_ffm         FFM rank 8, 39 fields: forward / predict+grad kernels, the all-reduced step, an AdaGrad epoch
  cd_epoch_s     C1 / C2 CD epochs on rank 0 (CD does not shard)
  uniform        N=1: the headline kernel on uniform-random columns (no cache help: the DRAM-bound case)
  e2e.pageable   the end-to-end call fed from PAGEABLE caller arrays (what a Nim seq is)
  cpu_baseline   N=1: the oracle port timed on the host cores, per config
See DESIGN.md "Measurement" for the byte accounting behind every `roofline`.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D_FEATURES = 1_000_000
Z = 39            # nnz per row: 13 numeric + 26 categorical slots
N_NUM, N_CAT = 13, 26
DEGREE, K, N_ORDERS = 3, 32, 2
# algorithmic bytes per row (SURVEY 8d; indices counted at the device width 4, every gathered or
# scattered parameter element once, no cache credit)
B_FWD = Z * (8 + 4 + 8 + 8 * K * N_ORDERS) + 8 + 8
B_GRAD = B_FWD + 8 + Z * (8 * K * N_ORDERS + 8)
B_ADA = Z * (8 + 4 + 40 + 40 * K * N_ORDERS) + 24
K3 = 16           # C3: FM degree 2 rank 16, one order
B3_FWD = Z * (8 + 4 + 8 + 8 * K3) + 16
B3_GRAD = B3_FWD + 8 + Z * (8 * K3 + 8)
N_FIELDS, K5 = 39, 8
B5_FWD = N_FIELDS * (8 + 4 + 4 + 8) + N_FIELDS * (N_FIELDS - 1) * 8 * K5 + 16
B5_GRAD = B5_FWD + 8 + N_FIELDS * (N_FIELDS - 1) * 8 * K5 + N_FIELDS * 8
B5_ADA = N_FIELDS * N_FIELDS * K5 * 40      # reference semantics: all fields x row features x k (SURVEY 8d)
# --dump-outputs: grad P columns of this many features (N_ORDERS * K * 8 B each: 32 MB in all)
DUMP_FEATURES, DUMP_SEED = 1 << 16, 2024


def gen_criteo_rows(n, seed, d=D_FEATURES, dist="criteo"):
    """Criteo-shaped synthetic CSR in the reference dtypes: 13 numeric slots (features 0..12, values
    U(0,1]) and 26 categorical slots, each with its own hashed id range and a Zipf(1.05)-like rank
    distribution (bounded inverse-CDF), value 1.0; indices sorted and unique within a row; y = +-1."""
    rng = np.random.default_rng(seed)
    R = (d - N_NUM) // N_CAT
    indices = np.empty((n, Z), dtype=np.int64)
    data = np.empty((n, Z), dtype=np.float64)
    indices[:, :N_NUM] = np.arange(N_NUM)[None, :]
    s = 1.05
    step = 1 << 20
    for a in range(0, n, step):
        b = min(n, a + step)
        data[a:b, :N_NUM] = 1.0 - rng.random((b - a, N_NUM))
        u = rng.random((b - a, N_CAT))
        rank = np.floor(((R ** (1.0 - s) - 1.0) * u + 1.0) ** (1.0 / (1.0 - s))).astype(np.int64) - 1
        np.clip(rank, 0, R - 1, out=rank)
        indices[a:b, N_NUM:] = N_NUM + np.arange(N_CAT)[None, :] * R + rank
    data[:, N_NUM:] = 1.0
    if dist != "criteo":   # experiments only (never the reported workload)
        R2 = d // Z
        for a in range(0, n, step):
            b = min(n, a + step)
            if dist == "uniform":      # every slot uniform over its own id range: no hot features at all
                rank = rng.integers(0, R2, size=(b - a, Z))
            else:                      # "zipfall": every slot Zipf-like, no always-present columns
                u = rng.random((b - a, Z))
                rank = np.floor(((R2 ** (1.0 - s) - 1.0) * u + 1.0) ** (1.0 / (1.0 - s))).astype(np.int64) - 1
                np.clip(rank, 0, R2 - 1, out=rank)
            indices[a:b] = np.arange(Z)[None, :] * R2 + rank
    indptr = np.arange(n + 1, dtype=np.int64) * Z
    y = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    return data.reshape(-1), indices.reshape(-1), indptr, y


def gen_ffm_rows(n, seed, n_fields=N_FIELDS, d=D_FEATURES):
    """libffm-shaped field CSR: one feature per field, field f owns its own contiguous id range with a
    Zipf(1.05)-like rank distribution; two thirds of the values are 1.0, the rest U(0,1); y = +-1."""
    rng = np.random.default_rng(seed)
    R = d // n_fields
    s = 1.05
    idx = np.empty((n, n_fields), dtype=np.int64)
    data = np.empty((n, n_fields), dtype=np.float64)
    step = 1 << 20
    for a in range(0, n, step):
        b = min(n, a + step)
        u = rng.random((b - a, n_fields))
        rank = np.floor(((R ** (1.0 - s) - 1.0) * u + 1.0) ** (1.0 / (1.0 - s))).astype(np.int64) - 1
        np.clip(rank, 0, R - 1, out=rank)
        idx[a:b] = np.arange(n_fields)[None, :] * R + rank
        v = rng.random((b - a, n_fields))
        data[a:b] = np.where(rng.random((b - a, n_fields)) < 0.66, 1.0, v)
    fields = np.tile(np.arange(n_fields, dtype=np.int64), n)
    y = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    return data.reshape(-1), idx.reshape(-1), np.arange(n + 1, dtype=np.int64) * n_fields, fields, y


def gen_ml100k(n=100_000, n_users=943, n_items=1682, seed=5):
    rng = np.random.default_rng(seed)
    u = rng.integers(0, n_users, n)
    v = rng.integers(0, n_items, n) + n_users
    idx = np.stack([u, v], axis=1).astype(np.int64)
    y = rng.integers(1, 6, n).astype(np.float64)
    return np.ones(2 * n), idx.reshape(-1), np.arange(n + 1, dtype=np.int64) * 2, y, n_users + n_items


def model_params(seed, d=D_FEATURES):
    rng = np.random.default_rng(seed)
    P = rng.standard_normal((N_ORDERS, K, d)) * 0.01      # newFactorizationMachine scale=0.01
    w = rng.standard_normal(d) * 0.01
    return P, w, 0.0


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_profile():
    """per-row counters of the dominant kernels from the committed `ncu --set full` captures (profiles/traffic.json:
    DRAM / L2 bytes per row and the capture each comes from), or {}"""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return {}
    return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines, self.t0 = index, None, [], 0.0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def mark(self):
        """the timed region begins now: nvidia-smi was started before the warm-up (its start-up takes longer than a
        short timed region), only samples that arrive from here on are reported"""
        self.t0 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t1 = time.time() + 0.06        # one sampling period of pipe latency
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if ts < self.t0 or ts > t1:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ====================================================================== CPU legs (oracle port, timed only)
def cpu_port_rate(orc, rows, seed, min_seconds, threads_note=True):
    """Time the oracle port of updateGradient (minibatch_psgd.nim:67-88 + sgd.nim:191-202), 1 thread,
    on `rows` rows of the same workload; returns (samples/s, rows used, seconds)."""
    from oracle.oracle import CSR
    data, indices, indptr, y = gen_criteo_rows(rows, seed)
    P, w, b = model_params(7)
    csr = CSR(data, indices, indptr, rows, D_FEATURES)
    Pf = orc.to_feature_major(P)
    del P
    gP, gw, gb = np.zeros_like(Pf), np.zeros(D_FEATURES), C.c_double(0.0)
    dA = np.zeros_like(Pf)
    lib = orc.lib()
    done, t0 = 0, time.perf_counter()
    chunk = max(1000, rows // 20)
    while done < rows:
        e = min(rows, done + chunk)
        lib.ref_fm_loss_grad(C.c_int64(D_FEATURES), orc._d(csr.data), orc._i(csr.indices), orc._i(csr.indptr),
                             orc._d(y), C.c_int64(done), C.c_int64(e), C.c_int(DEGREE), C.c_int(K), C.c_int(N_ORDERS),
                             C.c_int(0), C.c_int(1), C.c_int(1), orc._d(Pf), orc._d(w), C.c_double(b),
                             C.c_int(orc.LOSS["logistic"]), C.c_double(1.0), C.c_int64(rows), orc._d(gP), orc._d(gw),
                             C.byref(gb), None, orc._d(dA))
        done = e
        if time.perf_counter() - t0 > min_seconds and done >= chunk * 2:
            break
    dt = time.perf_counter() - t0
    return done / dt, done, dt


def cpu_hogwild_rate(orc, rows, seed, threads, reps=2):
    """Time the oracle port of the reference's multithreaded path for this workload: Hogwild AdaGrad
    epochs (adagrad_multi.nim:15-101: per sample predictWithGrad + lazy update + updateG, lock-free),
    `threads` threads over `rows` rows; optimizer state is allocated outside the timed call.
    Returns (samples/s of the best repetition, rows)."""
    from oracle.oracle import CSR
    data, indices, indptr, y = gen_criteo_rows(rows, seed)
    P, w, b = model_params(7)
    csr = CSR(data, indices, indptr, rows, D_FEATURES)
    Pf = orc.to_feature_major(P)
    del P
    lib = orc.lib()
    best = 0.0
    for _ in range(reps):
        gsP, gnP = np.zeros_like(Pf), np.full_like(Pf, 1e-10)
        gsw, gnw = np.zeros(D_FEATURES), np.full(D_FEATURES, 1e-10)
        gsb, gnb, bb = C.c_double(0.0), C.c_double(1e-10), C.c_double(b)
        itc, viol = C.c_int64(1), C.c_double(0.0)
        Pw, ww = Pf.copy(), w.copy()
        t0 = time.perf_counter()
        lib.ref_hogwild_adagrad_epoch(
            C.c_int(0), C.c_int64(rows), C.c_int64(D_FEATURES), orc._d(csr.data), orc._i(csr.indices),
            orc._i(csr.indptr), None, orc._d(y), C.c_int(DEGREE), C.c_int(K), C.c_int(N_ORDERS), C.c_int(0), C.c_int(0),
            C.c_int(1), C.c_int(1), orc._d(Pw), orc._d(ww), C.byref(bb), C.c_int(orc.LOSS["logistic"]), C.c_double(1.0),
            C.c_double(0.1), C.c_double(1e-6), C.c_double(1e-3), C.c_double(1e-3), C.byref(itc), orc._d(gsP), orc._d(gnP),
            orc._d(gsw), orc._d(gnw), C.byref(gsb), C.byref(gnb), None, C.c_int(threads), C.byref(viol))
        best = max(best, rows / (time.perf_counter() - t0))
    return best, rows


def hogwild_threads():
    """nThreads of sgd_multi.nim:13-18 for maxThreads < 0: 2 x countProcessors, capped by MaxThreadPoolSize (256)"""
    return min(2 * (os.cpu_count() or 1), 256)


def cpu_config_baselines(orc, budget_s=4.0):
    """The reference's own solvers for the other configs (oracle port, release flags), each on a bounded sample of
    the same synthetic workload: C1/C2 CD and C3 MBPSGD single-threaded (as the reference runs them), C5 FFM
    AdaGrad as Hogwild on 2 x cores threads (sgd_multi.nim:13-18)."""
    from oracle.oracle import CSR
    out = {}
    # C1 / C2: CD epochs (cd.nim:110-194), 1 thread
    data, idx, ptr, y, d = gen_ml100k()
    n = len(y)
    csc = orc.csr_to_csc(CSR(data, idx, ptr, n, d))
    for tag, degree in (("c1_cd_epoch_s", 2), ("c2_cd_epoch_s", 3)):
        P = np.random.default_rng(1).standard_normal((degree - 1, 30, d)) * 0.01
        t0 = time.perf_counter()
        orc.cd_fit(csc, y, P, np.zeros(d), 0.0, degree, "squared", max_iter=2, alpha0=1e-10, alpha=1e-10, beta=1e-3)
        out[tag] = (time.perf_counter() - t0) / 2
    # C3: one MBPSGD epoch (minibatch_psgd.nim:91-124) at the reference-default minibatch, 1 thread
    rows = 200_000
    data, idx, ptr, y = gen_criteo_rows(rows, 2000)
    csr = CSR(data, idx, ptr, rows, D_FEATURES)
    P = np.random.default_rng(2).standard_normal((1, K3, D_FEATURES)) * 0.01
    t0 = time.perf_counter()
    orc.mbpsgd_fit(csr, y, P, np.zeros(D_FEATURES), 0.0, 2, "logistic", max_iter=1, gamma=0.0, reg="identity", it=1)
    dt = time.perf_counter() - t0
    out["c3_mbpsgd_samples_per_s"] = rows / dt
    out["c3_sample"] = (f"{rows} rows, one epoch at the reference-default minibatch ({D_FEATURES * rows // (rows * Z)} rows: "
                        "the dense passes over P dominate, as in the reference)")
    # C5: Hogwild FFM AdaGrad (adagrad_ffm_multi.nim:16-104)
    rows = 20_000
    data, idx, ptr, fields, y = gen_ffm_rows(rows, 4000)
    csr = CSR(data, idx, ptr, rows, D_FEATURES, fields=fields, n_fields=N_FIELDS)
    Pf = np.ascontiguousarray(np.random.default_rng(3).standard_normal((N_FIELDS, D_FEATURES, K5)) * 0.01)
    T = hogwild_threads()
    t0 = time.perf_counter()
    orc.hogwild_adagrad_epoch(csr, y, Pf, np.zeros(D_FEATURES), 0.0, 2, T, is_ffm=True, loss_kind="logistic", n_rows=rows)
    out["c5_hogwild_adagrad_samples_per_s"] = rows / (time.perf_counter() - t0)
    out["c5_threads"] = T
    out["kind"] = "port (oracle restatement; Nim toolchain unavailable)"
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path.  The Nim toolchain is not
    in this image, so this is the oracle PORT of MBPSGD.updateGradient, which the reference runs on ONE
    thread (it has no multithreaded MBPSGD; its only threading is Hogwild SGD/AdaGrad)."""
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    sample_rows = args.ref_rows
    # each step is a bounded sample; size it so the whole run ends within minutes
    rate0, used0, dt0 = cpu_port_rate(orc, min(sample_rows, 20000), 123, 1.0)
    per_step = int(max(2000, min(sample_rows, rate0 * 2.0)))    # ~2 s per step
    times = []
    for s in range(args.warmup + args.steps):
        r, used, dt = cpu_port_rate(orc, per_step, 123, 1e9)
        if s >= args.warmup:
            times.append(dt / used)
    per_row = float(np.mean(times))
    single = 1.0 / per_row
    # all the host threads the reference can use on this workload: its Hogwild AdaGrad (the C4 solver)
    T = hogwild_threads()
    hog, hog_rows = cpu_hogwild_rate(orc, min(args.ref_rows * 4, 400_000), 123, T)
    value = max(single, hog)
    line = {
        "impl": "reference", "metric": "samples/sec FM/HOFM predict+grad", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_row * per_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world, per_step),
        "value_is": ("hogwild_adagrad (predict+grad AND the update, all host threads)" if hog >= single
                     else "single_thread_update_gradient (the same op as the GPU arm)"),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": T if hog >= single else 1, "kind": "port",
                         "sample": f"the faster of (a) {per_step} rows/step through the oracle port of "
                                   "minibatch_psgd.updateGradient on 1 thread (the reference's MBPSGD is "
                                   f"single-threaded): {single:.0f} samples/s, and (b) {hog_rows} rows through the "
                                   f"oracle port of its Hogwild AdaGrad (adagrad_multi.nim) on {T} threads: "
                                   f"{hog:.0f} samples/s; Nim toolchain unavailable",
                         "single_thread_update_gradient": single, "hogwild_adagrad": hog, "hogwild_threads": T,
                         "host_cores": os.cpu_count()},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def workload_config(args, world, rows_per_step):
    return {"workload": "C4: synthetic Criteo-shaped CSR (39 nnz/row, 1M hashed features), HOFM degree 3 "
                        "rank 32 explicit lower orders, logistic loss, predict+grad "
                        "(sgd.predictWithGrad + minibatch_psgd.updateGradient)",
            "rows_per_gpu": rows_per_step, "nnz_per_row": Z, "n_features": D_FEATURES, "degree": DEGREE,
            "rank": K, "n_orders": N_ORDERS, "parallelism": f"row-sharded x{world}, NCCL allreduce of grad P/w",
            "l2": "inputs larger than L2 (no flush needed)"}


# ====================================================================== the GPU arm
class Bench:
    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import nimfm_b200 as nf
        from nimfm_b200 import _lib, distributed as nd
        self.args, self.torch, self.dist, self.nf, self._lib, self.nd = args, torch, dist, nf, _lib, nd
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.lib = _lib.load()
        self.ctx = _lib.ctx(self.local_rank)
        nd.init_comm(self.rank, self.world)   # library-owned NCCL communicator (the id travels over torch.distributed)
        self.peak, self.peak_src = measured_peak()
        self.skip = set(x for x in args.skip.split(",") if x)

    # ---- plumbing
    def on(self, tag):
        return tag not in self.skip

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def maxr(self, v):
        t = self.torch.tensor([float(v)], device="cuda", dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    @staticmethod
    def l2_add(prof, payload_per_row, rows, backward_ms, kernel_ms=None):
        """the gradient scatter against the L2's measured FP64-add rate (scratch/red_rate.cu, profiles/r02_red_rate.txt):
        RED payload of the launch over the time the backward pass adds to the forward-only kernel"""
        hi, lo = prof.get("l2_fp64_add_ceiling_resident_GBs"), prof.get("l2_fp64_add_ceiling_missing_GBs")
        if not payload_per_row or not hi or backward_ms <= 0:
            return None
        ach = payload_per_row * rows / (backward_ms / 1e3) / 1e9
        out = {"red_payload_bytes_per_row": payload_per_row, "backward_ms": backward_ms, "achieved_GBs": ach,
               "ceiling_resident_lines_GBs": hi, "ceiling_missing_lines_GBs": lo, "frac_of_resident_ceiling": ach / hi,
               "note": "achieved = payload / (grad kernel - forward-only kernel), i.e. all of the extra time charged to "
                       "the scatter; over_whole_kernel = payload / grad kernel, the rate if the scatter overlapped the "
                       "forward pass completely -- the truth lies between",
               "source": prof.get("l2_fp64_add_source")}
        if kernel_ms:
            out["over_whole_kernel_GBs"] = payload_per_row * rows / (kernel_ms / 1e3) / 1e9
        return out

    def timed(self, fn, reps=1):
        """device time (ms) of `reps` calls of fn on the library's stream (CUDA events), MAX over ranks"""
        ms = C.c_float()
        self.barrier()
        self._lib.check(self.lib.nimfm_timer_start(self.ctx))
        for _ in range(reps):
            fn()
        self._lib.check(self.lib.nimfm_timer_stop(self.ctx, C.byref(ms)))
        return self.maxr(ms.value) / reps

    def frac(self, bytes_per_row, rows_per_s_per_gpu):
        return bytes_per_row * rows_per_s_per_gpu / 1e9 / self.peak

    # ---- parity of the sharded paths, before anything is timed (N > 1)
    def parity_check(self):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from oracle import oracle as orc
        if self.rank == 0:
            orc.build()
        self.barrier()
        import sharded_parity
        try:
            res = sharded_parity.run_checks(self.rank, self.world)
        except Exception as exc:   # a crash on one rank must not leave the others in a collective
            res = {"ok": False, "max_rel": float("inf"), "ranks": self.world, "failed": [repr(exc)], "cases": {}}
        ok = self.torch.tensor([1.0 if res["ok"] else 0.0, -res["max_rel"] if np.isfinite(res["max_rel"]) else -1e300],
                               device="cuda", dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(ok, op=self.dist.ReduceOp.MIN)
        res["ok"] = bool(ok[0].item() == 1.0)
        res["max_rel"] = float(-ok[1].item())
        res["what"] = ("tests/sharded_parity.py: decisionFunction, MBPSGD (L1 / L21: reduce-scatter + sharded step + "
                       "all-gather; SquaredL12: all-reduce), AdaGrad, minibatch SGD, FFM grad + AdaGrad on uneven "
                       "shards vs the CPU oracle; ok = every rank passed, max_rel = worst over ranks")
        return res

    # ---- C4: the headline + e2e + the other C4 paths
    def run_c4(self, line):
        args, lib, ctx, _lib, nf, world = self.args, self.lib, self.ctx, self._lib, self.nf, self.world
        n = args.rows
        t_gen = time.perf_counter()
        data, indices, indptr, y = gen_criteo_rows(n, 1000 + self.rank, dist=args.dist)
        ds = nf.newCSRDataset(data, indices, indptr, n, D_FEATURES)
        ds.set_targets(y)
        ds.handle()
        P, w, b = model_params(7)
        fm = nf.newFactorizationMachine(nf.classification, degree=DEGREE, nComponents=K, fitLower=nf.explicit)
        fm.P, fm.w, fm.intercept, fm.isInitialized = P, w, b, True
        h = fm._to_device(D_FEATURES)
        t_gen = time.perf_counter() - t_gen
        loss_kind = nf.Logistic().kind
        mb_global = n * world

        def step():
            ls = C.c_double()
            _lib.check(lib.nimfm_fm_loss_grad(ctx, h, ds.handle(), loss_kind, 1.0, 0, n, None, mb_global, 1,
                                              int(world > 1), C.byref(ls)))
            return ls.value

        sampler = ClockSampler(self.local_rank)
        sampler.start()
        for _ in range(args.warmup):
            step()
        self.barrier()
        sampler.mark()
        l0 = _lib.launch_count()
        _lib.check(lib.nimfm_timer_start(ctx))
        for _ in range(args.steps):
            loss_sum = step()
        ms = C.c_float()
        _lib.check(lib.nimfm_timer_stop(ctx, C.byref(ms)))
        launches = _lib.launch_count() - l0
        self.barrier()
        clocks = sampler.stop()
        if args.dump_outputs and self.rank == 0:
            dump_outputs(args.dump_outputs, self.c4_outputs(h, loss_sum))
        ms_per_step = self.maxr(ms.value) / args.steps
        value = n * world / (ms_per_step / 1e3)

        # ---- dominant kernel alone (CUDA events on the launching stream inside the library)
        kms, fms = C.c_float(), C.c_float()
        _lib.check(lib.nimfm_fm_time_loss_grad(ctx, h, ds.handle(), loss_kind, n, mb_global, max(args.steps, 3), 1, C.byref(kms)))
        _lib.check(lib.nimfm_fm_time_loss_grad(ctx, h, ds.handle(), loss_kind, n, mb_global, max(args.steps, 3), 0, C.byref(fms)))
        achieved = B_GRAD * n / (kms.value / 1e3) / 1e9
        prof = ncu_profile()
        dram_row = prof.get("fm_rows_grad_dram_bytes_per_row")
        l2_row = prof.get("fm_rows_grad_l2_bytes_per_row")
        # NOTE on frac > 1: `achieved` counts ALGORITHMIC bytes (every gathered / scattered parameter element once, no
        # cache credit, SURVEY 8d).  On the Zipf-shaped workload ~2/3 of those sectors hit L2, so the figure can
        # exceed the DRAM copy peak; `dram_frac` is the same launch's real DRAM traffic (ncu) over the peak, and the
        # `uniform` key below is the cache-free case where the two coincide.
        roofline = {"bound": "hbm", "kernel": "fm_rows_stream_kernel<3,true,MODE_GRAD,32>", "achieved": achieved,
                    "peak": self.peak, "unit": "GB/s", "frac": achieved / self.peak, "peak_source": self.peak_src,
                    "traffic": None if dram_row is None else dram_row * n,
                    "traffic_source": prof.get("fm_rows_grad_source"),
                    "dram_frac": None if dram_row is None else dram_row * n / (kms.value / 1e3) / 1e9 / self.peak,
                    "l2_bytes_per_row": l2_row,
                    "l2_GBs": None if l2_row is None else l2_row * n / (kms.value / 1e3) / 1e9,
                    "what_bounds_it": prof.get("fm_rows_grad_bound"),
                    "l2_fp64_add": self.l2_add(prof, prof.get("fm_rows_grad_red_payload_bytes_per_row"), n, kms.value - fms.value,
                                               kms.value),
                    "algorithmic_bytes_per_row": B_GRAD, "kernel_ms": kms.value,
                    "kernel_share_of_step": kms.value / ms_per_step, "frac_of_nominal_8TBs": achieved / 8000.0,
                    "forward_only": {"kernel": "fm_rows_stream_kernel<3,true,MODE_PREDICT,32>", "kernel_ms": fms.value,
                                     "samples_per_s": n / (fms.value / 1e3), "algorithmic_bytes_per_row": B_FWD,
                                     "achieved": B_FWD * n / (fms.value / 1e3) / 1e9,
                                     "frac": B_FWD * n / (fms.value / 1e3) / 1e9 / self.peak}}
        line.update({"value": value, "ms_per_step": ms_per_step, "clocks": clocks, "gpu_launches": int(launches),
                     "roofline": roofline, "loss_sum": loss_sum, "setup_seconds": t_gen})
        if self.on("det"):
            # the atomic-free route (csrc/fm_cols.cu) on the same step, timed beside the RED route
            os.environ["NIMFM_DETERMINISTIC"] = "1"
            try:
                t0 = time.perf_counter()
                det_loss = step()                          # first call builds the CSC twin + column segments
                first = time.perf_counter() - t0
                det_ms = self.timed(step, 2)
                det_loss2 = step()
            finally:
                del os.environ["NIMFM_DETERMINISTIC"]
            line["deterministic"] = {
                "samples_per_s": n * world / (det_ms / 1e3), "ms_per_step": det_ms, "first_call_seconds": first,
                "vs_red_route": ms_per_step / det_ms, "loss_sum": det_loss, "repeat_bit_identical": det_loss == det_loss2,
                "loss_sum_rel_diff_vs_red": abs(det_loss - loss_sum) / abs(loss_sum),
                "what": "NIMFM_DETERMINISTIC=1: stash-forward row kernel + column kernel over the CSC twin (every "
                        "gradient element summed in ascending row order, plain stores, no atomics), same step"}
        fwd_ms = self.maxr(fms.value)
        line["c4_decision_function"] = {"samples_per_s": n * world / (fwd_ms / 1e3), "kernel_ms": fwd_ms, "rows_per_gpu": n,
                                        "what": "batched decisionFunction kernel over the resident shards (no collective)",
                                        "frac": self.frac(B_FWD, n / (fwd_ms / 1e3))}
        if self.on("e2e"):
            self.run_e2e(line, h, data, indices, indptr, y, n, loss_kind)
        if self.on("c4_adagrad"):
            self.run_c4_adagrad(line, h, ds, n, loss_kind)
        lib.nimfm_fm_free(ctx, h)
        del fm, P, w
        if self.on("c3"):
            self.run_c3(line, ds, n, loss_kind)
        ds.free()

    def c4_outputs(self, h, loss_sum):
        """what the last timed step hands its caller: the loss sum and the gradient (all-reduced when N > 1).
        grad P is 512 MB, so only the columns of a fixed, seeded sample of features are kept."""
        gP, gw, gb = np.zeros((N_ORDERS, K, D_FEATURES)), np.zeros(D_FEATURES), C.c_double()
        self._lib.check(self.lib.nimfm_fm_get_grads(self.ctx, h, self._lib.ptr(gP), self._lib.ptr(gw), C.byref(gb)))
        feats = np.sort(np.random.default_rng(DUMP_SEED).choice(D_FEATURES, DUMP_FEATURES, replace=False))
        return {"loss_sum": np.array([loss_sum]), "grad_intercept": np.array([gb.value]), "grad_w": gw,
                "grad_P_sampled": np.ascontiguousarray(gP[:, :, feats]),
                "grad_P_sampled_features": feats.astype(np.float64)}

    def run_e2e(self, line, h, data, indices, indptr, y, n, loss_kind):
        """end to end through the C ABI with HOST buffers, H2D inside the timed region: caller-pinned arrays,
        PAGEABLE arrays (numpy == a Nim seq), and pageable arrays page-locked once (nimfm_host_register)"""
        args, lib, ctx, _lib, world, torch = self.args, self.lib, self.ctx, self._lib, self.world, self.torch
        ne = min(args.e2e_rows if args.e2e_rows > 0 else (10_000_000 if world == 1 else 2_000_000), n)
        host = [data[:ne * Z], indices[:ne * Z], indptr[:ne + 1], y[:ne]]
        nbytes = sum(a.nbytes for a in host)

        def run(ptrs, steps, predict_out=None):
            def one():
                if predict_out is not None:
                    _lib.check(lib.nimfm_fm_decision_function_host(ctx, h, ne, D_FEATURES, ptrs[0], ptrs[1], ptrs[2], 0,
                                                                   predict_out))
                    return 0.0
                ls = C.c_double()
                _lib.check(lib.nimfm_fm_loss_grad_host(ctx, h, ne, D_FEATURES, ptrs[0], ptrs[1], ptrs[2], ptrs[3], loss_kind,
                                                       1.0, ne * world, 0, 1, int(world > 1), C.byref(ls)))
                return ls.value
            one()
            one()          # (a fresh pageable result array is still being faulted in during the first call)
            self.barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                one()      # blocking: returns after the result has been read back
            torch.cuda.synchronize()
            dt = self.maxr(time.perf_counter() - t0)
            a, b_, t_ = C.c_int64(), C.c_int64(), C.c_int32()
            _lib.check(lib.nimfm_stream_stats(ctx, C.byref(a), C.byref(b_), C.byref(t_)))
            return ne * world * steps / dt, a.value, b_.value, t_.value

        # (1) caller-pinned
        hb = [torch.from_numpy(a).pin_memory() for a in host]
        hp = [C.c_void_p(t_.data_ptr()) for t_ in hb]
        v, h2d, d2h, thr = run(hp, args.e2e_steps)
        pred_host = torch.empty(ne, dtype=torch.float64).pin_memory()
        vp, ph2d, pd2h, _ = run(hp, args.e2e_steps, C.c_void_p(pred_host.data_ptr()))
        del hb, hp, pred_host
        # (2) pageable: the caller's numpy arrays as they are
        pp = [_lib.ptr(a) for a in host]
        vg, gh2d, gd2h, gthr = run(pp, args.e2e_steps)
        pred_pg = np.empty(ne)
        vgp, _, _, _ = run(pp, args.e2e_steps, _lib.ptr(pred_pg))
        # (3) pageable arrays page-locked once per dataset by the host layer
        t0 = time.perf_counter()
        for a in host:
            _lib.check(lib.nimfm_host_register(ctx, _lib.ptr(a), a.nbytes))
        t_reg = time.perf_counter() - t0
        vr, _, _, _ = run(pp, args.e2e_steps)
        for a in host:
            _lib.check(lib.nimfm_host_unregister(ctx, _lib.ptr(a)))
        line["e2e"] = {
            "value": v, "unit": "samples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "rows_per_step": ne, "host_bytes_per_step": int(nbytes), "host_staging_threads": int(thr),
            "host_memory": "caller-pinned arrays (the base contract's e2e); `pageable` is what a Nim seq gives",
            "pageable": {"value": vg, "h2d_bytes_per_step": int(gh2d), "d2h_bytes_per_step": int(gd2h),
                         "host_staging_threads": int(gthr),
                         "what": "the same call on PAGEABLE arrays (numpy == a Nim seq): values, ids and targets all go "
                                 "through the library's host staging threads into pinned slots"},
            "registered": {"value": vr, "register_seconds_once": t_reg,
                           "what": "the same pageable arrays after nimfm_host_register (page-locked once per dataset)"},
            "d2h_note": "the result read back per step is the loss sum (8 B); the gradient stays on the device for the "
                        "solver step",
            "note": "nimfm_fm_loss_grad_host: host CSR in the reference dtypes (f64 data, i64 indices/indptr, f64 y) -> "
                    "ids narrowed to int32 by the host staging threads -> chunked H2D overlapped with the kernel -> loss "
                    "read back; h2d/d2h bytes are what the library put on the link (nimfm_stream_stats)"}
        line["e2e_predict"] = {"value": vp, "unit": "samples/s", "h2d_bytes_per_step": int(ph2d), "d2h_bytes_per_step": int(pd2h),
                               "pageable": {"value": vgp, "what": "pageable arrays in, pageable result array out"},
                               "what": "nimfm_fm_decision_function_host: the same host CSR -> chunked H2D overlapped "
                                       "with the forward kernel -> predictions copied back"}

    def run_c4_adagrad(self, line, h, ds, n, loss_kind):
        lib, ctx, _lib, world = self.lib, self.ctx, self._lib, self.world
        local = min(self.args.adagrad_mb, n)
        # eta0 small: the synchronous variant accumulates SUMS over the minibatch (adagrad.nim:119-124 per sample),
        # so its first dual-averaging step scales like eta0 * sqrt(minibatch)
        cfg = _lib.AdagradCfg(loss_kind, 1.0, 1e-4, 1e-6, 1e-3, 1e-3, 1e-10, local)
        _lib.check(lib.nimfm_fm_adagrad_init(ctx, h, 1e-10, 1))
        it = C.c_int64(1)
        viol, ls = C.c_double(), C.c_double()

        def epoch():
            _lib.check(lib.nimfm_fm_adagrad_epoch(ctx, h, ds.handle(), C.byref(cfg), C.byref(it), None, n,
                                                  C.byref(viol), C.byref(ls)))
        epoch()                                        # the first epoch has no refresh pass on its first minibatch
        l0 = _lib.launch_count()
        ms = min(self.timed(epoch), self.timed(epoch))
        rate = n * world / (ms / 1e3)
        line["c4_adagrad"] = {"samples_per_s": rate, "s_per_epoch": ms / 1e3, "rows_per_gpu": n,
                              "minibatch_rows_per_gpu": local, "global_minibatch": local * world,
                              "epoch_loss": ls.value / (n * world), "gpu_launches_2_epochs": int(_lib.launch_count() - l0),
                              "algorithmic_bytes_per_row": B_ADA, "frac": self.frac(B_ADA, rate / world),
                              "what": "AdaGrad synchronous-minibatch epoch (count -> refresh -> row kernel -> "
                                      "[all-reduce of the delta block -> apply]), HOFM degree 3 rank 32, logistic"}

    def run_c3(self, line, ds, n, loss_kind):
        """C3: FM degree 2 rank 16, MBPSGD logistic (gamma = 0), epochs over the same Criteo-shaped shards"""
        lib, ctx, _lib, nf, world = self.lib, self.ctx, self._lib, self.nf, self.world
        rng = np.random.default_rng(2)
        P3 = rng.standard_normal((1, K3, D_FEATURES)) * 0.01
        w3 = np.zeros(D_FEATURES)
        fm = nf.newFactorizationMachine(nf.classification, degree=2, nComponents=K3, warmStart=True)
        fm.P, fm.w, fm.intercept, fm.isInitialized = P3, w3, 0.0, True
        h = fm._to_device(D_FEATURES)
        n_glob, nnz_glob = n * world, n * world * Z
        default_mb = max(D_FEATURES * n_glob // nnz_glob, 1)              # minibatch_psgd.nim:157-160
        out = {"what": "MBPSGD epoch (K2 per minibatch -> [reduce-scatter] -> step (+prox) -> [all-gather]), FM degree 2 "
                       "rank 16, logistic, gamma = 0; samples/s over all ranks", "rows_per_gpu": n,
               "algorithmic_bytes_per_row_sparse": B3_GRAD, "dense_step_bytes_per_minibatch": 4 * 8 * (K3 + 1) * D_FEATURES}
        variants = [("reference_default", default_mb, 400), ("256Ki_per_gpu", (1 << 18) * world, None),
                    ("1Mi_per_gpu", (1 << 20) * world, None)]
        for tag, mb, cap in variants:
            local = self.nd.local_batch(mb, self.rank, world)
            inner = max((n_glob - 1) // mb + 1, 1)                         # :161-164
            capped = cap is not None and inner > cap
            if capped:
                inner = cap
            _lib.check(lib.nimfm_fm_set_params(ctx, h, _lib.ptr(P3), _lib.ptr(w3), 0.0, None))
            cfg = _lib.MbpsgdCfg(loss_kind, 1.0, 0.1, 1e-6, 1e-3, 1e-4, 0.0, _lib.REG_L1, _lib.SCHED["optimal"], 1.0, mb, inner)
            it, ii, rl = C.c_int64(1), C.c_int64(0), C.c_double()

            def epoch():
                _lib.check(lib.nimfm_fm_mbpsgd_epoch(ctx, h, ds.handle(), C.byref(cfg), local, C.byref(it), C.byref(ii),
                                                     None, C.byref(rl)))
            epoch()
            l0 = _lib.launch_count()
            ms = min(self.timed(epoch), self.timed(epoch))
            rate = mb * inner / (ms / 1e3)
            out[tag] = {"global_minibatch": mb, "rows_per_gpu_per_minibatch": local, "inner_iterations": inner,
                        "inner_capped": capped, "s_per_epoch": ms / 1e3, "samples_per_s": rate,
                        "us_per_minibatch": ms * 1e3 / inner, "epoch_loss": rl.value,
                        "gpu_launches_2_epochs": int(_lib.launch_count() - l0),
                        "frac_sparse": self.frac(B3_GRAD, rate / world)}
        lib.nimfm_fm_free(ctx, h)
        line["c3_mbpsgd"] = out

    # ---- C5: FFM
    def run_c5(self, line):
        args, lib, ctx, _lib, nf, world = self.args, self.lib, self.ctx, self._lib, self.nf, self.world
        n = args.ffm_rows
        t0 = time.perf_counter()
        data, idx, ptr, fields, y = gen_ffm_rows(n, 6000 + self.rank)
        ds = nf.newCSRFieldDataset(data, idx, ptr, fields, n, D_FEATURES, N_FIELDS)
        ds.set_targets(y)
        ds.handle()
        del data, idx, fields
        base = np.random.default_rng(3).standard_normal((D_FEATURES, K5)) * 0.01
        P = np.empty((N_FIELDS, D_FEATURES, K5))
        for f in range(N_FIELDS):                       # distinct per field without 312 M normal draws
            np.multiply(base, 1.0 + 0.01 * f, out=P[f])
        m = nf.newFieldAwareFactorizationMachine(nf.classification, nComponents=K5, warmStart=True)
        m.P, m.w, m.intercept, m.isInitialized = P, np.zeros(D_FEATURES), 0.0, True
        h = m._to_device(ds)
        setup = time.perf_counter() - t0
        out = {"what": f"FFM {N_FIELDS} fields rank {K5}, one feature per field, d={D_FEATURES}, logistic; samples/s over "
                       "all ranks", "rows_per_gpu": n, "setup_seconds": setup}
        for tag, grad, bts in (("forward", 0, B5_FWD), ("predict_grad", 1, B5_GRAD)):
            ms = C.c_float()
            _lib.check(lib.nimfm_ffm_time_loss_grad(ctx, h, ds.handle(), 2, n, n * world, 2, grad, C.byref(ms)))
            t = self.maxr(ms.value)
            out[tag] = {"kernel_ms": t, "samples_per_s": n * world / (t / 1e3), "algorithmic_bytes_per_row": bts,
                        "frac": self.frac(bts, n / (t / 1e3))}
        # the pair gradient is z(z-1) vectors of k FP64 adds per row; against the L2's measured FP64-add rate
        out["predict_grad"]["l2_fp64_add"] = self.l2_add(ncu_profile(), N_FIELDS * (N_FIELDS - 1) * K5 * 8 + N_FIELDS * 8, n,
                                                         out["predict_grad"]["kernel_ms"] - out["forward"]["kernel_ms"],
                                                         out["predict_grad"]["kernel_ms"])
        ls = C.c_double()

        def step():
            _lib.check(lib.nimfm_ffm_loss_grad(ctx, h, ds.handle(), 2, 1.0, 0, n, None, n * world, 1, int(world > 1),
                                               C.byref(ls)))
        step()
        ms = self.timed(step, 2)
        out["step"] = {"ms_per_step": ms, "samples_per_s": n * world / (ms / 1e3),
                       "what": "zero grads + pair kernel + all-reduce of [gP | gw | gb, loss] (2.5 GB)",
                       "frac": self.frac(B5_GRAD, n / (ms / 1e3))}
        local = min(args.adagrad_mb, n)
        cfg = _lib.AdagradCfg(2, 1.0, 1e-4, 1e-6, 1e-3, 1e-3, 1e-10, local)
        _lib.check(lib.nimfm_ffm_adagrad_init(ctx, h, 1e-10, 1))
        it, viol = C.c_int64(1), C.c_double()

        def epoch():
            _lib.check(lib.nimfm_ffm_adagrad_epoch(ctx, h, ds.handle(), C.byref(cfg), C.byref(it), None, n, C.byref(viol),
                                                   C.byref(ls)))
        epoch()
        ms = self.timed(epoch)
        rate = n * world / (ms / 1e3)
        out["adagrad"] = {"samples_per_s": rate, "s_per_epoch": ms / 1e3, "minibatch_rows_per_gpu": local,
                          "epoch_loss": ls.value / (n * world), "algorithmic_bytes_per_row": B5_ADA,
                          "frac": self.frac(B5_ADA, rate / world),
                          "what": "AdaGrad synchronous-minibatch epoch (count -> refresh -> pair kernel, gradient blocks "
                                  "added by TMA bulk reductions -> [all-reduce of the 5 GB delta block -> apply])"}
        lib.nimfm_ffm_free(ctx, h)
        ds.free()
        line["c5_ffm"] = out

    # ---- C1 / C2: CD on rank 0 (the coordinate loop is sequential: it does not shard)
    def run_cd(self, line):
        nf, _lib = self.nf, self._lib
        if self.rank == 0:
            data, idx, ptr, y, d = gen_ml100k()
            n = len(y)
            order = np.argsort(idx, kind="stable")          # CSC of the 2-nnz-per-row CSR (columns ascending, rows stable)
            csc_idx = (order // 2).astype(np.int64)
            csc_ptr = np.concatenate([[0], np.cumsum(np.bincount(idx, minlength=d))]).astype(np.int64)
            ds = nf.newCSCDataset(np.ones(2 * n), csc_idx, csc_ptr, n, d)
            out = {"what": f"CD epoch seconds, ML-100K shape n={n} d={d} nnz={2 * n}, rank 30, squared loss (rank 0 only: "
                           "CD stays single-GPU)"}
            for tag, degree in (("c1", 2), ("c2", 3)):
                P = np.random.default_rng(1).standard_normal((degree - 1, 30, d)) * 0.01
                kw = dict(alpha0=1e-10, alpha=1e-10, beta=1e-3)
                fm = nf.newFactorizationMachine(nf.regression, degree=degree, nComponents=30, warmStart=True)
                fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), np.zeros(d), 0.0, True
                nf.newCD(maxIter=1, verbose=0, tol=0.0, **kw).fit(ds, y, fm)       # warm-up (batches, graph capture)
                fm.P, fm.w, fm.intercept = P.copy(), np.zeros(d), 0.0
                opt = nf.newCD(maxIter=5, verbose=0, tol=0.0, **kw)
                l0 = _lib.launch_count()
                opt.fit(ds, y, fm)
                ep = float(np.median(opt.epoch_seconds))
                steps = (degree - 1) * 30 * d + d + 1
                out[tag] = {"degree": degree, "epoch_s": ep, "coordinate_steps_per_epoch": steps,
                            "us_per_coordinate_step": ep / steps * 1e6,
                            "objective_after_5_epochs": opt.history[-1][1] + opt.history[-1][2],
                            "kernel_launches_per_epoch": (_lib.launch_count() - l0) / 5}
            ds.free()
            line["cd_epoch_s"] = out["c2"]["epoch_s"]
            line["cd"] = out
        self.barrier()

    # ---- the per-sample solvers (SGD, AdaGrad miniBatchSize=1, PSGD): strictly sequential in the reference, one
    # persistent thread block here ("replicas only" for multi-GPU) -- rank 0, with the oracle's loops timed beside it
    def run_seq(self, line):
        nf = self.nf
        if self.rank == 0:
            n = 50_000
            data, idx, ptr, y = gen_criteo_rows(n, 2000)
            ds = nf.newCSRDataset(data, idx, ptr, n, D_FEATURES)
            P, w, b = model_params(7)
            kw = dict(maxIter=2, loss=nf.Logistic(), verbose=0, tol=0.0, shuffle=False)
            solvers = (("sgd", lambda: nf.newSGD(eta0=0.01, **kw)),
                       ("adagrad_mb1", lambda: nf.newAdaGrad(eta0=0.1, miniBatchSize=1, **kw)),
                       ("psgd_l1", lambda: nf.newPSGD(eta0=0.01, gamma=1e-5, reg=nf.newL1(), **kw)),
                       ("psgd_l21", lambda: nf.newPSGD(eta0=0.01, gamma=1e-5, reg=nf.newL21(), **kw)))
            out = {"what": f"samples/s of one epoch over {n} C4-shape rows (degree 3, k = 32), one GPU: the reference's "
                           "per-sample loops (sgd.nim:255-338, adagrad.nim:164-181, psgd.nim:76-215), same iterates",
                   "rows": n}
            for tag, mk in solvers:
                fm = nf.newFactorizationMachine(nf.classification, degree=DEGREE, nComponents=K, warmStart=True)
                fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), b, True
                opt = mk()
                opt.fit(ds, y, fm)
                ep = float(np.min(opt.epoch_seconds))
                out[tag] = {"samples_per_s": n / ep, "s_per_epoch": ep}
            ds.free()
            if not self.args.no_cpu_baseline:
                from oracle import oracle as orc
                from oracle.oracle import CSR
                orc.build()
                m = 20_000
                csr = CSR(data[:ptr[m]], idx[:ptr[m]], ptr[:m + 1], m, D_FEATURES)
                cpu = {"rows": m, "kind": "port, one thread (the loops are sequential in the reference too)"}
                for tag, fn in (("sgd", lambda: orc.sgd_fit(csr, y[:m], P, w, b, DEGREE, "logistic", max_iter=1, eta0=0.01)),
                                ("adagrad_mb1", lambda: orc.adagrad_fit(csr, y[:m], P, w, b, DEGREE, "logistic", max_iter=1,
                                                                        eta0=0.1, mini_batch_size=1)),
                                ("psgd_l1", lambda: orc.psgd_fit(csr, y[:m], P, w, b, DEGREE, "logistic", max_iter=1,
                                                                 eta0=0.01, gamma=1e-5, reg="l1"))):
                    t0 = time.perf_counter()
                    fn()
                    cpu[tag] = m / (time.perf_counter() - t0)
                out["cpu"] = cpu
            line["sequential_solvers"] = out
        self.barrier()

    # ---- the headline kernel without cache help
    def run_uniform(self, line):
        args, lib, ctx, _lib, nf = self.args, self.lib, self.ctx, self._lib, self.nf
        n = min(args.uniform_rows, args.rows)
        data, indices, indptr, y = gen_criteo_rows(n, 77, dist="uniform")
        ds = nf.newCSRDataset(data, indices, indptr, n, D_FEATURES)
        ds.set_targets(y)
        P, w, b = model_params(7)
        fm = nf.newFactorizationMachine(nf.classification, degree=DEGREE, nComponents=K, fitLower=nf.explicit)
        fm.P, fm.w, fm.intercept, fm.isInitialized = P, w, b, True
        h = fm._to_device(D_FEATURES)
        kms, fms = C.c_float(), C.c_float()
        _lib.check(lib.nimfm_fm_time_loss_grad(ctx, h, ds.handle(), 2, n, n, 3, 1, C.byref(kms)))
        _lib.check(lib.nimfm_fm_time_loss_grad(ctx, h, ds.handle(), 2, n, n, 3, 1, C.byref(kms)))
        _lib.check(lib.nimfm_fm_time_loss_grad(ctx, h, ds.handle(), 2, n, n, 3, 0, C.byref(fms)))
        prof = ncu_profile()
        dram_row = prof.get("fm_rows_grad_uniform_dram_bytes_per_row")
        g = B_GRAD * n / (kms.value / 1e3) / 1e9
        line["uniform"] = {"what": "the headline kernels on uniform-random column ids (every slot uniform over its own id "
                                   "range: no hot features, no L2 reuse) -- the DRAM-bound case", "rows": n,
                           "grad": {"kernel_ms": kms.value, "samples_per_s": n / (kms.value / 1e3), "achieved": g,
                                    "frac": g / self.peak, "dram_bytes_per_row": dram_row,
                                    "dram_frac": None if dram_row is None else dram_row * n / (kms.value / 1e3) / 1e9 / self.peak,
                                    "traffic_source": prof.get("fm_rows_grad_uniform_source")},
                           "forward": {"kernel_ms": fms.value, "samples_per_s": n / (fms.value / 1e3),
                                       "frac": B_FWD * n / (fms.value / 1e3) / 1e9 / self.peak}}
        lib.nimfm_fm_free(ctx, h)
        ds.free()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000, help="rows per GPU (weak scaling)")
    ap.add_argument("--ffm-rows", type=int, default=10_000_000, help="FFM rows per GPU")
    ap.add_argument("--uniform-rows", type=int, default=4_000_000)
    ap.add_argument("--adagrad-mb", type=int, default=1 << 19, help="AdaGrad rows per GPU per synchronous minibatch")
    ap.add_argument("--e2e-rows", type=int, default=0,
                    help="rows per end-to-end step (host buffers); default: the whole 10 M-row batch of the "
                         "device-resident step on one GPU, 2 M rows per rank under torchrun (pinned host memory "
                         "of 8 ranks on one box)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="bounded CPU-baseline sample")
    ap.add_argument("--ref-rows", type=int, default=100_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip", default="", help="comma list of sections to skip: parity,det,e2e,c4_adagrad,c3,c5,cd,seq,uniform")
    ap.add_argument("--dist", default="criteo", choices=["criteo", "uniform", "zipfall"],
                    help="index distribution; anything but 'criteo' is an experiment, not the reported workload")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed headline step returned (loss sum, gradient; grad P at a fixed "
                         "sample of features) to DIR/<name>.npy as float64, for comparing two builds on the same "
                         "seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    B = Bench(args)
    line = {
        "metric": "samples/sec FM/HOFM predict+grad", "value": None, "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world, args.rows),
    }
    if args.dist != "criteo":
        line["config"]["experiment_dist"] = args.dist
    if world > 1 and B.on("parity"):
        line["parity_check"] = B.parity_check()
        if not line["parity_check"]["ok"]:
            if rank == 0:
                print(json.dumps(line), flush=True)
            B.barrier()
            sys.exit(3)
    B.run_c4(line)
    if B.on("c5"):
        B.run_c5(line)
    if B.on("cd"):
        B.run_cd(line)
    if world == 1 and B.on("seq"):
        B.run_seq(line)          # sequential solvers do not shard ("replicas only"): measured at N = 1
    elif B.on("seq"):
        line["sequential_solvers"] = {"skipped": "per-sample SGD / AdaGrad / PSGD are sequential (replicas only): "
                                                 "the host mirror refuses them while a communicator is up; see the N = 1 line"}
    if world == 1 and B.on("uniform"):
        B.run_uniform(line)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as orc
        orc.build()
        rate, used, dt = cpu_port_rate(orc, 1_500_000, 1000, args.cpu_seconds)
        T = hogwild_threads()
        hog, hog_rows = cpu_hogwild_rate(orc, 300_000, 1000, T, reps=1)
        line["cpu_baseline"] = {"value": rate, "unit": "samples/s", "cores": 1, "kind": "port",
                                "hogwild_adagrad": {"value": hog, "threads": T, "rows": hog_rows,
                                                    "what": "oracle port of adagrad_multi.nim (the reference's "
                                                            "multithreaded path), racy by design, timed only"},
                                "sample": f"first {used} rows of the same workload in {dt:.1f} s, oracle port of "
                                          "minibatch_psgd.updateGradient + sgd.predictWithGrad (the reference "
                                          "runs MBPSGD on one thread)", "host_cores": os.cpu_count(),
                                "configs": cpu_config_baselines(orc)}
        # the two ratios side by side: the same op on one thread, and the reference's all-threads solver
        line["vs_cpu"] = {"predict_grad_vs_single_thread_update_gradient": line["value"] / rate,
                          "e2e_vs_single_thread_update_gradient": line["e2e"]["value"] / rate if "e2e" in line else None,
                          "c4_adagrad_vs_hogwild_adagrad": (line["c4_adagrad"]["samples_per_s"] / hog
                                                            if "c4_adagrad" in line else None)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        B.dist.destroy_process_group()


if __name__ == "__main__":
    main()
