#!/usr/bin/env python
"""bench.py — PIR server queries/sec on the "1 GiB DB" Spiral workload (BASELINE.json configs[1]).

A step = one pass of the hot path (spiral_rs::server::process_query, lib/spiral-rs/src/server.rs:650-741)
over one batch of `--batch` synthetic queries against the HBM-resident database.

  * `value`     : queries/s with the queries already resident in HBM (device-timed, CUDA events,
                  barrier + synchronize on both sides, max over ranks)
  * `e2e`       : the same metric through the reference-facing C-ABI call b200pir_process_query_bytes with HOST buffers
                  (pinned): `batch` serialized queries (Query::serialize wire format, 16 416 bytes each) in, response
                  bytes out; deserialization (ChaCha20 seed expansion), H2D and D2H are inside the timed region
  * `roofline`  : the dominant kernel (multiply_reg_by_database, server.rs:155-221), algorithmic bytes
                  per launch / its CUDA-event duration measured live in the timed region, against the
                  measured HBM peak of MEASURED_PEAKS.json
  * `cpu_baseline` / `--impl reference` : the CPU restatement of the reference (oracle/, "port": no Rust
                  toolchain exists in the image) on the host cores: FULL process_query calls on the same parameter set
                  (measured, one query at a time as the reference processes them), with the bounded-sample extrapolation
                  of round 1 beside it

Workloads (SURVEY.md §8 table): N=1 -> S8 = 2^17 Spiral items x 8 KiB = 2^20 x 1 KiB records, 1 GiB of
plaintext = 8 GiB HBM-resident.  N>1 (strong scaling) -> the SAME database with its second-dimension rows
sharded ii mod N (1/N of the bytes per GPU), the same `--batch` queries per step: every rank expands the
queries it received, NCCL all-gathers the expanded queries and, after the local first dimension + fold
rounds, the surviving ciphertexts; each rank finishes its own queries (DESIGN.md "multi-GPU").

Synthetic data: the server computation is data-oblivious, so public parameters and query ciphertexts
are uniformly random residues of the right shape; the database is generated on the GPU from a
counter PRNG (plaintext -> NTT -> packed words).  Correctness is covered by tests/, not here.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# NCCL prints its version banner on stdout at VERSION level; stdout must carry exactly one JSON line
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"

Q0, Q1 = 268369921, 249561089
POLY = 2048

S8 = dict(n=2, nu_1=9, nu_2=8, p=256, q2_bits=22, t_gsw=8, t_conv=4, t_exp_left=8, t_exp_right=8, instances=1,
          db_item_size=8192, version=0)
WORKLOADS = {
    "S8": S8,                                     # 8 GiB HBM-resident = 1 GiB plaintext (configs[1])
    "S1": dict(n=2, nu_1=9, nu_2=5, p=256, q2_bits=22, t_gsw=7, t_conv=3, t_exp_left=5, t_exp_right=5, instances=1,
               db_item_size=8192, version=1),     # 1 GiB HBM-resident
    # configs[2]: 32 GiB plaintext = 256 GiB of packed words, row-sharded over 8 GPUs (32 GiB per GPU)
    "S256": dict(n=2, nu_1=10, nu_2=12, p=256, q2_bits=22, t_gsw=8, t_conv=4, t_exp_left=8, t_exp_right=8, instances=1,
                 db_item_size=8192, version=0),
    "T": dict(n=2, nu_1=6, nu_2=2, p=256, q2_bits=20, t_gsw=8, t_conv=4, t_exp_left=8, t_exp_right=8, instances=1,
              db_item_size=8192, version=0),      # unit-test size (CI smoke of this script)
}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def derived(kw):
    import math
    dim0, num_per = 1 << kw["nu_1"], 1 << kw["nu_2"]
    slices = kw["instances"] * kw["n"] ** 2
    g = math.ceil(math.log2(kw["t_gsw"] * kw["nu_2"] + dim0))
    stop_round = math.ceil(math.log2(kw["t_gsw"] * kw["nu_2"])) if kw["nu_2"] else 0
    num_packing = kw["n"] if kw["version"] == 0 else 2
    has_right = kw["version"] == 0 or kw["t_exp_right"] != kw["t_exp_left"]
    return dict(dim0=dim0, num_per=num_per, slices=slices, g=g, stop_round=stop_round, num_packing=num_packing,
                has_right=has_right)


def random_ntt(rng, npolys):
    import numpy as np
    a = np.empty((npolys, 2, POLY), dtype=np.uint64)
    a[:, 0, :] = rng.integers(0, Q0, (npolys, POLY), dtype=np.uint64)
    a[:, 1, :] = rng.integers(0, Q1, (npolys, POLY), dtype=np.uint64)
    return a.reshape(-1)


def synthetic_pp(kw, rng):
    d = derived(kw)
    pp = dict(pack=random_ntt(rng, d["num_packing"] * (kw["n"] + 1) * kw["t_conv"]),
              left=random_ntt(rng, d["g"] * 2 * kw["t_exp_left"]),
              right=random_ntt(rng, (d["stop_round"] + 1) * 2 * kw["t_exp_right"]) if d["has_right"] else None,
              conv=random_ntt(rng, 2 * 2 * kw["t_conv"]))
    return pp


class ClockSampler:
    """nvidia-smi sampler running during the timed region (B200_PROFILING.md 'clocks line')."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def wait_first(self, timeout=15.0):
        """nvidia-smi needs up to seconds to start (longer on an 8-GPU box): do not enter the timed region before its first line,
        or a short region ends unsampled."""
        t = time.time()
        while self.proc is not None and not self.lines and self.proc.poll() is None and time.time() - t < timeout:
            time.sleep(0.02)

    def stop(self, t0, t1):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        sm, smax, reasons = [], 0.0, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ts, line in self.lines:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1]))
                smax = max(smax, float(f[2]))
                for name, val in zip(names, f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_SAMPLE = 1 << 20      # --dump-outputs: elements kept of a larger output (at most 8 MB per array as float64)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: write each output of the timed path's last step as <out_dir>/<name>.npy, so that two builds run with the
    same arguments (hence the same inputs) can be compared output for output.  Bytes become float32, wider integers float64
    (int32 buffers hold u32 words), both exact.  An output of more than DUMP_SAMPLE elements is cut down to the elements at a
    fixed, seeded set of flat positions, the same in every run."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = torch.as_tensor(a)
        if a.numel() > DUMP_SAMPLE:
            pos = np.sort(np.random.default_rng(1).choice(a.numel(), DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[torch.from_numpy(pos).to(a.device)]
        h = a.cpu().numpy()
        if h.dtype == np.int32:
            h = h.view(np.uint32)
        np.save(os.path.join(out_dir, name + ".npy"), h.astype(np.float32 if h.dtype.itemsize == 1 else np.float64))


def ncu_traffic(workload, batch, db_format):
    """dram bytes per launch of the multiply kernel from the committed ncu --set full capture of this configuration, if any
    (profiles/roofline_traffic.json; key = workload, queries per step, database format)."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            d = json.load(f)
        return d.get("%s_batch%d_format%d" % (workload, batch, db_format))
    except Exception:
        return None


# ------------------------------------------------------------------------------------------- CPU legs
def cpu_process_query_sample(kw, threads=None, sample_rows=64):
    """Time the oracle's process_query (CPU restatement of the reference) on a bounded sample:
    the full query expansion plus a `sample_rows`-row slab of every slice (multiply + fold + pack),
    scaling the row-proportional part to the full num_per.  Returns seconds per query (estimate)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import oracle_lib as O
    simd = "AVX2 first dimension" if O.LIB.orc_use_avx2_multiply(1) else "scalar first dimension"
    simd += " and transforms" if O.LIB.orc_use_avx2_ntt(1) else ", scalar transforms"
    if threads:
        O.LIB.orc_set_num_threads(int(threads))
    else:
        # pick the thread count that serves the CPU path best (all logical CPUs often lose to one thread per core)
        ncpu = os.cpu_count() or 1
        ckw = dict(kw, nu_2=min(3, kw["nu_2"]))
        cal = O.Params(**ckw)
        cal_rng = np.random.default_rng(3)
        cal_pp = synthetic_pp(ckw, cal_rng)
        cal_q = dict(ct=cal_rng.integers(0, cal.modulus, 2 * POLY, dtype=np.uint64))
        cal_db = cal_rng.integers(0, Q1, cal.slices * cal.dim0 * cal.num_per * POLY, dtype=np.uint64)
        best = None
        for t in sorted({ncpu, max(ncpu // 2, 1), max(ncpu // 4, 1)}, reverse=True):
            O.LIB.orc_set_num_threads(t)
            t0 = time.perf_counter()
            cal.process_query(cal_pp, cal_q, cal_db)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, t)
        O.LIB.orc_set_num_threads(best[1])
    cores = int(O.LIB.orc_num_threads())
    full_rows = 1 << kw["nu_2"]
    rows = min(sample_rows, full_rows)
    skw = dict(kw)
    skw["nu_2"] = rows.bit_length() - 1
    P = O.Params(**skw)
    Pfull = O.Params(**kw)
    rng = np.random.default_rng(7)
    pp = synthetic_pp(skw, rng)
    pp_full = synthetic_pp(kw, rng)
    q = dict(ct=rng.integers(0, P.modulus, 2 * POLY, dtype=np.uint64))
    db = (rng.integers(0, Q0, P.slices * P.dim0 * P.num_per * POLY, dtype=np.uint64)
          | (rng.integers(0, Q1, P.slices * P.dim0 * P.num_per * POLY, dtype=np.uint64) << np.uint64(32)))
    t0 = time.perf_counter()
    Pfull.expand_query(pp_full, q["ct"])                       # full-size expansion (g rounds of the real config)
    t_expand_full = time.perf_counter() - t0
    # the row-proportional part, timed directly on the sample slab: multiply + from_ntt + fold per slice, pack, encode
    vreg, vf = P.expand_query(pp, q["ct"])
    slice_words = P.dim0 * P.num_per * POLY
    use_avx2 = simd.startswith("AVX2")
    t0 = time.perf_counter()
    vfn = P.get_v_folding_neg(vf)
    folded = []
    for sl in range(P.slices):
        dsl = db[sl * slice_words:(sl + 1) * slice_words]
        if use_avx2:
            mult = np.zeros(P.num_per * 4 * POLY, dtype=np.uint64)
            O._ck(O.LIB.orc_multiply_reg_by_database_avx2(P.hp, O._p64(mult), O._p64(dsl), O._p64(vreg),
                                                          O.C.c_size_t(P.dim0), O.C.c_size_t(P.num_per)))
        else:
            mult = P.multiply_reg_by_database(dsl, vreg)
        raw = P.from_ntt(mult)
        folded.append(P.fold_ciphertexts(raw, vf, vfn)[: 2 * POLY])
    t_rows = time.perf_counter() - t0
    t0 = time.perf_counter()
    nn = P.n * P.n
    packed = [P.from_ntt(P.pack(np.concatenate(folded[i * nn:(i + 1) * nn]), pp["pack"])) for i in range(P.instances)]
    P.encode(np.concatenate(packed))
    t_tail = time.perf_counter() - t0
    est = t_expand_full + t_rows * (full_rows / rows) + t_tail
    sample = ("oracle process_query (" + simd + ", OpenMP): full query expansion (%.2fs) + %d of %d second-dimension "
              "rows of every slice (multiply+from_ntt+fold %.2fs, scaled x%d) + pack/encode (%.3fs)"
              % (t_expand_full, rows, full_rows, t_rows, full_rows // rows, t_tail))
    return est, cores, sample


class CpuFullQuery:
    """The oracle's process_query (CPU restatement of the reference, AVX2 + OpenMP) on the FULL parameter set: one call = one
    query against the whole database, exactly what the reference's /private-read handler does per request.  The database
    is a host array of the right size (a random block tiled: the computation is data-oblivious)."""

    def __init__(self, kw, threads=None):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import numpy as np
        import oracle_lib as O
        self.O, self.np = O, np
        self.simd = "AVX2 first dimension" if O.LIB.orc_use_avx2_multiply(1) else "scalar first dimension"
        self.simd += " and transforms" if O.LIB.orc_use_avx2_ntt(1) else ", scalar transforms"
        rng = np.random.default_rng(7)
        self.P = O.Params(**kw)
        self.pp = synthetic_pp(kw, rng)
        self.q = dict(ct=rng.integers(0, self.P.modulus, 2 * POLY, dtype=np.uint64))
        words = self.P.slices * self.P.dim0 * self.P.num_per * POLY
        block = min(words, 1 << 22)
        blk = (rng.integers(0, Q0, block, dtype=np.uint64) | (rng.integers(0, Q1, block, dtype=np.uint64) << np.uint64(32)))
        self.db = np.tile(blk, words // block) if words > block else blk
        self.db_bytes = self.db.nbytes
        ncpu = os.cpu_count() or 1
        if threads:
            O.LIB.orc_set_num_threads(int(threads))
        else:
            # pick the thread count that serves the CPU path best (all logical CPUs often lose to one thread per core)
            best = None
            for t in sorted({ncpu, max(ncpu // 2, 1)}, reverse=True):
                O.LIB.orc_set_num_threads(t)
                dt = self.one()
                if best is None or dt < best[0]:
                    best = (dt, t)
            O.LIB.orc_set_num_threads(best[1])
        self.cores = int(O.LIB.orc_num_threads())

    def one(self):
        t0 = time.perf_counter()
        self.response = self.P.process_query(self.pp, self.q, self.db)
        return time.perf_counter() - t0

    def sample(self, n):
        return ("oracle process_query (%s, OpenMP, %d threads): %d full quer%s against the whole %.2f GiB database, one at a "
                "time (measured, not extrapolated)" % (self.simd, self.cores, n, "y" if n == 1 else "ies", self.db_bytes / 2**30))


def run_reference_arm(args, kw, workload_name, rank, world):
    if rank != 0:
        return
    cpu = CpuFullQuery(kw)
    per_step = []
    for i in range(args.warmup + args.steps):
        dt = cpu.one()                       # a step = one full process_query on the host cores
        if i >= args.warmup:
            per_step.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"responses": cpu.response.reshape(1, -1)})
    sec = sum(per_step) / len(per_step)
    qps = 1.0 / sec
    cores, sample = cpu.cores, cpu.sample(len(per_step))
    out = {
        "impl": "reference", "metric": "PIR server queries/sec (Spiral process_query)", "value": qps, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name, "params": kw, "batch": 1},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------- kernel-level workloads
def kernel_workload(args):
    """BASELINE configs #4 (DoublePIR 2^24 x 1366 packed words, HBM GB/s vs roofline) and #5 (NTT / INTT throughput, poly_len
    2048 and 4096, 2^16 polynomials x 2 CRT moduli) as bench lines: `--workload dpir`, `--workload ntt`.  Single GPU."""
    import ctypes as C
    import numpy as np
    import torch
    import sdk_b200.spiral as S
    import sdk_b200.doublepir as D
    from sdk_b200._lib import LIB, check
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    peak, peak_src = measured_peak()
    stream = torch.cuda.current_stream()

    def timed(fn):
        for _ in range(max(args.warmup, 3)):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    sampler = ClockSampler(0)
    sampler.start()
    sampler.wait_first()
    t0 = time.time()
    if args.workload == "dpir":
        rows, cols = 1 << 24, 1366                                   # 2^24 x ceil(2^12 / 3) u32 = 91.7 GB, larger than L2 by far
        m = D.PackedMatrix(rows=rows, cols=cols, synthetic_seed=7)
        check(LIB.b200pir_dpir_set_stream(m._h, C.c_void_p(stream.cuda_stream)))
        rng = np.random.default_rng(11)
        hb = rng.integers(0, 1 << 32, 3 * cols, dtype=np.uint64).astype(np.uint32)
        b = torch.from_numpy(hb.view(np.int32)).cuda()
        out = torch.zeros(rows, dtype=torch.int32, device="cuda")
        ms = timed(lambda: check(LIB.b200pir_dpir_matvec_packed_dev(m._h, b.data_ptr(), out.data_ptr(), 0)))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"dpir_matvec": out})
        alg = 4 * rows * cols + 12 * cols + 4 * rows
        ho = np.zeros(rows, dtype=np.uint32)
        t1 = time.perf_counter()
        for _ in range(3):
            check(LIB.b200pir_dpir_matvec_packed(m._h, hb.ctypes.data, ho.ctypes.data))           # host b in, host out
        e2e_ms = (time.perf_counter() - t1) / 3 * 1e3
        # CPU port on a bounded row sample (2^18 rows = 1.4 GB), scaled
        import oracle_lib as O
        srows = 1 << 18
        a_s = rng.integers(0, 1 << 30, srows * cols, dtype=np.uint32)
        t1 = time.perf_counter()
        O.dpir_matvec_packed(a_s, hb, srows, cols)
        cpu_s = (time.perf_counter() - t1) * (rows / srows)
        line = {"metric": "DoublePIR matrix_mul_vec_packed HBM GB/s (2^24 x 1366 packed words)", "value": alg / ms / 1e6, "unit": "GB/s",
                "ms_per_step": ms, "dtype": "u32", "config": {"workload": "dpir: BASELINE configs[3], 2^24 rows x 1366 words (3 x 10 bit), 91.7 GB",
                                                               "l2": "inputs larger than L2"},
                "roofline": {"bound": "hbm", "kernel": "k_dpir_matvec_row", "achieved": alg / ms / 1e6, "peak": peak, "unit": "GB/s",
                             "frac": alg / ms / 1e6 / peak, "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg},
                "e2e": {"value": alg / e2e_ms / 1e6, "unit": "GB/s", "h2d_bytes_per_step": 12 * cols, "d2h_bytes_per_step": 4 * rows},
                "cpu_baseline": {"value": alg / cpu_s / 1e9, "unit": "GB/s", "cores": int(O.LIB.orc_num_threads()), "kind": "port",
                                 "sample": "oracle matrix_mul_vec_packed (OpenMP) on 2^18 of 2^24 rows, scaled x64"},
                "gpu_launches": args.steps}
        m.close()
    else:
        kw = WORKLOADS["T"]
        G = S.Params(**kw)
        G.set_stream(stream.cuda_stream)
        count = 1 << 16
        res = {}
        for poly_len, fn in ((2048, LIB.b200pir_ntt32_dev), (4096, LIB.b200pir_ntt4096_dev)):
            x = torch.randint(0, Q1, (count * 2 * poly_len,), dtype=torch.int32, device="cuda",
                              generator=torch.Generator(device="cuda").manual_seed(poly_len))
            for name, inv in (("forward", 0), ("inverse", 1)):
                if inv:
                    check(fn(G._h, x.data_ptr(), count, 0))               # inverse timed on canonical transform outputs
                ms = timed(lambda: check(fn(G._h, x.data_ptr(), count, inv)))
                if args.dump_outputs:                                     # the transforms run in place: x is the output
                    dump_outputs(args.dump_outputs, {"ntt%d_%s" % (poly_len, name): x})
                byt = 2 * count * 2 * poly_len * 4
                res["%d_%s" % (poly_len, name)] = {"ms": ms, "polys_per_s": count / ms * 1e3, "GB/s_u32": byt / ms / 1e6,
                                                   "frac_of_hbm_peak_u32": byt / ms / 1e6 / peak}
            del x
        f = res["2048_forward"]
        line = {"metric": "NTT throughput, 2^16 polynomials x 2 CRT moduli (28-bit), poly_len 2048 forward", "value": f["polys_per_s"],
                "unit": "polynomials/s", "ms_per_step": f["ms"], "dtype": "u32",
                "config": {"workload": "ntt: BASELINE configs[4], poly_len 2048 and 4096, forward and inverse",
                           "l2": "batch (1 GiB at 2048, 2 GiB at 4096) larger than L2"},
                "sweep": res,
                "roofline": {"bound": "hbm", "kernel": "k_ntt32 (relaxed-range butterflies)", "achieved": f["GB/s_u32"], "peak": peak, "unit": "GB/s",
                             "frac": f["frac_of_hbm_peak_u32"], "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": 2 * count * 2 * 2048 * 4,
                             "note": "the transform is bound by the integer-multiply pipe (scripts/ubench/bfly.cu: 915-1100 clocks per "
                                     "transform per SM), not by HBM"},
                "gpu_launches": 4 * args.steps}
        G.close()
    clocks = sampler.stop(t0, time.time())
    line.update({"n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "higher_is_better": True, "scaling": "weak",
                 "vs_baseline": None, "data": "synthetic", "clocks": clocks})
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default=None)
    ap.add_argument("--batch", type=int, default=None,
                    help="queries per step (whole job); must be a multiple of --gpus.  Default: --batch-per-gpu x GPUs")
    ap.add_argument("--batch-per-gpu", type=int, default=int(os.environ.get("B200PIR_BENCH_BATCH", "16")),
                    help="concurrent queries per GPU (BASELINE.json config #3: 128 concurrent queries on 8 GPUs)")
    ap.add_argument("--exchange", default=os.environ.get("B200PIR_BENCH_EXCHANGE", "ce"), choices=["ce", "nccl"],
                    help="N > 1: how the expanded queries reach the other ranks.  ce = pushed into the peers' gather buffers by the "
                         "copy engines over CUDA-IPC mappings (no SM-resident collective kernels competing with the compute kernels; "
                         "a 4-byte NCCL all-reduce per wave orders the ranks); nccl = ncclAllGather")
    ap.add_argument("--no-pipeline", dest="pipeline", action="store_false",
                    help="N > 1, copy-engine exchange: do not enqueue the expansion + pushes of step k + 1 before the first dimension "
                         "of step k")
    ap.add_argument("--timeline", action="store_true", help="N > 1: print a CUDA-event timeline of four steps to stderr")
    ap.add_argument("--waves", type=int, default=None,
                    help="N > 1: each rank's queries are processed in this many waves so that the all-gather of one wave's "
                         "expanded queries overlaps the expansion / first dimension of the other")
    ap.add_argument("--mul-variant", type=int, default=0)
    ap.add_argument("--db-format", type=int, default=int(os.environ.get("B200PIR_BENCH_DB_FORMAT", "-1")),
                    help="-1 = the library's choice (tcgen05 tile images wherever supported), 0 = IMAD layout, "
                         "1 = mma.sync fragment order, 2 = tcgen05 tile images")
    ap.add_argument("--fold-variant", type=int, default=2)
    ap.add_argument("--intt-variant", type=int, default=0)
    ap.add_argument("--imma-variant", type=int, default=0)
    ap.add_argument("--expand-variant", type=int, default=0)
    ap.add_argument("--queries-per-pass", type=int, default=None,
                    help="queries per database pass (1, 2, 4, 8 or 16).  Default: 16 on the tcgen05 path (the pass stays "
                         "HBM-bound), 8 on the mma.sync path (its 16-query pass is bound by the legacy tensor pipe)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the concurrent-queries sweep (Q = 1, 32, 128; N = 1 only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true",
                    help="N > 1: skip the correctness check of the NCCL flow (every rank recomputes its own queries of the last step "
                         "on an unsharded copy of the same database with the single-GPU path and compares the response bytes)")
    ap.add_argument("--steps-only", action="store_true",
                    help="profiling aid: skip the single-query latency probe and the e2e leg (clean ncu launch lists)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (for the Spiral workloads the response bytes of "
                         "every query of the step) as DIR/<name>.npy in float32 / float64; an output of more than 2^20 elements is "
                         "cut to a fixed, seeded sample")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        log("warning: WORLD_SIZE %d != --gpus %d" % (world, args.gpus))
    N = max(world, 1)
    if N > 1:
        # main + copy + one stream per peer + NCCL's: more streams than the default 8 hardware queues, and streams that share
        # a queue serialise behind each other's waits
        os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    if args.batch is None:
        args.batch = args.batch_per_gpu * N

    if args.workload in ("dpir", "ntt"):
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "kernel-level workloads carry their CPU baseline inside the GPU line"}))
            return
        if rank == 0:
            kernel_workload(args)
        return
    name = args.workload or "S8"
    kw = dict(WORKLOADS[name])
    import math
    base_name = {"S8": "S8: Spiral 2^20 x 1 KiB records (2^17 items x 8 KiB), 1 GiB plaintext = 8 GiB HBM-resident",
                 "S1": "S1: 1 GiB HBM-resident (2^14 items x 8 KiB)", "T": "T: unit-test size",
                 "S256": "S256: Spiral 2^25 x 1 KiB records (2^22 items x 8 KiB), 32 GiB plaintext = 256 GiB HBM-resident"}[name]
    if N > 1:
        if N & (N - 1):
            raise SystemExit("--gpus must be a power of two")
        if args.batch % N:
            raise SystemExit("--batch must be a multiple of --gpus")
        # the SAME database at every N, second-dimension rows sharded ii mod N (1/N of the bytes per GPU); the number of
        # concurrent queries grows with N (fixed per GPU), so per-GPU work is constant: weak scaling
        workload_name = "%s; rows sharded ii mod %d over %d GPUs" % (base_name, N, N)
    else:
        workload_name = base_name

    if args.impl == "reference":
        run_reference_arm(args, kw, workload_name, rank, world)
        return

    import numpy as np
    import torch
    import sdk_b200.spiral as S
    from sdk_b200._lib import LIB, check
    import ctypes as C

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if N > 1:
        import torch.distributed as dist
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))

    d = derived(kw)
    B = args.batch
    G = S.Params(device=local_rank, **kw)
    stream = torch.cuda.current_stream()
    G.set_stream(stream.cuda_stream)
    G.set_option("mul_variant", args.mul_variant)
    G.set_option("fold_variant", args.fold_variant)
    G.set_option("intt_variant", args.intt_variant)
    G.set_option("imma_variant", args.imma_variant)
    G.set_option("expand_variant", args.expand_variant)
    gdb = S.Database(G, shard_index=rank if N > 1 else 0, shard_count=N, fmt=None if args.db_format < 0 else args.db_format)
    args.db_format = gdb.info()["format"]
    if args.queries_per_pass is None:
        args.queries_per_pass = 16 if args.db_format == 2 else 8
    per_pass = min(args.queries_per_pass, 16 if B >= 16 else (8 if B >= 8 else (4 if B >= 4 else (2 if B >= 2 else 1))))
    G.set_option("batch", per_pass)
    gdb.fill_synthetic(0xB1755)
    rng = np.random.default_rng(20260923)
    pp = synthetic_pp(kw, rng)
    gpp = S.PublicParameters(G, pp["pack"], pp["left"], pp["right"], pp["conv"])
    modulus = Q0 * Q1
    rb = G.response_bytes
    q_words = (B // N) * 2 * POLY
    # pinned host buffers for the e2e leg
    h_q = torch.empty(q_words, dtype=torch.int64).pin_memory()
    h_q.numpy().view(np.uint64)[:] = rng.integers(0, modulus, q_words, dtype=np.uint64)
    h_out = torch.empty((B // N) * rb, dtype=torch.uint8).pin_memory()
    # wire-format queries (Query::serialize, client.rs:279-301: 32-byte seed || row 1 of ct) for the e2e leg
    qb = G.query_bytes
    h_qbytes = torch.empty((B // N) * qb, dtype=torch.uint8).pin_memory()
    qv = h_qbytes.numpy().reshape(B // N, qb)
    qv[:, :32] = rng.integers(0, 256, (B // N, 32), dtype=np.uint8)
    qv[:, 32:] = rng.integers(0, modulus, (B // N, (qb - 32) // 8), dtype=np.uint64).view(np.uint8).reshape(B // N, qb - 32)
    d_q = h_q.cuda(non_blocking=False)
    d_out = torch.zeros((B // N) * rb, dtype=torch.uint8, device="cuda")
    rows_local = d["num_per"] // N
    Bl = B // N                                      # queries this rank receives / answers per step
    W = 1
    if N > 1:
        if args.waves is None:
            args.waves = 1 if (args.exchange == "ce" and args.pipeline) else 2     # the pipeline already hides the transfer
        W = args.waves if (args.waves >= 1 and Bl % args.waves == 0) else 1
        Blw, Bw = Bl // W, (Bl // W) * N             # per wave: local queries, global queries
        fold_words = kw["nu_2"] * 2 * 2 * kw["t_gsw"] * 2 * POLY
        ct_words = 4 * POLY
        zi = lambda n: torch.zeros(n, dtype=torch.int32, device="cuda")
        d_qexp_l = [zi(Blw * d["dim0"] * POLY * 4) for _ in range(W)]
        d_vf_l = [zi(Blw * fold_words) for _ in range(W)]
        d_qexp = [zi(Bw * d["dim0"] * POLY * 4) for _ in range(W)]
        d_vf = [zi(Bw * fold_words) for _ in range(W)]
        d_partial = [zi(Bw * d["slices"] * ct_words) for _ in range(W)]
        d_gather = [zi(N * Bw * d["slices"] * ct_words) for _ in range(W)]
        coll_bytes = W * (N - 1) * (d_qexp_l[0].numel() + d_vf_l[0].numel() + d_partial[0].numel()) * 4
        # ---- copy-engine exchange: gather buffers allocated through the library (cudaMalloc + IPC handle), double-buffered across
        # steps, every peer's buffers mapped into this process
        exchange = args.exchange
        if exchange == "ce":
            try:
                # tcgen05 databases: the expanded queries travel as UMMA tile images (one image per rank and wave, re-tiled once by
                # the rank that expanded them); other layouts: uint4 [query][dim0][2048]
                use_images = args.db_format == 2 and Blw <= 16
                qexp_b = int(LIB.b200pir_query_image_bytes(G._h)) if use_images else Blw * d["dim0"] * POLY * 16
                vf_b = Blw * fold_words * 4                                               # bytes one rank contributes per wave
                mine, handles = {}, {}
                NBUF = 3
                for par in range(NBUF):
                    for w in range(W):
                        for kind, nbytes in (("q", N * qexp_b), ("v", N * vf_b)):
                            ptr, h = C.c_void_p(), C.create_string_buffer(64)
                            check(LIB.b200pir_peer_alloc(local_rank, nbytes, C.byref(ptr), h))
                            mine[(par, w, kind)] = ptr.value
                            handles[(par, w, kind)] = h.raw
                all_handles = [None] * N
                dist.all_gather_object(all_handles, handles)
                peer = {}
                for r in range(N):
                    if r == rank:
                        continue
                    for key, h in all_handles[r].items():
                        ptr = C.c_void_p()
                        check(LIB.b200pir_peer_open(local_rank, h, C.byref(ptr)))
                        peer[(r,) + key] = ptr.value
                copy_stream = torch.cuda.Stream()
                # one stream per peer: pushes to different peers run on different copy engines at the same time (a single stream
                # serialises them on one engine: 2.7 GB per step at N = 8 took ~14 ms, profiles/bench_r02_n8_single_copy_stream.json)
                peer_streams = {r: torch.cuda.Stream() for r in range(N) if r != rank}
                tiny = [torch.zeros(1, dtype=torch.int32, device="cuda") for _ in range(W)]
                # the "pushes landed" all-reduces get their own communicator: on the default one the survivors' all-gather of
                # step k would queue behind barrier(k + 1), i.e. behind the whole transfer of step k + 1 (measured: 4.3 ms of a
                # 12.8 ms step at N = 8, profiles/timeline_r02_n8.md)
                bar_group = dist.new_group(backend="nccl")
                prev_barrier = [None] * W
                barriers = {}
                step_no = [0]
            except Exception as e:
                log("peer-memory exchange unavailable (%r): falling back to ncclAllGather" % (e,))
                exchange = "nccl (peer setup failed: %s)" % (str(e)[:120],)

    # ---- N > 1, copy-engine exchange.  NBUF gather-buffer sets rotate over the steps.  Safety of a push into set (k % NBUF) at
    # the peers: they last read that set in step k - NBUF; barrier(k - 1) (a 4-byte all-reduce each rank issues after its
    # pushes of step k - 1) has completed before the push starts, hence every rank has issued its pushes of step k - 1, and
    # those are stream-ordered after that rank's first dimension of step k - 1 - (pipelined ? 1 : 0) >= k - NBUF.
    # (tests/test_exchange_protocol_sim.py replays this schedule with random timings: no hazard with three sets; two would also
    # do, but only thanks to the survivors' all-gather, which this argument does not rely on.)
    TL = []                                         # --timeline: (label, step, CUDA event) in stream order
    tl_on = [False]

    def mark(label, k, stream=None):
        if tl_on[0]:
            e = torch.cuda.Event(enable_timing=True)
            e.record(stream if stream is not None else torch.cuda.current_stream())
            TL.append((label, k, e))

    def ce_expand_push(k):
        bset = k % NBUF
        cur = torch.cuda.current_stream()
        for w in range(W):
            mark("expand.begin", k)
            # expand straight into this rank's slot of its own gather buffers, then push the slot to every peer
            q_own = mine[(bset, w, "q")] + rank * qexp_b
            v_own = mine[(bset, w, "v")] + rank * vf_b
            if use_images:
                check(LIB.b200pir_expand_queries_images_dev(G._h, gpp._h, d_q.data_ptr() + w * Blw * 2 * POLY * 8, Blw, q_own, v_own))
            else:
                check(LIB.b200pir_expand_queries_dev(G._h, gpp._h, d_q.data_ptr() + w * Blw * 2 * POLY * 8, Blw, q_own, v_own))
            mark("expand.end", k)
            ev = torch.cuda.Event()
            ev.record(cur)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev)
                if prev_barrier[w] is not None:
                    prev_barrier[w].wait()
                go = torch.cuda.Event()
                go.record(copy_stream)
                mark("push.begin", k, copy_stream)
                for r, ps in peer_streams.items():
                    ps.wait_event(go)
                    check(LIB.b200pir_peer_copy_async(peer[(r, bset, w, "q")] + rank * qexp_b, q_own, qexp_b, ps.cuda_stream))
                    check(LIB.b200pir_peer_copy_async(peer[(r, bset, w, "v")] + rank * vf_b, v_own, vf_b, ps.cuda_stream))
                    done = torch.cuda.Event()
                    done.record(ps)
                    copy_stream.wait_event(done)
                mark("push.end", k, copy_stream)
                # 4-byte all-reduce ordered after the pushes: complete when every rank's pushes have landed
                prev_barrier[w] = dist.all_reduce(tiny[w], group=bar_group, async_op=True)
            barriers[(k, w)] = prev_barrier[w]

    def ce_compute(k):
        bset = k % NBUF
        sv = []
        for w in range(W):
            barriers.pop((k, w)).wait()
            mark("first_dim.begin (all pushes landed)", k)
            if use_images:
                check(LIB.b200pir_first_dim_fold_images_dev(G._h, gdb._h, mine[(bset, w, "q")], N, Blw, mine[(bset, w, "v")],
                                                            d_partial[w].data_ptr()))
            else:
                check(LIB.b200pir_first_dim_fold_dev(G._h, gdb._h, mine[(bset, w, "q")], mine[(bset, w, "v")], Bw, d_partial[w].data_ptr()))
            mark("first_dim+local_fold.end", k)
            sv.append(dist.all_gather_into_tensor(d_gather[w], d_partial[w], async_op=True))
        for w in range(W):
            sv[w].wait()
            mark("survivors gathered", k)
            check(LIB.b200pir_finish_queries_dev(G._h, gpp._h, d_gather[w].data_ptr(), N, Bw, rank * Blw, Blw,
                                                 mine[(bset, w, "v")] + rank * vf_b, d_out.data_ptr() + w * Blw * rb))
            mark("finish.end", k)

    def step_dev():
        if N == 1:
            check(LIB.b200pir_process_query_batch_dev(G._h, gdb._h, gpp._h, d_q.data_ptr(), B, d_out.data_ptr()))
        elif exchange == "ce":
            # each rank expands the Bl queries it received and pushes them to every peer; every rank runs the first dimension +
            # local fold rounds of ALL B queries on its rows; survivors are all-gathered (NCCL, 32 KiB per query and slice); each
            # rank finishes its own Bl queries.  Pipelined: the expansion and the pushes of step k + 1 are enqueued BEFORE the
            # first dimension of step k, so the NVLink transfer (24 MiB per query to every peer) runs under step k's compute.
            k = step_no[0]
            step_no[0] += 1
            if args.pipeline:
                if k == 0:
                    ce_expand_push(0)
                ce_expand_push(k + 1)
                ce_compute(k)
            else:
                ce_expand_push(k)
                ce_compute(k)
        else:
            # NCCL all-gather of the expanded queries in W waves: the collectives are asynchronous (NCCL's stream), so wave w's
            # all-gather runs under wave w+1's expansion and wave w-1's first dimension
            ag = []
            for w in range(W):
                check(LIB.b200pir_expand_queries_dev(G._h, gpp._h, d_q.data_ptr() + w * Blw * 2 * POLY * 8, Blw,
                                                     d_qexp_l[w].data_ptr(), d_vf_l[w].data_ptr()))
                ag.append((dist.all_gather_into_tensor(d_qexp[w], d_qexp_l[w], async_op=True),
                           dist.all_gather_into_tensor(d_vf[w], d_vf_l[w], async_op=True)))
            sv = []
            for w in range(W):
                ag[w][0].wait()
                ag[w][1].wait()
                check(LIB.b200pir_first_dim_fold_dev(G._h, gdb._h, d_qexp[w].data_ptr(), d_vf[w].data_ptr(), Bw,
                                                     d_partial[w].data_ptr()))
                sv.append(dist.all_gather_into_tensor(d_gather[w], d_partial[w], async_op=True))
            for w in range(W):
                sv[w].wait()
                check(LIB.b200pir_finish_queries_dev(G._h, gpp._h, d_gather[w].data_ptr(), N, Bw, rank * Blw, Blw,
                                                     d_vf_l[w].data_ptr(), d_out.data_ptr() + w * Blw * rb))

    def step_e2e():
        if N == 1:
            n = C.c_size_t(0)
            check(LIB.b200pir_process_query_bytes(G._h, gdb._h, gpp._h, h_qbytes.data_ptr(), B * qb, B, h_out.data_ptr(),
                                                  C.byref(n)))
        else:
            d_q.copy_(h_q, non_blocking=True)
            step_dev()
            h_out.copy_(d_out, non_blocking=True)
            torch.cuda.current_stream().synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing
    for _ in range(args.warmup):
        step_dev()
    barrier()
    launches0 = LIB.b200pir_kernel_launches()
    sampler = ClockSampler(local_rank)
    if rank == 0:                    # rank 0 prints the line; N concurrent nvidia-smi processes only slow each other down
        sampler.start()
        sampler.wait_first()
    time.sleep(0.1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        step_dev()
    ev1.record()
    barrier()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1)
    launches = LIB.b200pir_kernel_launches() - launches0
    ms_total = ev0.elapsed_time(ev1)
    if args.dump_outputs:
        # the responses of the last timed step, rank by rank; taken now, before the passes below reuse d_out
        responses = d_out
        if dist is not None:
            responses = torch.empty(N * d_out.numel(), dtype=torch.uint8, device="cuda")
            dist.all_gather_into_tensor(responses, d_out)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"responses": responses.reshape(B, rb)})
        del responses
    if args.timeline and N > 1 and exchange == "ce":
        # where a step's time goes on this rank's streams (a separate, short pass; printed by every rank to stderr)
        tl_on[0] = True
        for _ in range(4):
            step_dev()
        barrier()
        tl_on[0] = False
        t_first = TL[0][2]
        lines = ["rank %d timeline (ms since the first mark; main stream unless push.*)" % rank]
        for label, k, e in TL:
            lines.append("  %9.3f  step %2d  %s" % (t_first.elapsed_time(e), k, label))
        log("\n".join(lines)) if rank in (0, N - 1) else None
    # per-stage / per-kernel times come from a SEPARATE pass of the same steps with per-stage CUDA events on
    # (the timed region above is un-instrumented)
    G.set_option("profile", 2)
    for _ in range(args.steps):
        step_dev()
    barrier()
    stage = G.last_stage_ms()
    G.set_option("profile", 0)
    if dist is not None:
        t = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    qps = B * 1e3 / ms_per_step

    # ---- single-query latency (device-resident, batch of 1), N == 1 only
    single_ms = None
    single_p99 = None
    single_roofline = None
    if N == 1 and not args.steps_only:
        for _ in range(3):
            check(LIB.b200pir_process_query_batch_dev(G._h, gdb._h, gpp._h, d_q.data_ptr(), 1, d_out.data_ptr()))
        torch.cuda.synchronize()
        G.set_option("profile", 2)
        # SURVEY 8d config #2: median of >= 100 single queries after warm-up, query already on the device
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(100)]
        for e0, e1 in evs:
            e0.record()
            check(LIB.b200pir_process_query_batch_dev(G._h, gdb._h, gpp._h, d_q.data_ptr(), 1, d_out.data_ptr()))
            e1.record()
        torch.cuda.synchronize()
        lat = sorted(e0.elapsed_time(e1) for e0, e1 in evs)
        single_ms = lat[len(lat) // 2]
        single_p99 = lat[98]
        st1 = G.last_stage_ms()
        G.set_option("profile", 0)
        k_ms = st1["multiply"] / max(st1["multiply_launches"], 1)
        db_b = d["slices"] * d["dim0"] * rows_local * POLY * 8
        op_b = (d["dim0"] * POLY * 16 if args.db_format == 0 else
                2 * POLY * ((d["dim0"] + 31) // 32) * 4096 if args.db_format == 2 else
                2 * POLY * ((d["dim0"] + 31) // 32) * 4 * 32 * 8)
        alg1 = db_b + op_b + d["slices"] * rows_local * 4 * POLY * 4
        pk, _src = measured_peak()
        single_roofline = {"queries_per_launch": 1, "kernel_ms": k_ms, "achieved": alg1 / (k_ms * 1e-3) / 1e9, "peak": pk,
                           "unit": "GB/s", "frac": alg1 / (k_ms * 1e-3) / 1e9 / pk, "algorithmic_bytes_per_launch": alg1}

    # ---- concurrent-queries sweep (SURVEY 8d config #2: Q in {1, 8, 32, 128} in flight), device-resident, N == 1 only
    sweep = None
    if N == 1 and not args.steps_only and not args.no_sweep:
        sweep = {}
        for Q in (8, 32, 128):
            dq = torch.from_numpy(rng.integers(0, modulus, Q * 2 * POLY, dtype=np.uint64).view(np.int64)).cuda()
            do = torch.zeros(Q * rb, dtype=torch.uint8, device="cuda")
            reps = max(2, min(args.steps, 256 // Q))
            for _ in range(2):
                check(LIB.b200pir_process_query_batch_dev(G._h, gdb._h, gpp._h, dq.data_ptr(), Q, do.data_ptr()))
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                check(LIB.b200pir_process_query_batch_dev(G._h, gdb._h, gpp._h, dq.data_ptr(), Q, do.data_ptr()))
            e1.record()
            torch.cuda.synchronize()
            sweep["Q%d" % Q] = {"queries_per_s": Q * reps * 1e3 / e0.elapsed_time(e1), "ms_per_batch": e0.elapsed_time(e1) / reps}
            del dq, do
        sweep["Q1"] = {"queries_per_s": 1e3 / single_ms, "ms_per_batch": single_ms}

    # ---- end to end (host buffers, copies inside the timed region)
    e2e_steps = 0 if args.steps_only else args.steps
    for _ in range(0 if args.steps_only else 2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    barrier()
    e2e_s = max(time.perf_counter() - t0, 1e-9)
    if dist is not None:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_qps = B * e2e_steps / e2e_s

    # ---- N > 1: correctness of the real multi-GPU run (the reference's model is chunked_end_to_end_test,
    # lib/doublepir/src/doublepir/doublepir.rs:607-716: partial results combined, outcome compared).  Every rank holds the
    # responses to ITS queries from the last step (d_out); it recomputes them on an UNSHARDED copy of the same synthetic
    # database with the single-GPU path (itself checked against the oracle by tests/) and the bytes must be identical.
    verified = None
    full_db_bytes = d["slices"] * d["dim0"] * d["num_per"] * POLY * 8
    verify_note = None
    if N > 1 and not args.no_verify and full_db_bytes > 96 * 2**30:
        verify_note = "skipped: the unsharded database (%.0f GiB) does not fit one GPU beside the shard" % (full_db_bytes / 2**30)
    elif N > 1 and not args.no_verify:
        step_dev()
        torch.cuda.synchronize()
        full = S.Database(G, shard_index=0, shard_count=1, fmt=args.db_format)
        full.fill_synthetic(0xB1755)
        d_ref = torch.zeros(Bl * rb, dtype=torch.uint8, device="cuda")
        check(LIB.b200pir_process_query_batch_dev(G._h, full._h, gpp._h, d_q.data_ptr(), Bl, d_ref.data_ptr()))
        torch.cuda.synchronize()
        ok = torch.tensor([1 if torch.equal(d_ref, d_out) else 0], device="cuda", dtype=torch.int32)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        verified = bool(ok.item())
        full.close()
        del d_ref

    # ---- roofline of the dominant kernel (multiply_reg_by_database)
    mul_launches = max(int(stage["multiply_launches"]), 1)
    mul_ms = stage["multiply"] / mul_launches
    nq_per_launch = B * args.steps / mul_launches
    db_bytes = d["slices"] * d["dim0"] * rows_local * POLY * 8
    if args.db_format == 0:
        operand_bytes = nq_per_launch * d["dim0"] * POLY * 16
    elif args.db_format == 2:   # tcgen05 tile images of the query operand: [n][z][dim0/32][4096 B], 16 queries
        operand_bytes = 2 * POLY * ((d["dim0"] + 31) // 32) * 4096
    else:   # limb fragments of the query operand: [n][z][column tiles][dim0/32][4 limbs][32 lanes] x 8 B
        tiles = 4 if nq_per_launch > 8 else (2 if nq_per_launch > 4 else 1)
        operand_bytes = 2 * POLY * tiles * ((d["dim0"] + 31) // 32) * 4 * 32 * 8
    alg_bytes = db_bytes + operand_bytes + nq_per_launch * d["slices"] * rows_local * 4 * POLY * 4
    peak, peak_src = measured_peak()
    achieved = alg_bytes / (mul_ms * 1e-3) / 1e9
    kname = {0: "k_multiply (IMAD)", 1: "k_multiply_imma (INT8 MMA limbs)", 2: "k_multiply_tc5 (tcgen05 kind::i8 limbs)"}[args.db_format]
    roofline = {"bound": "hbm", "kernel": kname + " = multiply_reg_by_database, server.rs:155-221",
                "queries_per_launch": nq_per_launch,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": ncu_traffic(name, B, args.db_format), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": mul_ms,
                "frac_of_nominal_8_tb_s": achieved / 8000.0,      # north_star quotes "~8 TB/s"; `frac` uses the measured copy peak
                "kernel_share_of_step": stage["multiply"] / max(stage["total"], 1e-9),
                "note": "kernel_ms = CUDA-event time of the multiply kernel alone; the re-tiling of the query operand that precedes it "
                        "is stage 'query_image'"}

    if rank == 0:
        cpu = None
        if N == 1 and not args.no_cpu_baseline:
            try:
                full = CpuFullQuery(kw)
                times = [full.one() for _ in range(3)]
                sec = sorted(times)[1]                                   # median of three full queries
                cpu = {"value": 1.0 / sec, "unit": "queries/s", "cores": full.cores, "kind": "port",
                       "sample": full.sample(3) + "; median", "full_query_s": times}
                threads = full.cores
                del full
                est, _cores, sample = cpu_process_query_sample(kw, threads=threads)
                cpu["extrapolated_value"] = 1.0 / est
                cpu["extrapolated_sample"] = sample
                if single_ms:
                    # like for like: one query at a time on both sides (the reference has no batching)
                    cpu["gpu_single_query_vs_cpu"] = (1e3 / single_ms) / cpu["value"]
            except Exception as e:      # the oracle is only a reported baseline; never fail the bench on it
                cpu = {"value": None, "unit": "queries/s", "cores": None, "kind": "port", "sample": "failed: %r" % (e,)}
        out = {
            "metric": "PIR server queries/sec (Spiral process_query)", "value": qps, "unit": "queries/s",
            "n_gpus": N, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload_name, "params": kw, "batch": B, "batch_per_gpu": B // N, "waves": W, "queries_per_pass": per_pass,
                       "exchange": (exchange if N > 1 else None), "pipelined": bool(N > 1 and exchange == "ce" and args.pipeline),
                       "exchange_format": ("UMMA tile images" if (N > 1 and exchange == "ce" and use_images) else "uint4 [query][dim0][2048]") if N > 1 else None,
                       "db_bytes_per_gpu": db_bytes,
                       "plaintext_bytes": d["slices"] * d["dim0"] * d["num_per"] * POLY,
                       "first_dimension_kernel": kname,
                       "parallelism": ("rows ii mod %d, %d concurrent queries per GPU; queries expanded by the receiving rank; expanded "
                                       "queries exchanged by %s, surviving ciphertexts by asynchronous NCCL all-gather, in %d "
                                       "waves (%d bytes received per rank per step)"
                                       % (N, B // N, "copy-engine pushes into peer memory (CUDA IPC over NVLink)" if exchange == "ce"
                                          else "asynchronous NCCL all-gather", W, coll_bytes))
                       if N > 1 else "single GPU",
                       "l2": "inputs larger than L2 (database %.1f GiB per GPU streamed every step)" % (db_bytes / 2**30)},
            "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": (B * qb) if N == 1 else B * 2 * POLY * 8,
                    "d2h_bytes_per_step": B * rb,
                    "call": "b200pir_process_query_bytes (Query::deserialize + process_query, wire-format queries)" if N == 1
                            else "three-phase device entry points around NCCL all-gathers, query ciphertexts copied from pinned host memory"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "stage_ms_per_step": {k: v / args.steps for k, v in stage.items() if k not in ("multiply_launches",)},
            "single_query_latency_ms": single_ms, "single_query_latency_p99_ms": single_p99,
            "single_query_latency_note": "median / 99th percentile of 100 device-resident single queries after warm-up",
            "single_query_roofline": single_roofline,
            "concurrent_queries_sweep": sweep,
            "verified": verified, "verify_note": verify_note,
            "timed_region": "un-instrumented; stage_ms_per_step and roofline.kernel_ms come from a separate pass of the same steps "
                            "with per-stage CUDA events",
        }
        if cpu is not None:
            out["cpu_baseline"] = cpu
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
