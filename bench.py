#!/usr/bin/env python
"""bench.py — Stark::prove() wall-clock at padded height 2^20 on B200 (BASELINE.json metric).

One "step" = one complete prove() of a synthetic instance (uniform random main / aux traces and
randomizers of the real shape: 379 main columns, 91 aux columns, trace length 2^20, LDT domain 2^23,
security 160, expansion 4, FRI) through the public C ABI call `tvm_prove` with HOST buffers
(pinned), i.e. host->device copies of the traces are inside the timed region (`e2e`).
`value` is the same call with the traces already resident in HBM (device pointers; the library
accepts both kinds), timed the same way over its own K steps.  Trace generation (VM, table fill/extend) is outside the
hot path (SURVEY.md §8) and outside the timed region: the aux-trace callback only hands back a
pointer to pre-generated pinned memory.

`--impl reference` times the CPU restatement of the same path (oracle/, C + OpenMP on all host
cores) on a bounded sample and extrapolates to the full prove — the Rust reference cannot be built
in this image (no cargo), see DESIGN.md.

N > 1 (torchrun): ONE proof sharded over the N GPUs by evaluation-domain cosets (SURVEY.md 8(e)):
columns are uploaded/interpolated column-sharded, every rank extends, hashes and evaluates the AIR on
its N-th of the rows; NCCL all-gathers move interpolant coefficients, leaf digests, the quotient and
the DEEP codeword.  Strong scaling: value = wall time of that one proof (max over ranks).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "triton-vm_b200", "py"))

import numpy as np  # noqa: E402

P = (1 << 64) - (1 << 32) + 1
NM, NA = 379, 91


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


def measured_lde_traffic(alg_bytes):
    """DRAM bytes (read + write) of the LDE kernels from the committed ncu capture, scaled to this workload:
    profiles/r02h_ntt_traffic.json holds dram bytes per algorithmic byte of the tile-NTT passes of a column LDE at 2^20."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02h_ntt_traffic.json")))
        return float(t["dram_bytes_per_algorithmic_byte"]) * alg_bytes, t.get("source")
    except Exception:
        return None, None


def algorithmic_lde_bytes(n, ncols):
    # SURVEY.md §8(d): column LDE reads 8 B per trace element and writes 64 B (8x blow-up): 72 B per trace element
    return 72 * n * ncols


def dump_outputs(out_dir, proof):
    """--dump-outputs: the proof words of the last timed step as DIR/proof.npy, float64 [words, 2] holding the low and the high
    32 bits of each word (exact in float64; word = low + high * 2^32).  A proof stays below 10^6 words (16 MB as written) at
    every padded height the library accepts, so it is written whole."""
    os.makedirs(out_dir, exist_ok=True)
    w = np.asarray(proof, dtype=np.uint64)
    np.save(os.path.join(out_dir, "proof.npy"), np.stack([w & np.uint64(0xFFFFFFFF), w >> np.uint64(32)], axis=1).astype(np.float64))


# ---- CPU baseline (oracle port) --------------------------------------------------------------------
def workload_string(log2_height, ldt_name, forced, num_rand):
    return (f"Stark::prove (Stark::default(): security 160, expansion 4, low-degree test {ldt_name}"
            f"{' (forced)' if forced else ' as the reference selects at this height'}) at padded height "
            f"2^{log2_height}: 379 main + 91 aux columns, {num_rand} trace randomizers, "
            f"trace domain 2^{log2_height}, LDT domain 2^{log2_height + 3}")


def _oracle_threads():
    """one OpenMP thread per physical core: on the hyper-threaded hosts of this pool 2 threads per core made the memory-bound
    NTTs 5x slower, which would flatter the GPU arm; also undoes torchrun's OMP_NUM_THREADS=1 at N > 1"""
    from oracle import corc
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or 0
    except Exception:
        phys = 0
    if phys and phys != corc.num_threads():
        corc.set_num_threads(phys)
    return corc.num_threads()


class OracleInstance:
    """synthetic instance of the GPU arm's shape at a given padded height, for oracle/fast.py (complete CPU proves)"""
    def __init__(self, log2_height, ldt):
        from oracle import stark as S
        self.S = S
        self.stark = S.Stark(160, 2, None if ldt == "auto" else ldt)
        self.log2_height = log2_height
        d = self.d = self.stark.derive(1 << log2_height)
        n, h = d["trace_len"], d["num_trace_randomizers"]
        rng = np.random.default_rng(0x5452_4954 + log2_height)
        r = lambda *shape: rng.integers(0, P, size=shape, dtype=np.uint64)
        self.main, self.mrand, self.aux, self.arand = r(NM, n), r(NM, h), r(NA, n, 3), r(NA, h, 3)
        self.qrand = r(d["num_quotient_randomizer_coefficients"], 3)
        self.claim = S.Claim([1, 2, 3, 4, 5], [7, 8, 9], [10])

    def prove(self):
        """one COMPLETE prove (all stages, proof words out) -> (seconds, per-stage seconds)"""
        from oracle import fast
        tm = {}
        t0 = time.perf_counter()
        proof = fast.prove(self.stark, self.claim, self.main, self.mrand, lambda ch: (self.aux, self.arand), self.qrand,
                           padded_height=1 << self.log2_height, timings=tm)
        dt = time.perf_counter() - t0
        self.proof = proof
        return dt, tm


def nlogn_scale(log2_from, log2_to):
    """work model of the prove: n log2(LDT domain) (NTTs dominate the CPU path; hashing and the AIR are linear in n)"""
    return (2.0 ** (log2_to - log2_from)) * (log2_to + 3) / (log2_from + 3)


def cpu_baseline(log2_height, ldt="auto", budget_s=30.0):
    """Complete CPU proves (oracle/fast.py: C + OpenMP, every stage, same low-degree test as the GPU arm) at the largest
    padded height whose prove fits the time budget; the figure for 2^log2_height is that MEASUREMENT scaled by the
    n log n work model and labelled as such.  Returns (ms, cores, sample text, per-stage ms, details)."""
    cores = _oracle_threads()
    calib = OracleInstance(12, ldt)
    calib.prove()                                     # warms the OpenMP pool and the AIR build
    t12, _ = calib.prove()
    # the low-degree test must be the one the GPU arm runs: Stark::default() switches to STIR at 2^16
    sample_log2 = 16
    if t12 * nlogn_scale(12, 16) * 2.2 > budget_s:
        sample_log2 = 14 if ldt == "fri" else 16      # never below 2^16 with the automatic choice (FRI there != STIR here)
    inst = OracleInstance(min(sample_log2, log2_height), ldt)
    times, stage_acc = [], {}
    reps = 2 if t12 * nlogn_scale(12, inst.log2_height) * 2.2 <= budget_s else 1
    for _ in range(reps):
        dt, tm = inst.prove()
        times.append(dt)
        for k, v in tm.items():
            stage_acc.setdefault(k, []).append(v)
    t_meas = float(np.median(times))
    scale = nlogn_scale(inst.log2_height, log2_height) if inst.log2_height != log2_height else 1.0
    stages = {k: float(np.median(v)) * scale * 1e3 for k, v in stage_acc.items()}
    sample = (f"{reps} complete prove(s) of the C+OpenMP restatement (oracle/fast.py, every stage, low-degree test "
              f"{inst.d['ldt'].upper()}) at padded height 2^{inst.log2_height}: median {t_meas:.2f} s on {cores} threads; value = that "
              f"measurement x {scale:.1f} (n log n work model) for 2^{log2_height} - extrapolated, see --impl reference for the "
              f"measured 2^16 -> 2^18 ratio")
    details = {"measured_log2_height": inst.log2_height, "measured_ms": t_meas * 1e3, "scale_to_target": scale,
               "ldt": inst.d["ldt"], "extrapolated": inst.log2_height != log2_height}
    return t_meas * scale * 1e3, cores, sample, stages, details


# ---- clocks ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(device_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ---- GPU arm -------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import tvm_b200
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        import torch.distributed as dist
        # rank 0 prints ONE JSON line on stdout: anything libraries print meanwhile (NCCL's version banner) is sent to
        # stderr by pointing fd 1 at fd 2 until the result is ready
        sys.stdout.flush()
        saved_stdout_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    torch.cuda.set_device(local_rank)
    ldt_choice = {"auto": tvm_b200.LDT_AUTO, "fri": tvm_b200.LDT_FRI, "stir": tvm_b200.LDT_STIR}[args.ldt]
    dom = tvm_b200.derive_domains(160, 2, 1 << args.log2_height, ldt_choice)
    ldt_name = {tvm_b200.LDT_FRI: "FRI", tvm_b200.LDT_STIR: "STIR"}[dom["ldt"]]
    n, h = dom["trace_len"], dom["num_trace_randomizers"]
    nqr = dom["num_quotient_randomizer_coefficients"]

    def pinned(shape):
        t = torch.empty(shape, dtype=torch.int64, pin_memory=True)
        return t, t.numpy().view(np.uint64)

    rng = np.random.default_rng(0x5452_4954)   # identical inputs on every rank (one sharded proof)
    keep = []

    def fill(shape):
        t, a = pinned(shape)
        flat = a.reshape(-1)
        step = 1 << 24
        for s in range(0, flat.size, step):
            flat[s:s + step] = rng.integers(0, P, size=min(step, flat.size - s), dtype=np.uint64)
        keep.append(t)
        return a

    main_trace, main_rand = fill((NM, n)), fill((NM, h))
    aux_trace, aux_rand = fill((NA, n, 3)), fill((NA, h, 3))
    quot_rand = fill((nqr, 3))
    claim = ([1, 2, 3, 4, 5], [7, 8, 9], [10])
    b = tvm_b200.Backend(local_rank)
    if args.low_memory is not None:
        b.set_low_memory(args.low_memory)
    comm = None
    if world > 1:
        from tvm_b200.dist import TorchDistComm
        comm = TorchDistComm(f"cuda:{local_rank}")
        b.set_comm(comm)

    def aux_provider(_challenges):
        return aux_trace, aux_rand          # pre-generated: tracegen is outside the hot path

    # device-resident copies of the same inputs for the `value` leg
    dev = torch.device(f"cuda:{local_rank}")
    d_main_trace, d_main_rand = keep[0].to(dev), keep[1].to(dev)
    d_aux_trace, d_aux_rand = keep[2].to(dev), keep[3].to(dev)

    def step_host():
        return b.prove(claim, main_trace, main_rand, aux_provider, quot_rand, 160, 2, 1 << args.log2_height, ldt_choice)

    def step_dev():
        return b.prove(claim, d_main_trace, d_main_rand, lambda _c: (d_aux_trace, d_aux_rand), quot_rand, 160, 2,
                       1 << args.log2_height, ldt_choice)

    def timed(step):
        """W warm-up steps, then exactly K timed steps: barrier + synchronize on both sides, max over ranks."""
        for _ in range(args.warmup):
            proof = step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        launches0 = b.launches
        stage_acc = {}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            proof = step()
            for name, ms in b.last_prove_timings():
                stage_acc[name] = stage_acc.get(name, 0.0) + ms
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1e3
        if world > 1:
            t = torch.tensor([wall_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            wall_ms = float(t.item())
            dist.barrier()
        return wall_ms / args.steps, {k: v / args.steps for k, v in stage_acc.items()}, b.launches - launches0, proof

    sampler = ClockSampler(local_rank) if rank == 0 else None
    try:
        e2e_ms, e2e_stages, _, proof = timed(step_host)
        device_ms, stages, launches, proof_dev = timed(step_dev)
    finally:                                    # never leave the nvidia-smi sampler running
        clocks = sampler.stop() if sampler else None
    assert np.array_equal(proof, proof_dev), "host-input and device-input proofs differ"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, proof_dev)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
        sys.stdout.flush()
        import ctypes
        ctypes.CDLL(None).fflush(None)          # NCCL prints through C stdio: drain its buffer while fd 1 still is stderr
        os.dup2(saved_stdout_fd, 1)
        os.close(saved_stdout_fd)
    if rank != 0:
        return
    lde_ms = stages.get("upload+LDE(main)", 0.0) + stages.get("upload+LDE(aux)", 0.0)
    peaks = measured_peaks()
    peak = (peaks["hbm_gbs"] if peaks else 6650.0) * world   # aggregate over the GPUs sharing the proof
    alg = algorithmic_lde_bytes(n, NM + 3 * NA)
    achieved = alg / (lde_ms * 1e-3) / 1e9 if lde_ms else 0.0
    traffic, traffic_src = measured_lde_traffic(alg)
    out = {
        "metric": "prove() ms @ padded height 2^%d; NTT GF(p) elems/s vs HBM roofline" % args.log2_height,
        "value": device_ms, "unit": "ms", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": device_ms, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
        "dtype": "u64",
        "data": "synthetic",
        "config": {"workload": workload_string(args.log2_height, ldt_name, args.ldt != "auto", dom['num_trace_randomizers']),
                   "parallelism": "single GPU" if world == 1 else
                   f"one proof sharded over {world} GPUs by evaluation-domain cosets (NCCL all-gathers: "
                   f"{comm.calls['all_gather'] // max(1, 2 * (args.steps + args.warmup))} per proof)",
                   "l2": "inputs (GBs) larger than L2",
                   "lde_tables": "just-in-time (low-memory mode)" if b.last_prove_low_memory else "cached in HBM",
                   "value_leg": "traces resident in HBM (device pointers through tvm_prove)",
                   "e2e_leg": "traces in pinned host memory, uploads overlapped with the LDE inside tvm_prove"},
        "e2e": {"value": e2e_ms, "unit": "ms",
                "h2d_bytes_per_step": int(main_trace.nbytes + main_rand.nbytes + aux_trace.nbytes + aux_rand.nbytes + quot_rand.nbytes),
                "d2h_bytes_per_step": int(proof.nbytes)},
        "gpu_launches": int(launches),
        "stages_ms": {k: round(v, 3) for k, v in stages.items()},
        "e2e_stages_ms": {k: round(v, 3) for k, v in e2e_stages.items()},
        "roofline": {"bound": "hbm", "kernel": "coset LDE (ntt_tile_kernel: interpolation + 8-coset evaluation passes) of the 652 table columns",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650",
                     "algorithmic_bytes": alg,
                     "ntt_gelems_per_s": (NM + 3 * NA) * 8 * n / (lde_ms * 1e-3) / 1e9 if lde_ms else None},
        "clocks": clocks,
    }
    # After the timed region: the proof the GPU just produced goes through Stark::verify (tvm_verify, host code).  The tables
    # are synthetic, so only the out-of-domain AIR identity is skipped; transcript, Merkle openings, DEEP and the low-degree
    # test are checked in full.  Informational: a rejection is reported, it does not abort the bench line.
    try:
        t0 = time.perf_counter()
        accepted, reason = tvm_b200.verify(claim, proof, 160, 2, ldt_choice=ldt_choice, skip_air_check=True)
        out["proof_check"] = {"verifier": "tvm_verify (Stark::verify; AIR identity skipped: synthetic tables)", "accepted": bool(accepted),
                              "reason": reason, "ms": round(1e3 * (time.perf_counter() - t0), 1), "proof_words": int(proof.size)}
    except Exception as e:  # noqa: BLE001 - never lose the measurement over the post-check
        out["proof_check"] = {"accepted": None, "reason": "verifier call failed: " + repr(e)[:200]}
    if world == 1 and not args.no_cpu_baseline:
        total, cores, sample, cstages, details = cpu_baseline(args.log2_height, args.ldt)
        out["cpu_baseline"] = {"value": total, "unit": "ms", "cores": cores, "kind": "port", "sample": sample,
                               "stages_ms": {k: round(v, 1) for k, v in cstages.items()}, **details}
    print(json.dumps(out))


def run_gpu_workload(args):
    """The reference's own benchmark workload (ProgramToBench::spin / prove_fib: triton-dev-util/src/lib.rs:49-75,
    benches/prove_fib.rs:8-28) from files written by tools/make_workload.py — trace generation is outside the hot path and
    outside the timed region.  One step = tvm_prove_tables: upload of the 149 table columns + randomness, degree-lowering
    columns, LDE, commitments, MasterMainTable::extend on the device, quotient, DEEP, low-degree test, openings.  After the
    timed region the proof goes through tvm_verify INCLUDING the AIR identity."""
    import torch
    import tvm_b200
    d = args.workload_dir
    txt = open(os.path.join(d, "claim.txt")).read().split()
    security, log2_exp, ldtc, padded_height = (int(v) for v in txt[:4])
    digest = [int(v) for v in txt[4:9]]
    ni = int(txt[9]); inp = [int(v) for v in txt[10:10 + ni]]
    no = int(txt[10 + ni]); outp = [int(v) for v in txt[11 + ni:11 + ni + no]]
    claim = (digest, inp, outp)
    dom = tvm_b200.derive_domains(security, log2_exp, padded_height, ldtc)
    n, h, nqr = dom["trace_len"], dom["num_trace_randomizers"], dom["num_quotient_randomizer_coefficients"]
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")

    def load(name, shape):
        a = np.fromfile(os.path.join(d, name + ".u64"), dtype="<u8").reshape(shape)
        t = torch.empty(shape, dtype=torch.int64, pin_memory=True)
        t.numpy().view(np.uint64)[...] = a
        return t
    main_t = load("main", (NM, n)); main_rand = load("main_rand", (NM, h)); aux_rand = load("aux_rand", (NA, h, 3))
    col90 = load("col90", (n, 3)); quot_rand = load("quot_rand", (nqr, 3)).numpy().view(np.uint64)
    b = tvm_b200.Backend(0)
    if args.low_memory is not None:
        b.set_low_memory(args.low_memory)
    dv = [t.to(dev) for t in (main_t, main_rand, aux_rand, col90)]

    aet_host = aet_dev = None
    if args.from_aet:                              # tvm_prove_aet: the witness itself crosses the boundary, no table on the host
        import glob
        aet_host, aet_dev = {}, {}
        for f in sorted(glob.glob(os.path.join(d, "aet_*.u*"))):
            name, ext = os.path.basename(f)[4:].rsplit(".", 1)
            a = np.fromfile(f, dtype="<u4" if ext == "u32" else "<u8")
            if name in ("program", "instruction_multiplicities", "lookup_table_lookup_multiplicities"):
                aet_host[name] = aet_dev[name] = a                   # small; the multiplicities are widened on the host
                continue
            width = tvm_b200._AET_WIDTHS[name]
            t = torch.empty((a.size // width, width), dtype=torch.int64, pin_memory=True)
            t.numpy().view(np.uint64)[...] = a.reshape(-1, width)
            aet_host[name], aet_dev[name] = t, t.to(dev)
        assert len(aet_host) == 11, "no AET in the workload directory: tools/make_workload.py --aet"

    def step(tabs):
        if args.from_aet:
            return b.prove_aet(claim, aet_host if tabs[0] is main_t else aet_dev, tabs[1], tabs[2], tabs[3], quot_rand, security, log2_exp,
                               padded_height, ldtc)
        return b.prove_tables(claim, tabs[0], tabs[1], tabs[2], tabs[3], quot_rand, security, log2_exp, padded_height, ldtc)

    def timed(tabs):
        for _ in range(args.warmup):
            proof = step(tabs)
        torch.cuda.synchronize()
        l0, acc = b.launches, {}
        t0 = time.perf_counter()
        for _ in range(args.steps):
            proof = step(tabs)
            for name, ms in b.last_prove_timings():
                acc[name] = acc.get(name, 0.0) + ms
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / args.steps, {k: round(v / args.steps, 3) for k, v in acc.items()}, b.launches - l0, proof

    sampler = ClockSampler(0)
    try:
        e2e_ms, e2e_stages, _, proof = timed((main_t, main_rand, aux_rand, col90))
        dev_ms, stages, launches, proof_dev = timed(dv)
    finally:
        clocks = sampler.stop()
    assert np.array_equal(proof, proof_dev)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, proof_dev)
    t0 = time.perf_counter()
    accepted, reason = tvm_b200.verify(claim, proof, security, log2_exp, ldt_choice=ldtc, skip_air_check=False)
    verify_ms = (time.perf_counter() - t0) * 1e3
    log2h = padded_height.bit_length() - 1
    ldt_name = {tvm_b200.LDT_FRI: "FRI", tvm_b200.LDT_STIR: "STIR"}[dom["ldt"]]
    print(json.dumps({
        "metric": "prove() ms @ padded height 2^%d; NTT GF(p) elems/s vs HBM roofline" % log2h,
        "value": dev_ms, "unit": "ms", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms,
        "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "u64",
        "data": "real execution trace of the reference's benchmark program (tables from tools/make_workload.py, outside the timed region)",
        "config": {"workload": f"{os.path.basename(os.path.normpath(d))}: " + workload_string(log2h, ldt_name, ldtc != 0, h),
                   "entry_point": ("tvm_prove_aet: the AlgebraicExecutionTrace in; MasterMainTable::new + pad, degree-lowering columns + "
                                   "MasterMainTable::extend on the device" if args.from_aet else
                                   "tvm_prove_tables: 149 table columns in, degree-lowering columns + MasterMainTable::extend on the device"),
                   "parallelism": "single GPU", "lde_tables": "just-in-time (low-memory mode)" if b.last_prove_low_memory else "cached in HBM"},
        "e2e": {"value": e2e_ms, "unit": "ms",
                "h2d_bytes_per_step": int(8 * ((sum(int(np.prod(v.shape)) for v in aet_host.values()) if args.from_aet else 149 * n)
                                               + NM * h + NA * h * 3 + n * 3 + nqr * 3)), "d2h_bytes_per_step": int(proof.nbytes)},
        "gpu_launches": int(launches), "stages_ms": stages, "e2e_stages_ms": e2e_stages, "clocks": clocks,
        "proof_check": {"verifier": "tvm_verify (Stark::verify) INCLUDING the out-of-domain AIR identity", "accepted": bool(accepted),
                        "reason": reason, "ms": round(verify_ms, 1), "proof_words": int(proof.size)},
    }))


def run_reference(args):
    """The reference arm: the CPU restatement of the path (oracle/: C + OpenMP; the Rust reference cannot be built in this
    image) on all host cores.  One step = one COMPLETE prove (every stage, same low-degree test as the GPU arm) at the
    largest padded height that keeps the whole run within a few minutes; one more complete prove two doublings higher
    gives the measured scaling ratio with which the figure for the GPU arm's height is extrapolated (and labelled)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = _oracle_threads()
    target = args.log2_height
    calib = OracleInstance(12, args.ldt)
    calib.prove()                                                   # OpenMP pool + AIR build warm
    t12, _ = calib.prove()
    budget = 200.0                                                  # seconds for the K + W steps: bounds the sample height
    sample_log2 = min(16, target)
    est = t12 * nlogn_scale(12, sample_log2) * 1.3
    if est * (args.steps + args.warmup) > budget and args.ldt == "fri" and sample_log2 > 14:
        sample_log2 = 14                                            # with the automatic choice 2^16 is the smallest STIR height
    inst = OracleInstance(sample_log2, args.ldt)
    steps = args.steps
    for _ in range(args.warmup):
        inst.prove()
    times, stage_acc = [], {}
    t0 = time.perf_counter()
    for _ in range(steps):
        dt, tm = inst.prove()
        times.append(dt)
        for k, v in tm.items():
            stage_acc.setdefault(k, []).append(v)
    per_step = (time.perf_counter() - t0) * 1e3 / steps
    t_s = float(np.median(times))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, inst.proof)
    # scaling cross-check: one complete prove two doublings up (if it fits ~2 minutes and the target is higher still)
    ratio, t_hi, hi_log2 = None, None, None
    if target >= sample_log2 + 2 and t_s * nlogn_scale(sample_log2, sample_log2 + 2) < 150.0:
        hi_log2 = sample_log2 + 2
        hi = OracleInstance(hi_log2, args.ldt)
        t_hi, tm_hi = hi.prove()
        ratio = t_hi / t_s
    base_log2, base_t = (hi_log2, t_hi) if t_hi is not None else (sample_log2, t_s)
    if target == base_log2:
        value, how = base_t * 1e3, "measured"
    elif ratio is not None and (target - base_log2) % 2 == 0:
        value = base_t * 1e3 * ratio ** ((target - base_log2) // 2)
        how = (f"extrapolated: measured complete prove at 2^{base_log2} ({base_t:.2f} s) x the measured 2^{sample_log2} -> 2^{hi_log2} "
               f"ratio {ratio:.2f} per two doublings (n log n model: {nlogn_scale(sample_log2, hi_log2):.2f})")
    else:
        value = base_t * 1e3 * nlogn_scale(base_log2, target)
        how = f"extrapolated: measured complete prove at 2^{base_log2} ({base_t:.2f} s) x n log n work model"
    dom_name = inst.d["ldt"].upper()
    from oracle import stark as S
    dt_ = S.Stark(160, 2, None if args.ldt == "auto" else args.ldt).derive(1 << target)
    sample = (f"step = one complete prove at padded height 2^{sample_log2} ({dom_name}); median of {steps} steps {t_s:.2f} s on {cores} "
              f"threads" + (f"; one complete prove at 2^{hi_log2}: {t_hi:.2f} s" if t_hi is not None else "") + f"; value for 2^{target} {how}")
    print(json.dumps({
        "impl": "reference", "metric": "prove() ms @ padded height 2^%d; NTT GF(p) elems/s vs HBM roofline" % target,
        "value": value, "unit": "ms", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": per_step,
        "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_string(target, dt_["ldt"].upper(), args.ldt != "auto", dt_["num_trace_randomizers"]),
                   "implementation": "CPU restatement of the reference path (oracle/fast.py + oracle/c: C + OpenMP over the axes rayon uses); "
                                     "the Rust reference cannot be built in this image (no cargo)",
                   "sample": sample},
        "measured": {f"2^{sample_log2}": {"median_ms": t_s * 1e3, "all_ms": [round(t * 1e3, 1) for t in times],
                                          "stages_ms": {k: round(float(np.median(v)) * 1e3, 1) for k, v in stage_acc.items()}},
                     **({f"2^{hi_log2}": {"ms": t_hi * 1e3, "stages_ms": {k: round(v * 1e3, 1) for k, v in tm_hi.items()}}} if t_hi is not None else {}),
                     "ratio_per_two_doublings": ratio},
        "cpu_baseline": {"value": value, "unit": "ms", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def _count(minimum):
    def parse(s):
        v = int(s)
        if v < minimum:
            raise argparse.ArgumentTypeError(f"must be >= {minimum}")
        return v
    return parse


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_count(1), default=3, help="timed steps (complete proves) per leg")
    ap.add_argument("--warmup", type=_count(0), default=3, help="untimed proves before the timed steps of each leg")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the proof of the last one to DIR/proof.npy (see dump_outputs)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2-height", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--low-memory", type=int, default=None, choices=[0, 1, 2],
                    help="tvm_ctx_set_low_memory: 0 auto (default), 1 always just-in-time LDE, 2 always cache")
    ap.add_argument("--workload-dir", default=None,
                    help="directory written by tools/make_workload.py (e.g. spin_20): prove the reference's own benchmark program "
                         "from its 149 table columns with tvm_prove_tables (all table stages on the device) instead of synthetic tables")
    ap.add_argument("--from-aet", action="store_true",
                    help="with --workload-dir: tvm_prove_aet on the AET arrays written by tools/make_workload.py --aet (table fill on the device)")
    ap.add_argument("--ldt", default="auto", choices=["auto", "fri", "stir"],
                    help="low-degree test; auto = the reference's own choice (STIR from padded height 2^16 on)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.workload_dir:
        run_gpu_workload(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
