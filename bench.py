#!/usr/bin/env python3
"""bench.py -- pairings/sec of the batched BLS12-381 pairing path on N B200s (one process per GPU).

    python bench.py --gpus 1 --steps K --warmup W                       # our arm
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                                # CPU arm (C oracle port)
    python bench.py ... --dump-outputs DIR                              # also write the last step's Gt values

A "step" is one pass of the hot path (Miller loop + final exponentiation) over one batch of
2^LOG2 synthetic (G1,G2) pairs per GPU (weak scaling).  `value` times the kernels with inputs
already resident in HBM; `e2e` goes through the host-buffer C-ABI call (zkp_pairing_batch) from
pinned host memory, copies included.  Prints ONE JSON line on rank 0.

Besides the headline the line carries sub-records for the other BASELINE.json configs:
  N = 1 : `configs.miller_only`, `configs.final_exp_only` (config 2, 2^20), `configs.checks4` and
          `configs.checks4_prepared` (config 3, 2^18 Groth16-shaped 4-pair checks)
  N > 1 : `product` (per-rank shared-accumulator Miller loops -> Fp12 partial -> NCCL all_gather of the
          576-byte partials -> multiply -> one final exponentiation; checked bit for bit against the
          single-GPU product of the same seeded pairs), `config5` (2^24 pairings in total, sliced over the
          ranks) and `strong` (2^20 pairings in total, sliced over the ranks)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pairings_per_sec"
UNIT = "pairings/s"
# Algorithmic work (BASELINE.md section 2 / SURVEY 8d): Fp-muls x 300 wide MACs
MACS_PER_FP_MUL = 300
FP_MULS_MILLER, FP_MULS_MILLER_EXTRA_PAIR, FP_MULS_FINAL_EXP = 6916, 4684, 9101
MACS_MILLER = FP_MULS_MILLER * MACS_PER_FP_MUL
MACS_FINAL_EXP = FP_MULS_FINAL_EXP * MACS_PER_FP_MUL
MACS_PER_PAIRING = MACS_MILLER + MACS_FINAL_EXP
MACS_PER_CHECK4 = (FP_MULS_MILLER + 3 * FP_MULS_MILLER_EXTRA_PAIR + FP_MULS_FINAL_EXP) * MACS_PER_FP_MUL
MACS_PRODUCT_PAIR = (FP_MULS_MILLER + 3 * FP_MULS_MILLER_EXTRA_PAIR) * MACS_PER_FP_MUL / 4.0   # four pairs per shared accumulator
IO_BYTES_PER_PAIRING = 288 + 576
NOMINAL_WIDE_PEAK = 148 * 4 * 8 * 1.965e9     # one IMAD.WIDE per 4 cycles per scheduler: 148 SM x 4 x 8 lanes x max clock
EXECUTED_PROFILE = os.path.join(ROOT, "profiles", "executed_work.json")
# --dump-outputs: at most 2^15 Gt values (2^15 x 144 limbs x 8 bytes = 37.7 MB), rows above that drawn with a fixed seed
DUMP_ROWS = 1 << 15
DUMP_SEED = 0xD0D0


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f).get("hbm_gbs")
    except Exception:
        return 6650.0   # fallback of /opt/skills/guides/B200_PROFILING.md


def executed_profile():
    """Counters of the SHIPPED build read from a committed profile (tools/ncu_executed_work.py writes it from
    an ncu capture): wide-MAC instructions and DRAM bytes per pairing, with the build id they belong to."""
    try:
        with open(EXECUTED_PROFILE) as f:
            return json.load(f)
    except Exception:
        return None


def workload_config(log2: int):
    """The `config` object, identical in both arms (ours / reference)."""
    return {"workload": "2^%d independent random BLS12-381 pairings per GPU (a_i*G1gen, b_i*G2gen from seeded 64-bit scalars; "
                        "Miller loop + final exponentiation, Gt out)" % log2,
            "pairings_per_gpu_per_step": 1 << log2,
            "parallelism": "independent pairings sharded one contiguous slice per GPU, no data-path collective",
            "l2": "inputs+outputs per step = %.0f MB > 126 MB L2; the path is integer-multiply bound, not cache sensitive"
                  % ((1 << log2) * IO_BYTES_PER_PAIRING / 1e6)}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2-batch", type=int, default=20, help="pairings per GPU per step = 2^this")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the sub-records of the other BASELINE configs")
    ap.add_argument("--config5-log2", type=int, default=24, help="total pairings of the config5 sub-record (N > 1)")
    ap.add_argument("--ref-seconds", type=float, default=None, help="--impl reference: CPU seconds per step (default: bounded by the step count)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the Gt values of the last step (rank 0's batch) to DIR/gt.npy: float64 (k, 144), "
                         "each Fp12 as 144 little-endian 32-bit limbs; batches above 2^15 pairings are sampled with a fixed seed")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


# ------------------------------------------------------------------------------------------ CPU arm

def cpu_oracle_rate(n_sample: int, threads: int, seed: int = 0x5EED):
    """Times the C oracle (oracle/zkp_oracle.c, a port of the reference's CPU path with the
    reference's tower structure) on n_sample seeded pairings with `threads` host threads."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import coracle
    import util
    coracle.build()
    g1, i1, g2, i2 = util.oracle_points(coracle, seed, 0, n_sample)     # untimed input generation
    t0 = time.perf_counter()
    coracle.pairing_batch(g1, None, g2, None, nthreads=threads)
    dt = time.perf_counter() - t0
    return n_sample / dt, dt


def cpu_baseline(target_seconds: float):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import coracle
    cores = coracle.ncores()
    rate, _ = cpu_oracle_rate(8 * cores, cores)                        # calibration
    n = max(cores, int(rate * target_seconds))
    n = min(n, 1 << 16)
    rate, dt = cpu_oracle_rate(n, cores)
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d seeded pairings (a_i*G1, b_i*G2) in %.1f s on %d host threads, C restatement of the reference tower "
                      "(Montgomery Fp instead of the reference's BigUint)" % (n, dt, cores)}


def run_reference(args):
    """--impl reference: the reference's CPU path.  The Rust crate cannot be built here (no rustc,
    un-vendored sp1 git dependency) and its src/pairings.rs is empty, so this is the oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import coracle
    cores = coracle.ncores()
    rate0, _ = cpu_oracle_rate(8 * cores, cores)
    # bounded sample per step so that (steps + warmup) stays within a few minutes
    per_step_s = args.ref_seconds if args.ref_seconds else max(2.0, min(20.0, 150.0 / max(1, args.steps + args.warmup)))
    n = max(cores, min(1 << 16, int(rate0 * per_step_s)))
    for _ in range(args.warmup):
        cpu_oracle_rate(n, cores)
    t = 0.0
    for _ in range(args.steps):
        _, dt = cpu_oracle_rate(n, cores)
        t += dt
    rate = n * args.steps / t
    sample = ("%d seeded pairings per step on %d host threads: a bounded sample of the 2^%d-pairing workload (C restatement of the "
              "reference tower; the Rust crate has no pairing and cannot be built here)" % (n, cores, args.log2_batch))
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args.log2_batch),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------ GPU arm

class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons of one GPU during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import zkvm_pairings_b200 as z
    from zkvm_pairings_b200 import sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the pairing engine has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL's own log (communicator / rank lines) stays on: it goes to stderr with everything else that
        # libraries print (main() parks the real stdout), so rank 0's stdout still carries ONE JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "INFO"                   # never quieter than INFO: the communicator lines must be visible
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")  # (and no chattier than the init lines unless the caller asks)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n = 1 << args.log2_batch
    eng = z.PairingEngine([local])
    dev = torch.device("cuda", local)
    # the launches go on torch's CURRENT stream (a side stream here), so torch.cuda.Event timing sees them
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    st = tstream.cuda_stream

    def timed_ms(fn, steps, warmup):
        """CUDA-event time of `steps` back-to-back calls on the launching stream, per call (ms)."""
        for _ in range(warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    # ---- synthetic inputs, generated on the device (valid subgroup points), untimed
    g1 = torch.empty((n, 12), dtype=torch.int64, device=dev)
    g2 = torch.empty((n, 24), dtype=torch.int64, device=dev)
    i1 = torch.empty(n, dtype=torch.uint8, device=dev)
    i2 = torch.empty(n, dtype=torch.uint8, device=dev)
    out = torch.empty((n, 72), dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    SEED = 0x5EED5EED
    eng.gen_points_dev(SEED, sharding.synthetic_first_index(rank, n), n, g1, i1, g2, i2, stream=st)
    torch.cuda.synchronize()

    # ---- integer-multiply roofline denominators, measured in this run (every issued multiply counted,
    #      launch geometry swept inside zkp_imad_peak)
    peak_wide = eng.imad_peak(0)
    peak_lo = eng.imad_peak(1)
    peak_chain = eng.imad_peak(2)
    peak = max(peak_wide, peak_chain)

    def step():
        eng.pairing_dev(z.MODE_PAIRING, out, g1=g1, g2=g2, err=err, stream=st)

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    launches0 = eng.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev[0].record()
    for k in range(args.steps):
        step()
        ev[k + 1].record()
    barrier()
    kernel_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    total_ms = ev[0].elapsed_time(ev[-1])
    launches = eng.launch_count - launches0
    clocks = sampler.stop() if sampler else None
    assert int(err.item()) == 0, "non-canonical synthetic input?"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)        # before the records below reuse `out`
    max_ms = sharding.max_over_ranks(total_ms, world, dev)
    value = sharding.whole_job_rate(n, args.steps, world, max_ms)

    # ---- end to end through the host-buffer C-ABI call, pinned host memory, copies in the timed region
    e2e_n = n
    h_g1 = torch.empty((e2e_n, 12), dtype=torch.int64).pin_memory()
    h_g2 = torch.empty((e2e_n, 24), dtype=torch.int64).pin_memory()
    h_out = torch.empty((e2e_n, 72), dtype=torch.int64).pin_memory()
    h_g1.copy_(g1[:e2e_n])
    h_g2.copy_(g2[:e2e_n])
    n_g1, n_g2, n_out = h_g1.numpy().view(np.uint64), h_g2.numpy().view(np.uint64), h_out.numpy().view(np.uint64)
    lib = eng._lib
    import ctypes

    def p(a):
        return a.ctypes.data_as(ctypes.c_void_p)

    def e2e_step():
        rc = lib.zkp_pairing_batch(eng._ctx, p(n_g1), None, p(n_g2), None, e2e_n, p(n_out))
        assert rc == 0, lib.zkp_last_error()

    e2e_step()                      # warm-up (allocates the pipeline buffers)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_dt = time.perf_counter() - t0
    e2e_value = sharding.whole_job_rate(e2e_n, args.steps, world, 1e3 * sharding.max_over_ranks(e2e_dt, world, dev))
    # the e2e result must equal the device-resident result (same inputs)
    same = bool(torch.equal(h_out[:4096], out[:4096].cpu()))
    del h_g1, h_g2, h_out, n_g1, n_g2, n_out

    extra_launches0 = eng.launch_count
    configs, product, config5, strong = None, None, None, None
    if not args.no_configs:
        product = bench_product(eng, z, sharding, torch, dist, world, rank, dev, st, n, SEED, g1, g2, out, err, args.steps, barrier)
        if world == 1:
            configs = bench_configs(eng, z, torch, np, dev, st, n, g1, g2, out, err, peak, args.steps, timed_ms)
        else:
            del g1, g2, i1, i2, out
            torch.cuda.empty_cache()
            config5 = bench_sliced(eng, z, sharding, torch, dist, world, rank, dev, st, 1 << args.config5_log2, 0xC5C5, 1, barrier,
                                   with_product=True)
            strong = bench_sliced(eng, z, sharding, torch, dist, world, rank, dev, st, 1 << args.log2_batch, SEED, args.steps, barrier,
                                  with_product=False)
            strong["single_gpu_reference"] = "value of the N=1 line of the same sweep (same 2^%d pairings on one GPU)" % args.log2_batch

    if rank == 0:
        per_step_ms = sum(kernel_ms) / len(kernel_ms)
        pairs_per_s_kernel = n / (per_step_ms * 1e-3)
        achieved = pairs_per_s_kernel * MACS_PER_PAIRING
        prof = executed_profile()
        exe = prof["executed_wide_macs_per_pairing"] if prof else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": workload_config(args.log2_batch),
            "engine": eng.version(),
            # integer-multiply roofline (SURVEY 8d): ALGORITHMIC 32x32->64 MACs per second (16,017 Fp-muls x 300 per
            # pairing) against the best wide-MAC rate measured in this run on this GPU
            "roofline": {"bound": "imad", "achieved": achieved / 1e12, "peak": peak / 1e12, "unit": "T wide-MAC/s",
                         "frac": achieved / peak,
                         "traffic": (prof["dram_bytes_per_pairing"] * n) if prof and prof.get("dram_bytes_per_pairing") else None,
                         "traffic_source": ("%s (ncu dram__bytes_read.sum + dram__bytes_write.sum of one 2^%d step of build '%s', per pairing x this batch)"
                                            % (os.path.relpath(EXECUTED_PROFILE, ROOT), prof["log2_batch"], prof["build"])) if prof else None,
                         "kernel": "one step = k_pairing<1> + 2 halves x 6 x (k_fe_batch_inv + k_fe_stage)", "kernel_ms": per_step_ms,
                         "algorithmic_macs_per_pairing": MACS_PER_PAIRING,
                         # utilisation of the multiply pipe by the wide MACs the shipped build EXECUTES (opcode count from ncu,
                         # committed profile), against the nominal pipe rate at max clock and against the measured peak
                         "executed_macs_per_pairing": exe,
                         "executed_frac": (pairs_per_s_kernel * exe / NOMINAL_WIDE_PEAK) if exe else None,
                         "executed_frac_of_measured_peak": (pairs_per_s_kernel * exe / peak) if exe else None,
                         "executed_source": ("%s (ncu opcode count of IMAD.WIDE* for build '%s')" % (os.path.relpath(EXECUTED_PROFILE, ROOT), prof["build"])) if prof else None,
                         "note": "achieved/frac use SURVEY 8d's ALGORITHMIC count; the kernels reach the same field elements with fewer "
                                 "MACs (compressed cyclotomic squarings, factorised hard part), so frac can exceed 1 -- executed_frac "
                                 "(nominal pipe rate) is the honest utilisation figure",
                         "peak_source": "measured in this run (zkp_imad_peak): max of independent IMAD.WIDE.U32 chains and the "
                                        "carry-chained Montgomery rows over five launch geometries, every issued multiply counted",
                         "peak_wide_independent": peak_wide / 1e12, "peak_wide_carry_chain": peak_chain / 1e12,
                         "peak_imad_32bit": peak_lo / 1e12,
                         "nominal_wide_peak": NOMINAL_WIDE_PEAK / 1e12,
                         "hbm": {"algorithmic_bytes_per_pairing": IO_BYTES_PER_PAIRING,
                                 "achieved_gbs": pairs_per_s_kernel * IO_BYTES_PER_PAIRING / 1e9, "peak_gbs": hbm_peak(),
                                 "note": "HBM is three orders of magnitude away from binding (SURVEY 8d)"}},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": e2e_n * 288, "d2h_bytes_per_step": e2e_n * 576,
                    "steps": args.steps, "matches_device_path": same},
            "gpu_launches": launches,
            "gpu_launches_subrecords": eng.launch_count - extra_launches0,
            "clocks": clocks,
        }
        if configs:
            line["configs"] = configs
            line["roofline"]["dominant_kernel"] = configs["miller_only"]["roofline"]
        if product:
            line["product"] = product
        if config5:
            line["config5"] = config5
        if strong:
            line["strong"] = strong
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
        emit(line)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def dump_rows(n: int):
    """Rows of an n-pairing batch that --dump-outputs writes: all of them up to DUMP_ROWS, else DUMP_ROWS rows drawn
    without replacement by a fixed seed, in increasing order, so that every build dumps the same rows."""
    import numpy as np
    if n <= DUMP_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ROWS, replace=False))


def dump_outputs(path, out):
    """DIR/gt.npy: the rows dump_rows() picks from `out` (the (n, 72) int64 Gt tensor of the timed path), each Fp12 as
    144 little-endian 32-bit limbs in float64, which holds them exactly."""
    import numpy as np
    import torch
    rows = torch.from_numpy(dump_rows(out.shape[0])).to(out.device)
    gt = out.index_select(0, rows).cpu().numpy().view("<u4").astype(np.float64)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "gt.npy"), gt)


def _rate_record(units, ms, unit, macs_per_unit=None, peak=None, **extra):
    rec = {"value": units / (ms * 1e-3), "unit": unit, "ms_per_step": ms, "units_per_step": units}
    if macs_per_unit and peak:
        ach = rec["value"] * macs_per_unit
        rec["roofline"] = {"bound": "imad", "achieved": ach / 1e12, "peak": peak / 1e12, "unit": "T wide-MAC/s", "frac": ach / peak,
                           "algorithmic_macs_per_unit": macs_per_unit, "kernel_ms": ms}
    rec.update(extra)
    return rec


def bench_configs(eng, z, torch, np, dev, st, n, g1, g2, out, err, peak, steps, timed_ms):
    """N = 1 sub-records: the dominant kernel alone, BASELINE config 2 (final exponentiation only, 2^20) and
    config 3 (2^18 Groth16-shaped 4-pair checks, plain and with the three verifying-key G2 points prepared)."""
    from zkvm_pairings_b200 import workloads
    rec = {}
    ml = torch.empty((n, 72), dtype=torch.int64, device=dev)
    ms = timed_ms(lambda: eng.pairing_dev(z.MODE_MILLER, ml, g1=g1, g2=g2, err=err, stream=st), steps, 1)
    rec["miller_only"] = _rate_record(n, ms, "miller loops/s", MACS_MILLER, peak,
                                      kernel="k_pairing<1> launched alone (mode 1: Miller loop, canonical Fp12 out), 2^%d pairs" % (n.bit_length() - 1))
    ms = timed_ms(lambda: eng.pairing_dev(z.MODE_FINAL_EXP, out, in_fp12=ml, err=err, stream=st), steps, 1)
    rec["final_exp_only"] = _rate_record(n, ms, "final exponentiations/s", MACS_FINAL_EXP, peak,
                                         workload="BASELINE config 2: final exponentiation only on 2^%d Miller-loop outputs" % (n.bit_length() - 1))
    del ml
    nc = 1 << 18
    wl = workloads.groth16_checks(eng, nc)
    d_g1 = torch.from_numpy(wl["g1"].view(np.int64)).to(dev)
    d_g2 = torch.from_numpy(wl["g2"].view(np.int64)).to(dev)
    d_var = torch.from_numpy(wl["g2_var"].view(np.int64)).to(dev)
    d_fixed = torch.from_numpy(wl["fixed"].view(np.int64)).to(dev)
    one = torch.zeros(nc, dtype=torch.uint8, device=dev)
    gt = out[:nc]
    ms = timed_ms(lambda: eng.pairing_dev(z.MODE_PAIRING, gt, g1=d_g1, g2=d_g2, n_checks=nc, pairs_per_check=4, is_one=one, err=err, stream=st),
                  steps, 1)
    ok = bool(np.array_equal(one.cpu().numpy().astype(bool), wl["expect_one"]))
    ref_gt = gt.clone()
    rec["checks4"] = _rate_record(nc, ms, "checks/s", MACS_PER_CHECK4, peak, verdicts_match_construction=ok,
                                  workload="BASELINE config 3: 2^18 Groth16-shaped product checks of 4 pairs, shared final exponentiation, 1 % corrupted")
    tab = torch.empty((3, eng.G2_PREPARED_U64), dtype=torch.int64, device=dev)
    eng.g2_prepare_dev(d_fixed, 3, tab, err=err, stream=st)
    one.zero_()
    ms = timed_ms(lambda: eng.multi_pairing_prepared_dev(gt, d_g1, d_var, nc, 4, tab, 3, is_one=one, err=err, stream=st), steps, 1)
    ok = bool(np.array_equal(one.cpu().numpy().astype(bool), wl["expect_one"])) and bool(torch.equal(gt, ref_gt))
    rec["checks4_prepared"] = _rate_record(nc, ms, "checks/s", None, None, bit_identical_to_plain=ok,
                                           workload="same checks, the three verifying-key G2 points as prepared line tables (G2Prepared)")
    assert int(err.item()) == 0
    return rec


def _fold_partials(eng, torch, dev, st, parts):
    """Product of a few Fp12 partials (rows of a (k, 72) int64 device tensor) -> (72,) device tensor."""
    k = parts.shape[0]
    scratch = torch.empty(eng.product_scratch_elems(k) * 72, dtype=torch.int64, device=dev)
    res = torch.empty(72, dtype=torch.int64, device=dev)
    eng.fp12_product_dev(parts.contiguous(), k, scratch, res, stream=st)
    return res


def bench_product(eng, z, sharding, torch, dist, world, rank, dev, st, n, seed, g1, g2, out, err, steps, barrier):
    """The one real exchange of the path (SURVEY 8e, BASELINE config 5b): every rank folds its slice's pairs into one
    Fp12 partial (shared-accumulator Miller loops, four pairs each, then a product tree), the 576-byte partials are
    all-gathered over NCCL, multiplied, and ONE final exponentiation is applied.  Rank 0 then recomputes the product
    of all world*n seeded pairs on its own GPU and asserts the two are bit-identical."""
    nc4 = n // 4
    ml = out[:nc4]
    scratch = torch.empty(eng.product_scratch_elems(nc4) * 72, dtype=torch.int64, device=dev)
    partial = torch.empty(72, dtype=torch.int64, device=dev)
    gt = torch.empty((1, 72), dtype=torch.int64, device=dev)
    prod = [None]

    def one_product():
        eng.pairing_dev(z.MODE_MILLER_FOR_FINAL_EXP, ml, g1=g1, g2=g2, n_checks=nc4, pairs_per_check=4, err=err, stream=st)
        eng.fp12_product_dev(ml, nc4, scratch, partial, err=err, stream=st)
        gathered = sharding.gather_partials(partial, world)             # NCCL all_gather, ordered with the launching stream
        prod[0] = _fold_partials(eng, torch, dev, st, gathered)
        eng.pairing_dev(z.MODE_FINAL_EXP, gt, in_fp12=prod[0].view(1, 72), n_checks=1, err=err, stream=st)

    one_product()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = eng.launch_count
    e0.record()
    for _ in range(steps):
        one_product()
    e1.record()
    barrier()
    ms = sharding.max_over_ranks(e0.elapsed_time(e1), world, dev) / steps
    launches = (eng.launch_count - l0) // steps
    result_gt = gt[0].clone()
    # ---- verification on rank 0: the same world*n seeded pairs, one GPU, per-pair Miller loops (k = 1) folded
    matches = None
    if rank == 0:
        acc = None
        for r in range(world):
            if r == 0:
                vg1, vg2 = g1, g2
            else:
                vg1, vg2 = torch.empty_like(g1), torch.empty_like(g2)
                vi1 = torch.empty(n, dtype=torch.uint8, device=dev)
                vi2 = torch.empty(n, dtype=torch.uint8, device=dev)
                eng.gen_points_dev(seed, sharding.synthetic_first_index(r, n), n, vg1, vi1, vg2, vi2, stream=st)
            vml = out
            eng.pairing_dev(z.MODE_MILLER, vml, g1=vg1, g2=vg2, err=err, stream=st)
            vs = torch.empty(eng.product_scratch_elems(n) * 72, dtype=torch.int64, device=dev)
            vp = torch.empty(72, dtype=torch.int64, device=dev)
            eng.fp12_product_dev(vml, n, vs, vp, err=err, stream=st)
            acc = vp if acc is None else _fold_partials(eng, torch, dev, st, torch.stack([acc, vp]))
            torch.cuda.synchronize()
        vgt = torch.empty((1, 72), dtype=torch.int64, device=dev)
        eng.pairing_dev(z.MODE_FINAL_EXP, vgt, in_fp12=acc.view(1, 72), n_checks=1, err=err, stream=st)
        torch.cuda.synchronize()
        # (the timed path runs the Miller loops with free line scaling, so its un-exponentiated product differs from this
        # one by a subfield factor; the Gt values must be bit-identical)
        matches = bool(torch.equal(vgt[0], result_gt))
        assert matches, "sharded product differs from the single-GPU product"
    barrier()
    total = world * n
    rec = _rate_record(total, ms, "pairs/s", None, None,
                       workload="one product over %d x 2^%d seeded pairs: per-GPU shared-accumulator Miller loops (4 pairs each) -> Fp12 "
                                "partial -> gather -> multiply -> one final exponentiation" % (world, n.bit_length() - 1),
                       exchange=("ncclAllGather of one 576-byte Fp12 partial per rank (torch.distributed, NCCL over NVLink)" if world > 1
                                 else "single GPU: no exchange"),
                       bytes_gathered_per_rank=576 if world > 1 else 0, launches_per_step=launches,
                       bit_identical_to_single_gpu_product=matches, algorithmic_macs_per_pair=MACS_PRODUCT_PAIR)
    return rec


def bench_sliced(eng, z, sharding, torch, dist, world, rank, dev, st, total, seed, steps, barrier, with_product):
    """A FIXED total of independent pairings sliced contiguously over the ranks (SURVEY 8e): `config5` (2^24 in total,
    BASELINE config 5, plus its global product through the gather, checked by a checksum of checksums: the product of
    all Gt outputs equals the final exponentiation of the product of all Miller outputs) and `strong` (2^20 in total)."""
    lo, hi = sharding.slice_bounds(total, world, rank)
    m = hi - lo
    g1 = torch.empty((m, 12), dtype=torch.int64, device=dev)
    g2 = torch.empty((m, 24), dtype=torch.int64, device=dev)
    i1 = torch.empty(m, dtype=torch.uint8, device=dev)
    i2 = torch.empty(m, dtype=torch.uint8, device=dev)
    out = torch.empty((m, 72), dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    eng.gen_points_dev(seed, lo, m, g1, i1, g2, i2, stream=st)
    eng.pairing_dev(z.MODE_PAIRING, out, g1=g1, g2=g2, err=err, stream=st)    # full-size warm-up: grows the scratch pool (2.6 KB per pairing)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        eng.pairing_dev(z.MODE_PAIRING, out, g1=g1, g2=g2, err=err, stream=st)
    e1.record()
    barrier()
    ms = sharding.max_over_ranks(e0.elapsed_time(e1), world, dev) / steps
    rec = _rate_record(total, ms, UNIT, None, None, scaling="strong", pairings_per_gpu=m,
                       workload="2^%d independent pairings in total, one contiguous slice per GPU" % (total.bit_length() - 1))
    if with_product:
        def fold(t, k):
            s = torch.empty(eng.product_scratch_elems(k) * 72, dtype=torch.int64, device=dev)
            r = torch.empty(72, dtype=torch.int64, device=dev)
            eng.fp12_product_dev(t, k, s, r, err=err, stream=st)
            return r

        def gather_fold(partial):
            return _fold_partials(eng, torch, dev, st, sharding.gather_partials(partial, world))

        gt_checksum = gather_fold(fold(out, m))                      # product of all 2^24 Gt outputs
        nc4 = m // 4
        barrier()
        e0.record()
        eng.pairing_dev(z.MODE_MILLER_FOR_FINAL_EXP, out[:nc4], g1=g1, g2=g2, n_checks=nc4, pairs_per_check=4, err=err, stream=st)
        part = fold(out[:nc4], nc4)
        if m % 4:
            tail = torch.empty((m % 4, 72), dtype=torch.int64, device=dev)
            eng.pairing_dev(z.MODE_MILLER_FOR_FINAL_EXP, tail, g1=g1[4 * nc4:], g2=g2[4 * nc4:], err=err, stream=st)
            part = _fold_partials(eng, torch, dev, st, torch.cat([part.view(1, 72), tail]))
        prod = gather_fold(part)
        gt = torch.empty((1, 72), dtype=torch.int64, device=dev)
        eng.pairing_dev(z.MODE_FINAL_EXP, gt, in_fp12=prod.view(1, 72), n_checks=1, err=err, stream=st)
        e1.record()
        barrier()
        pms = sharding.max_over_ranks(e0.elapsed_time(e1), world, dev)
        ok = bool(torch.equal(gt[0], gt_checksum))
        assert ok, "product of the Gt outputs != final exponentiation of the Miller product"
        rec["product"] = {"value": total / (pms * 1e-3), "unit": "pairs/s", "ms": pms, "bytes_gathered_per_rank": 576,
                          "exchange": "ncclAllGather of one 576-byte Fp12 partial per rank",
                          "checksum_of_checksums_ok": ok}
    assert int(err.item()) == 0
    return rec


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract, written to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # Libraries write banners and logs to file descriptor 1 from C (NCCL prints there): park the real stdout and point
    # fd 1 at stderr until the JSON line is written, so stdout carries exactly one line and stderr carries the logs.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
