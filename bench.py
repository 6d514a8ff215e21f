#!/usr/bin/env python3
"""bench.py -- headline benchmark of the create_proof hot path (BASELINE.json configs[1]):
BN254 G1 Pippenger MSM over 2^20 random points / uniform scalars per GPU, B200 vs the CPU best_multiexp.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one batch of MSMS_PER_STEP = 16 commitments, each an MSM of n = 2^20 pairs per GPU against a resident basis
(create_proof commits its advice columns back to back against g_lagrange: 19 of them in the sync-step shape). With N ranks
every MSM of the batch is ONE MSM of N * 2^20 pairs sharded by point range (SURVEY.md 8e): every rank reduces its range to a
single point, the batch's 96-byte partials are all-gathered once over NCCL and folded in one C call.
`value` = pairs per second of the whole job with scalars resident in HBM; `e2e` = the same through the host-buffer C-ABI
call (pinned host scalars -> H2D -> kernels -> 96-byte results D2H inside the timed region).

Every N prints `parity` flags: the folded result of a timed step is compared with the point the oracle computes from the
known discrete logs of the bases (sum_i s_i * h_i) * G1; the sharded 2^23 MSM with the single-GPU one; the multi-device
NTT and proof with their single-device outputs, bit for bit.

Extra keys: `roofline` (dominant kernel msm_accumulate_kernel vs measured HBM peak, plus the INT32-pipe view that
actually binds it, plus the HBM-class quotient kernels), `cpu_baseline` (the oracle port of halo2's best_multiexp on this
box's cores, median of 5 after a full-size warm-up), `msm_sizes` (2^20 / 2^23 / 2^24 x scalar distributions),
`strong_scaling` (one 2^23 MSM on 1 GPU vs sharded over N), `ntt` (2^20 / 2^22 / 2^23 / 2^25; six-step across N devices),
`proof` (create_proof wall time: Python driver, compiled driver, N-device context), `stages_ms`, `clocks`, `gpu_launches`.

--impl reference times the CPU restatement of the reference's own path (oracle/_ref; the Rust crates cannot be
built in this image -- DESIGN.md) on the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only: nothing is written there, bytecode caches included

LOG_N = 20
N_PAIRS = 1 << LOG_N
MSMS_PER_STEP = 16  # commitments per step (one batch through spb_msm_batch*)
N_SCALAR_SETS = 8   # 8 x 32 MiB of scalars rotate through the timed steps: 256 MiB > 126 MB L2
R_MOD = 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001
STRONG_LOG_N = 23   # the north-star strong-scaling size: one 2^23 MSM on 1 GPU vs sharded over N
SEED_POINTS, SEED_SCALARS = 0x5eed0002, 0x5eed0003
BENCH_VK_DIGEST = 0x5eedd16e57   # stand-in for VerifyingKey::transcript_repr, the same in the Python and the compiled driver


def rand_fr(n, seed):
    """n pseudo-random valid Fr residues: uniform 252-bit values (top limb masked to 60 bits, < r) read as Montgomery limbs."""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 2**63, size=(n, 4), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 60) - 1)
    return a


def fr_limbs(v):
    m = v % R_MOD
    return np.array([(m >> (64 * j)) & 0xFFFFFFFFFFFFFFFF for j in range(4)], dtype=np.uint64)


def scalars_distribution(name, n, seed):
    """SURVEY.md 8d scalar families: (U) uniform, (W) witness-like: 70 % zero, 20 % < 2^16, 9 % < 2^104, 1 % uniform
    (halo2-lib advice columns; the small values come from pools of 4096 distinct ones, as witness columns repeat values),
    (E) every scalar = r - 1 (the worst case of the counting sort: one bucket per window)."""
    if name == "uniform":
        return rand_fr(n, seed)
    mont = (1 << 256) % R_MOD
    if name == "all_minus_one":
        return np.broadcast_to(fr_limbs((R_MOD - 1) * mont), (n, 4)).copy()
    rng = np.random.default_rng(seed)
    out = np.zeros((n, 4), dtype=np.uint64)
    u = rng.random(n)
    for lo, hi, bits in ((0.70, 0.90, 16), (0.90, 0.99, 104)):
        idx = np.nonzero((u >= lo) & (u < hi))[0]
        pool = np.stack([fr_limbs((int.from_bytes(rng.bytes(16), "little") % (1 << bits)) * mont) for _ in range(4096)])
        out[idx] = pool[rng.integers(0, 4096, size=len(idx))]
    big = np.nonzero(u >= 0.99)[0]
    out[big] = rand_fr(len(big), seed + 1)
    return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.stop_flag = False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0])); self.max_mhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def dump_commitments(out_dir, name, jacobian):
    """(count, 12) Jacobian Montgomery limbs -> out_dir/<name>.npy, float64 of shape (count, 2, 8): the affine x and y of each
    point as eight little-endian 32-bit limbs, which float64 holds exactly (the identity is x = y = 0). Affine coordinates
    are unique, so two builds that compute the same points write the same file."""
    from spectre_b200 import halo2
    xy = [halo2.jacobian_to_affine_ints(j) for j in np.asarray(jacobian, dtype=np.uint64).reshape(-1, 12)]
    limbs = np.array([[[(v >> (32 * i)) & 0xFFFFFFFF for i in range(8)] for v in p] for p in xy], dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), limbs)


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def workload_config():
    """`config` of the JSON line: the WORKLOAD, identical in both arms (--impl ours / reference); how each arm runs it is in
    `schedule` (ours) / `cpu_baseline.sample` (reference)."""
    return {"workload": workload_text(), "log_n": LOG_N, "msms_per_step": MSMS_PER_STEP, "scalar_bits": 252,
            "l2": "GPU arm: scalars rotate over 8 resident sets (256 MiB > 126 MB L2), the 64 MiB basis is reused as in the prover; "
                  "CPU arm: one scalar set, 96 MiB per MSM streams through the host caches"}


def workload_text():
    return ("BN254 G1 MSM 2^20 random points / uniform 252-bit scalars per GPU (BASELINE configs[1]); step = %d such commitments "
            "(one batch); N ranks = every MSM is one N*2^20 MSM sharded by point range" % MSMS_PER_STEP)


# ---- CPU arm ------------------------------------------------------------------------------------------------------------
def cpu_msm_samples(orc, sc, bases, threads, samples):
    """full-size warm-up, then `samples` timed full MSMs -> (list of seconds, last result)"""
    res = orc.best_multiexp(sc, bases, threads=threads)
    ts = []
    for _ in range(samples):
        t0 = time.perf_counter()
        res = orc.best_multiexp(sc, bases, threads=threads)
        ts.append(time.perf_counter() - t0)
    return ts, res


def run_reference(args):
    """CPU arm: the oracle's restatement of halo2 best_multiexp (the reference's own path) on the host cores. A step of the
    GPU arm is a batch of 16 MSMs; a CPU step is a bounded sample of it: ONE of the 16 (full 2^20 pairs)."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build(); orc.lib()
    threads = os.cpu_count() or 1
    sc = orc.fr_random_chacha(N_PAIRS, SEED_SCALARS)
    bases = orc.g1_fixed_base_mul(orc.fr_random_chacha(N_PAIRS, SEED_POINTS), threads=threads)
    for _ in range(max(1, min(args.warmup, 2))):              # full-size warm-up (page faults, thread pool, caches)
        orc.best_multiexp(sc, bases, threads=threads)
    ts = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        res = orc.best_multiexp(sc, bases, threads=threads)
        ts.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_commitments(args.dump_outputs, "msm_commitments", res)
    med = float(np.median(ts))
    val = N_PAIRS / med
    line = {
        "impl": "reference", "metric": "bn254_g1_msm_pairs_per_s", "value": val, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u256 (4x64-bit Montgomery limbs, CPU)", "data": "synthetic",
        "config": workload_config(),
        "sample": "one of a step's %d MSMs (full 2^20 pairs) per CPU step; value = 2^20 / median step seconds" % MSMS_PER_STEP,
        "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": threads, "kind": "port",
                         "sample": "one full 2^20-pair MSM per step after a full-size warm-up, median of %d; C restatement of halo2 best_multiexp "
                                   "(oracle/halo2_oracle.c); the Rust reference cannot be built here" % args.steps,
                         "seconds_min_median_max": [float(min(ts)), med, float(max(ts))]},
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- known-discrete-log check of an MSM result (oracle = checker only) ----------------------------------------------------
def mont_dot(orc, a, b):
    """sum_i a_i * b_i in Fr (Montgomery in / out): the oracle's restatement of arithmetic::compute_inner_product"""
    return orc.compute_inner_product(a, b).reshape(4)


def expected_point(orc, dots):
    """dots: list of (4,) Montgomery partial dot products (one per rank) -> affine (8,) limbs of (sum dots) * G1"""
    acc = np.ascontiguousarray(dots[0], dtype=np.uint64).reshape(4)
    for d in dots[1:]:
        acc = orc.fr_binop("fr_add", acc, np.ascontiguousarray(d, dtype=np.uint64).reshape(4))
    return orc.g1_fixed_base_mul(np.ascontiguousarray(acc.reshape(1, 4)), threads=1).reshape(8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ntt", action="store_true")
    ap.add_argument("--no-sizes", action="store_true", help="skip the MSM size / distribution table and the 2^23 strong-scaling block")
    ap.add_argument("--no-prove", action="store_true", help="skip keygen + create_proof of the two circuit shapes (spectre_b200/plonk.py and the compiled driver)")
    ap.add_argument("--no-cpp", action="store_true", help="skip the compiled driver (tests/cpp/prover_main.cpp) in the proof section")
    ap.add_argument("--prove-k", type=int, default=23, help="k of the aggregation-shaped proof")
    ap.add_argument("--prove-k-step", type=int, default=20, help="k of the sync-step-shaped proof")
    ap.add_argument("--no-tables", action="store_true", help="skip spb_srs_precompute (W separate bucket sets, Horner over windows)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the commitments of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from spectre_b200 import halo2
    from spectre_b200 import dist as spb_dist

    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    cpu_pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_pg = dist.new_group(backend="gloo")   # host-side barrier / object exchange: idle ranks must not spin a kernel on their GPU
    dev = torch.device("cuda", local_rank)
    be = halo2.Backend([local_rank])
    use_oracle = not args.no_cpu_baseline
    orc = None
    if use_oracle:
        from oracle import oracle as orc
        if rank == 0:
            orc.build()
        if world > 1:
            dist.barrier(group=cpu_pg)
        orc.lib()

    def cpu_barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=cpu_pg)

    def gather_rows(row):
        """(4,) uint64 per rank -> list over ranks (host-side gloo all_gather)"""
        if world == 1:
            return [row]
        t = torch.from_numpy(np.ascontiguousarray(row, dtype=np.uint64).view(np.int64).copy())
        out = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(out, t, group=cpu_pg)
        return [o.numpy().view(np.uint64) for o in out]

    # ---- inputs (untimed): this rank's point range and scalar sets ------------------------------------------
    h_pts = rand_fr(N_PAIRS, SEED_POINTS + 1000 * rank)       # discrete logs of this rank's bases (Montgomery limbs)
    pts = be.g1_fixed_base_mul(h_pts)                         # random points h_i * G1
    t_setup = time.perf_counter()
    params = halo2.ParamsKZG.from_parts(be, LOG_N, g_lagrange=pts)
    if not args.no_tables:
        params.precompute()   # one-time per SRS (static bases): 2^(c*j) window tables, W x the basis memory
    setup_s = time.perf_counter() - t_setup
    host_sets = [torch.from_numpy(rand_fr(N_PAIRS, SEED_SCALARS + 1000 * rank + s).view(np.int64)).pin_memory() for s in range(N_SCALAR_SETS)]
    dev_sets = [h.to(dev) for h in host_sets]
    host_np = [h.numpy().view(np.uint64) for h in host_sets]
    torch.cuda.synchronize()
    last = {}

    def fold(partials):
        """one all_gather for the whole batch of (count, 12) partial sums, then one C call folds it"""
        return spb_dist.fold_partials(partials, world, device=dev)

    def run_dev(first, steps):
        """`steps` steps of MSMS_PER_STEP commitments each through the batch entry point (three stream lanes), scalars in HBM"""
        for s in range(steps):
            ptrs = [dev_sets[(first + s * MSMS_PER_STEP + i) % N_SCALAR_SETS].data_ptr() for i in range(MSMS_PER_STEP)]
            last["dev"] = (first + s * MSMS_PER_STEP, fold(params.commit_batch_dev(halo2.BASIS_G_LAGRANGE, ptrs, N_PAIRS)))

    def run_e2e(first, steps):
        """same from pinned host buffers: H2D of every MSM's scalars and D2H of its result inside the call"""
        for s in range(steps):
            polys = [host_np[(first + s * MSMS_PER_STEP + i) % N_SCALAR_SETS] for i in range(MSMS_PER_STEP)]
            last["e2e"] = (first + s * MSMS_PER_STEP, fold(params.commit_batch(halo2.BASIS_G_LAGRANGE, polys)))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(run, steps, warmup):
        run(0, warmup)
        barrier()
        t0 = time.perf_counter()
        run(warmup * MSMS_PER_STEP, steps)
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        t = torch.tensor([wall_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    sampler = ClockSampler(local_rank); sampler.start()
    launches0 = be.kernel_launches
    wall_ms = timed(run_dev, args.steps, args.warmup)
    launches = be.kernel_launches - launches0
    sampler.stop_flag = True; sampler.join(timeout=2)
    adds = be.last_msm_adds // MSMS_PER_STEP       # the counter accumulates over a batch
    stages_pipelined = be.last_msm_stage_ms         # last MSM of the timed batch (other lane running concurrently)
    e2e_steps = max(3, args.steps // 2)
    e2e_wall_ms = timed(run_e2e, e2e_steps, 3)
    if args.dump_outputs and rank == 0:
        dump_commitments(args.dump_outputs, "msm_commitments", last["dev"][1])
        dump_commitments(args.dump_outputs, "msm_commitments_e2e", last["e2e"][1])

    # ---- parity of the timed path: last timed step, first MSM of the batch, vs (sum s_i h_i) * G1 from the oracle ------
    parity = {}
    if use_oracle:
        for tag in ("dev", "e2e"):
            first, folded = last[tag]
            dots = gather_rows(mont_dot(orc, host_np[first % N_SCALAR_SETS], h_pts))
            if rank == 0:
                want = expected_point(orc, dots)
                parity["msm_%s_result_equals_reference" % tag] = bool(np.array_equal(orc.g1_to_affine(folded[0]).reshape(8), want))
        if rank == 0:
            parity["msm_check"] = ("folded result of the last timed step (first of its %d MSMs, all %d rank shards) == (sum_i s_i h_i) G1 computed by the CPU oracle "
                                   "from the bases' known discrete logs" % (MSMS_PER_STEP, world))

    # one MSM at a time (what a caller that cannot batch sees), and its clean per-stage split
    lat, stages = [], {}
    for i in range(6):
        be_res = params.commit_dev(halo2.BASIS_G_LAGRANGE, dev_sets[i % N_SCALAR_SETS].data_ptr(), N_PAIRS)
        if i >= 2:
            lat.append(be.last_device_ms)
            for k_, v_ in be.last_msm_stage_ms.items():
                stages[k_] = stages.get(k_, 0.0) + v_ / 4
    del be_res
    single_ms = float(np.mean(lat))

    total_pairs = N_PAIRS * world * MSMS_PER_STEP
    ms_per_step = wall_ms / args.steps
    value = total_pairs / (ms_per_step * 1e-3)
    e2e_value = total_pairs / (e2e_wall_ms / e2e_steps * 1e-3)

    root_of_unity = pow(7, (R_MOD - 1) >> 28, R_MOD)

    def omega_limbs(k):
        return fr_limbs(pow(root_of_unity, 1 << (28 - k), R_MOD) * (1 << 256)).reshape(1, 4)

    # ---- strong scaling (north star): ONE 2^23 MSM on a single GPU vs sharded by point range over the N ranks -----------
    strong = None
    if not args.no_sizes:
        strong = {"log_n": STRONG_LOG_N}
        blocks = 1 << (STRONG_LOG_N - LOG_N)                  # 2^20-point blocks with seeds that do not depend on N
        mine = range(blocks * rank // world, blocks * (rank + 1) // world)

        def block_h(b): return rand_fr(N_PAIRS, SEED_POINTS + 77 + b)
        def block_s(b): return rand_fr(N_PAIRS, SEED_SCALARS + 77 + b)
        dev_sets = None; torch.cuda.empty_cache()
        h_mine = np.concatenate([block_h(b) for b in mine]); s_mine = np.concatenate([block_s(b) for b in mine])
        k_shard = STRONG_LOG_N - (world.bit_length() - 1)
        p_shard = halo2.ParamsKZG.from_parts(be, k_shard, g_lagrange=be.g1_fixed_base_mul(h_mine))
        if not args.no_tables:
            p_shard.precompute()
        d_s = torch.from_numpy(s_mine.view(np.int64)).to(dev)
        reps = 10

        def run_shard(first, steps):
            ptrs = [d_s.data_ptr()] * steps
            last["strong"] = fold(p_shard.commit_batch_dev(halo2.BASIS_G_LAGRANGE, ptrs, 1 << k_shard))
        sharded_ms = timed(lambda f, s: run_shard(f, s), reps, 3) / reps
        dots = gather_rows(mont_dot(orc, s_mine, h_mine)) if use_oracle else None
        if world == 1:
            strong.update({"ms_1gpu": sharded_ms, "pairs_per_s_1gpu": (1 << STRONG_LOG_N) / (sharded_ms * 1e-3)})
            if rank == 0 and use_oracle:
                strong["result_equals_reference"] = bool(np.array_equal(orc.g1_to_affine(last["strong"][0]).reshape(8), expected_point(orc, dots)))
        else:
            # rank 0 alone: the whole 2^23 MSM on its GPU (the other ranks wait on the CPU)
            cpu_barrier()
            if rank == 0:
                h_all = np.concatenate([block_h(b) for b in range(blocks)]); s_all = np.concatenate([block_s(b) for b in range(blocks)])
                p_all = halo2.ParamsKZG.from_parts(be, STRONG_LOG_N, g_lagrange=be.g1_fixed_base_mul(h_all))
                if not args.no_tables:
                    p_all.precompute()
                d_all = torch.from_numpy(s_all.view(np.int64)).to(dev)
                p_all.commit_batch_dev(halo2.BASIS_G_LAGRANGE, [d_all.data_ptr()] * 3, 1 << STRONG_LOG_N)
                torch.cuda.synchronize(); t0 = time.perf_counter()
                single_res = p_all.commit_batch_dev(halo2.BASIS_G_LAGRANGE, [d_all.data_ptr()] * reps, 1 << STRONG_LOG_N)
                torch.cuda.synchronize(); one_ms = (time.perf_counter() - t0) * 1e3 / reps
                strong.update({"ms_1gpu": one_ms, "ms_sharded": sharded_ms, "n_gpus": world, "speedup": one_ms / sharded_ms,
                               "sharded_equals_single_gpu": bool(np.array_equal(single_res[0], last["strong"][0])),
                               "timing": "wall per MSM over %d back-to-back MSMs (batch API); sharded: barrier-bracketed, max over ranks, incl. the all-gather and fold" % reps})
                if use_oracle:
                    strong["result_equals_reference"] = bool(np.array_equal(orc.g1_to_affine(last["strong"][0]).reshape(8), expected_point(orc, dots)))
                del p_all, d_all, h_all, s_all
            cpu_barrier()
        del p_shard, d_s
        torch.cuda.empty_cache()

    # ---- multi-GPU NTT: one process drives all N devices (six-step across devices, one all-to-all over NVLink) ----
    ntt_multi = None
    if world > 1 and not args.no_ntt:
        # rank 0 drives all N devices from one process; the other ranks wait on the CPU (a NCCL barrier would keep a
        # spinning kernel on their GPU, and kernels of two processes time-slice on one device)
        cpu_barrier()
        if rank == 0:
            import ctypes
            ntt_multi = {}
            be_all = halo2.Backend(list(range(world)))
            for k in (22, 24):
                omega = omega_limbs(k)
                src = rand_fr(1 << k, k)
                host = torch.from_numpy(src.view(np.int64).copy()).pin_memory()
                arr = host.numpy().view(np.uint64)
                nd_ms, wall = [], []
                for it in range(4):
                    arr[:] = src
                    t0 = time.perf_counter()
                    rc = be_all.lib.spb_ntt(be_all.ctx, arr.ctypes.data_as(ctypes.c_void_p), k, omega.ctypes.data_as(ctypes.c_void_p))
                    wall.append((time.perf_counter() - t0) * 1e3)
                    be_all.check(rc, "spb_ntt (multi-device)")
                    nd_ms.append(be_all.last_device_ms)
                single = be.best_fft(src, omega, k)                                  # this rank's own one-device context
                ntt_multi["2^%d" % k] = {"devices": world, "device_ms": float(np.median(nd_ms[1:])), "elems_per_s_device": (1 << k) / (float(np.median(nd_ms[1:])) * 1e-3),
                                         "e2e_ms_pinned_host": float(np.median(wall[1:])), "equals_single_gpu": bool(np.array_equal(arr, single)),
                                         "note": "device_ms = first pass + peer all-to-all + remaining passes (max over devices); e2e includes the strided H2D/D2H copies"}
            be_all.close()
        cpu_barrier()

    # ---- whole proofs on a context over all N devices (rank 0 drives): MSMs sharded by point range, quotient kernels by
    # row range, NTTs by polynomial; bytes compared with the one-device proof ------------------------------------------
    proof_multi = None
    if world > 1 and not args.no_prove:
        cpu_barrier()
        if rank == 0:
            be_multi = halo2.Backend(list(range(world)))
            try:
                proof_multi = prove_aggregation(torch, halo2, [be, be_multi], args.prove_k)
            except Exception as e:
                proof_multi = {"error": repr(e)}
            # every torch tensor that was ever used on be_multi's stream is gone by now (they were locals of prove_aggregation):
            # only then may the context -- and with it the stream torch recorded those uses on -- be destroyed
            torch.cuda.synchronize()
            be_multi.close()
        cpu_barrier()

    if rank != 0:
        be.close()
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_src = measured_peaks()
    c, W = be.msm_geometry(N_PAIRS, tables=not args.no_tables)
    # Launch duration of the dominant kernel: CUDA events on the lane stream it runs on. Inside the timed region three lanes are in
    # flight, so a launch's events also span the slices the OTHER lane's kernels got on the same SMs (two accumulate kernels
    # interleave: each takes ~2x as long and two finish per interval); the launch duration that states the GPU's rate on this
    # kernel is the one with the device to itself, measured by the same events on the 4 single-MSM calls above.
    acc_ms = stages.get("accumulate", 0.0)
    acc_ms_overlapped = stages_pipelined.get("accumulate", 0.0)
    algo_bytes = 96.0 * N_PAIRS  # SURVEY.md 8d: 32 B scalar + 64 B affine base per pair, per launch (one rank's MSM)
    achieved = algo_bytes / (acc_ms * 1e-3) / 1e9 if acc_ms > 0 else None
    # INT32 multiply-pipe view: a mixed XYZZ addition = 7 products + 2 squarings + the lazily reduced pair; in units of the
    # general product (measured peak 68 G/s) that is 9.25 (squaring 0.83, a*b-c*d 1.55: profiles/r02_field_ab.md)
    modmul_per_launch = 9.25 * (adds - 2 * (1 if not args.no_tables else W) * (1 << (c - 1)))
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath) and not args.no_tables:
        with open(tpath) as f:
            traffic = json.load(f)["msm_accumulate_kernel"]["dram_bytes_per_launch"]
    roofline = {
        "kernel": "msm_accumulate_kernel", "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
        "frac": (achieved / peaks["hbm_gbs"]) if achieved else None, "traffic": traffic, "peak_source": peak_src,
        "traffic_source": "ncu --set full capture of this kernel (profiles/ncu_traffic.json names the commit it was taken at)",
        "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": acc_ms, "kernel_ms_in_timed_region_two_lanes_interleaved": acc_ms_overlapped,
        "kernel_share_of_msm": acc_ms / single_ms if single_ms else None,
        "note": "integer-ALU bound, not HBM bound (SURVEY.md finding 6): see int32_pipe",
        "int32_pipe": {"achieved_gmodmul_per_s": modmul_per_launch / (acc_ms * 1e-3) / 1e9 if acc_ms > 0 else None,
                       "peak_gmodmul_per_s": 68.2, "peak_source": "tools/microbench.py modmul on this pool's B200 (profiles/r01_microbench.md)"},
    }
    if roofline["int32_pipe"]["achieved_gmodmul_per_s"]:
        roofline["int32_pipe"]["frac"] = roofline["int32_pipe"]["achieved_gmodmul_per_s"] / 68.2

    line = {
        "metric": "bn254_g1_msm_pairs_per_s", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u256 (8x32-bit Montgomery limbs, INT32 IMAD)",
        "data": "synthetic",
        "config": workload_config(),
        "schedule": {"window_bits": c, "windows": W, "precomputed_window_tables": not args.no_tables,
                     "pipelining": "each step is one spb_msm_batch(_dev) call: three stream lanes overlap one MSM's tail with the next one's sort/accumulate",
                     "collective": "one all_gather of the step's 16 x 96-byte partial sums (NCCL) + one C fold" if world > 1 else "none",
                     "timing": "wall clock between barrier + cuda synchronize pairs around exactly K steps, max over ranks; per-kernel times are CUDA events on the library's streams"},
        "ms_per_msm": ms_per_step / MSMS_PER_STEP, "single_msm_device_ms": single_ms, "g1_adds_per_s": adds * world * MSMS_PER_STEP / (ms_per_step * 1e-3),
        "stages_ms": stages_pipelined, "stages_ms_unpipelined": stages, "srs_setup_s": setup_s,
        "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": N_PAIRS * 32 * MSMS_PER_STEP, "d2h_bytes_per_step": 96 * MSMS_PER_STEP,
                "ms_per_step": e2e_wall_ms / e2e_steps},
        "gpu_launches": launches, "clocks": sampler.summary(), "roofline": roofline, "parity": parity,
    }
    if strong:
        line["strong_scaling"] = strong
    params = None
    torch.cuda.empty_cache()

    # ---- MSM sizes x scalar distributions (BASELINE.md 3.4 / SURVEY.md 8d), device-resident, one GPU ------------------------
    if not args.no_sizes and world == 1:
        sizes = {}
        for k in (20, 23, 24):
            n = 1 << k
            hk = np.concatenate([rand_fr(N_PAIRS, SEED_POINTS + 500 + b) for b in range(n >> LOG_N)])
            t0 = time.perf_counter()
            pk_ = halo2.ParamsKZG.from_parts(be, k, g_lagrange=be.g1_fixed_base_mul(hk))
            if not args.no_tables:
                pk_.precompute()
            row = {"setup_s": time.perf_counter() - t0, "window_bits": be.msm_geometry(n, tables=not args.no_tables)[0]}
            for name in ("uniform", "witness_like", "all_minus_one"):
                sc = np.concatenate([scalars_distribution(name, N_PAIRS, 900 + b) for b in range(n >> LOG_N)]) if name != "all_minus_one" else scalars_distribution(name, n, 0)
                d = torch.from_numpy(sc.view(np.int64)).to(dev)
                ts = []
                for _ in range(5):
                    res = pk_.commit_dev(halo2.BASIS_G_LAGRANGE, d.data_ptr(), n)
                    ts.append(be.last_device_ms)
                ms = float(np.median(ts[1:]))
                row[name] = {"device_ms": ms, "pairs_per_s": n / (ms * 1e-3), "stages_ms": {a: round(b, 3) for a, b in be.last_msm_stage_ms.items()}}
                if use_oracle and name != "uniform":          # uniform is checked by the strong-scaling block / the parity flags above
                    row[name]["result_equals_reference"] = bool(np.array_equal(orc.g1_to_affine(res).reshape(8), expected_point(orc, [mont_dot(orc, sc, hk)])))
                del d, sc
            sizes["2^%d" % k] = row
            del pk_, hk
            torch.cuda.empty_cache()
        line["msm_sizes"] = sizes

    # ---- the plain best_multiexp front door (what an unpatched call site binds): host scalars AND host bases per call vs resident bases
    if not args.no_sizes and world == 1:
        sc = host_np[0]
        walls = {"msm_raw": [], "resident_bases": []}
        res_b = halo2.ParamsKZG.from_bases(be, pts)
        for it in range(5):
            t0 = time.perf_counter(); r1 = be.best_multiexp(sc, pts); walls["msm_raw"].append(time.perf_counter() - t0)
            t0 = time.perf_counter(); r2 = res_b.multiexp(sc); walls["resident_bases"].append(time.perf_counter() - t0)
        line["best_multiexp_front_door"] = {
            "spb_msm_raw_ms": float(np.median(walls["msm_raw"][1:])) * 1e3, "spb_bases_upload_then_spb_msm_ms": float(np.median(walls["resident_bases"][1:])) * 1e3,
            "same_point": bool(np.array_equal(r1, r2)),
            "what": "wall ms of ONE 2^20 best_multiexp through the C ABI from pinned host scalars: spb_msm_raw re-uploads the 64 MiB of bases and runs without "
                    "window tables (c = 16, 16 bucket sets); against bases uploaded once (spb_bases_upload, no tables) only the 32 MiB of scalars move"}
        del res_b

    # ---- NTT throughput (the other half of BASELINE.json's metric), device-resident, rank 0 ------------------
    if not args.no_ntt:
        ntt = {}
        for k in ((20, 22, 23, 25) if world == 1 else (20, 22)):
            omega = omega_limbs(k)
            t = torch.from_numpy(rand_fr(1 << k, k).view(np.int64)).to(dev)
            times = []
            for _ in range(8):
                be.best_fft_dev(t.data_ptr(), omega, k)
                times.append(be.last_device_ms)
            ms = float(np.median(times[3:]))
            ntt["2^%d" % k] = {"ms": ms, "elems_per_s": (1 << k) / (ms * 1e-3), "algo_GBps": (1 << k) * 64 / (ms * 1e-3) / 1e9,
                               "hbm_frac": (1 << k) * 64 / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}
            del t
        if ntt_multi:
            ntt["multi_gpu"] = ntt_multi
        line["ntt"] = ntt
        torch.cuda.empty_cache()

    # ---- HBM-class kernels of evaluate_h: bytes = (#polynomials read + 1) x 32 B x E (SURVEY.md 8d) ---------------------------
    if not args.no_sizes and world == 1:
        try:
            line["roofline"]["quotient_kernels"] = quotient_roofline(torch, be, dev, peaks["hbm_gbs"])
        except Exception as e:
            line["roofline"]["quotient_kernels"] = {"error": repr(e)}
        torch.cuda.empty_cache()

    # ---- real proofs: keygen + create_proof of the two circuit shapes of a sync-step-compressed proof, every polynomial
    # resident in HBM (spectre_b200/plonk.py; the aggregation shape is the one the reference's verifier contract accepts) ----
    if not args.no_prove and world == 1:
        try:
            line["proof"] = prove_both(torch, halo2, be, args)
        except Exception as e:   # the MSM line must survive a failure of this optional section
            line["proof"] = {"error": repr(e)}
    if proof_multi is not None:
        line["proof"] = {"aggregation_shape_multi_gpu": proof_multi}

    # ---- CPU baseline (oracle port of best_multiexp) on this box's cores, bounded sample ----------------------
    if use_oracle and world == 1:
        threads = os.cpu_count() or 1
        sc = host_np[0]
        ts, cpu_res = cpu_msm_samples(orc, sc, pts, threads, 5)
        p1 = halo2.ParamsKZG.from_parts(be, LOG_N, g_lagrange=pts)
        gpu_res = p1.commit_lagrange(sc)
        same = bool(np.array_equal(orc.g1_to_affine(cpu_res), orc.g1_to_affine(gpu_res)))
        med = float(np.median(ts))
        line["cpu_baseline"] = {"value": N_PAIRS / med, "unit": "pairs/s", "cores": threads, "kind": "port",
                                "sample": "full 2^20-pair MSMs (same scalars and bases as a GPU step's MSM), one full-size warm-up then median of 5; C port of halo2 best_multiexp",
                                "seconds_min_median_max": [float(min(ts)), med, float(max(ts))], "result_equals_gpu": same}
        if not same:
            line["error"] = "GPU result differs from the CPU oracle"
    bad = [k_ for k_, v_ in parity.items() if v_ is False]
    if strong and (strong.get("result_equals_reference") is False or strong.get("sharded_equals_single_gpu") is False):
        bad.append("strong_scaling")
    if bad:
        line["error"] = "parity failure: " + ", ".join(bad)
    print(json.dumps(line), flush=True)
    be.close()
    if world > 1:
        dist.destroy_process_group()


# ---- sections ---------------------------------------------------------------------------------------------------------------
def quotient_roofline(torch, be, dev, hbm_gbs):
    """permutation_constraints / lookup_constraints / graph_evaluate on E = 2^22 extended rows with the sync-step shape's
    column counts: device ms (CUDA events inside the library) against the algorithmic bytes of SURVEY.md 8d."""
    from spectre_b200 import circuits, plonk
    E_LOG, K = 22, 20
    E = 1 << E_LOG
    rot_scale = 1 << (E_LOG - K)
    g = torch.Generator(device=dev); g.manual_seed(11)

    def col():
        t = torch.randint(-(1 << 63), (1 << 63) - 1, (E, 4), dtype=torch.int64, device=dev, generator=g)
        t[:, 3] &= (1 << 60) - 1
        return t
    cs = circuits.halo2lib_shape()
    rnd = lambda s: rand_fr(1, s).reshape(4)
    out = {}
    # permutation: 21 columns in 11 sets of 2
    n_cols, chunk = len(cs.permutation), cs.chunk_len()
    n_sets = -(-n_cols // chunk)
    z = [col() for _ in range(n_sets)]; cv = [col() for _ in range(n_cols)]; sg = [col() for _ in range(n_cols)]
    l0, ll, la, values = col(), col(), col(), col()
    wext = fr_limbs(pow(pow(7, (R_MOD - 1) >> 28, R_MOD), 1 << (28 - E_LOG), R_MOD) * (1 << 256))
    torch.cuda.synchronize()
    ts = []
    for _ in range(4):
        be.permutation_constraints_dev(values.data_ptr(), E, rot_scale, -6, chunk, [t.data_ptr() for t in z], [t.data_ptr() for t in cv], [t.data_ptr() for t in sg],
                                       l0.data_ptr(), ll.data_ptr(), la.data_ptr(), rnd(1), rnd(2), rnd(3), wext)
        ts.append(be.last_device_ms)
    ms = float(np.median(ts[1:]))
    reads = 3 * n_sets - 1 + 2 * n_cols + 3 + 1   # z at idx / next (/ last for all but one set), value + sigma per column, l0/l_last/l_active, values
    byts = (reads + 1) * 32.0 * E
    out["permutation_constraints_kernel"] = {"rows": E, "columns": n_cols, "sets": n_sets, "device_ms": ms, "algorithmic_bytes": byts,
                                             "achieved_GBps": byts / (ms * 1e-3) / 1e9, "hbm_frac": byts / (ms * 1e-3) / 1e9 / hbm_gbs}
    del z, sg
    # lookup constraints of one lookup
    pr, pi, pt, tv = col(), col(), col(), col()
    torch.cuda.synchronize()
    ts = []
    for _ in range(4):
        be.lookup_constraints_dev(values.data_ptr(), E, rot_scale, pr.data_ptr(), pi.data_ptr(), pt.data_ptr(), tv.data_ptr(), l0.data_ptr(), ll.data_ptr(), la.data_ptr(),
                                  rnd(1), rnd(2), rnd(3))
        ts.append(be.last_device_ms)
    ms = float(np.median(ts[1:]))
    byts = (10 + 1) * 32.0 * E   # product (idx, next), permuted input (idx, prev), permuted table, table value, l0, l_last, l_active, values
    out["lookup_constraints_kernel"] = {"rows": E, "device_ms": ms, "algorithmic_bytes": byts, "achieved_GBps": byts / (ms * 1e-3) / 1e9, "hbm_frac": byts / (ms * 1e-3) / 1e9 / hbm_gbs}
    del pr, pi, pt, tv
    # custom gates: 15 basic gates over 15 advice columns (4 rotations each) and 15 selectors
    p = cs.gates_program()
    G = 15
    fixed = cv[:cs.num_fixed] if len(cv) >= cs.num_fixed else cv + [col() for _ in range(cs.num_fixed - len(cv))]
    advice = [col() for _ in range(cs.num_advice)]
    torch.cuda.synchronize()
    ts = []
    for _ in range(4):
        be.graph_evaluate_dev(p["prog"], p["ncalc"], p["ncalc"], p["constants"], p["rotations"], [t.data_ptr() for t in fixed], [t.data_ptr() for t in advice], [l0.data_ptr()],
                              np.zeros((1, 4), np.uint64), rnd(1), rnd(2), rnd(3), rnd(4), values.data_ptr(), E, rot_scale)
        ts.append(be.last_device_ms)
    ms = float(np.median(ts[1:]))
    byts = (G * 4 + G + 1 + 1) * 32.0 * E   # 4 rotations of each gate column + its selector, values read + written
    out["graph_evaluate_kernel"] = {"rows": E, "gates": G, "calculations": int(p["ncalc"]), "device_ms": ms, "algorithmic_bytes": byts,
                                    "achieved_GBps": byts / (ms * 1e-3) / 1e9, "hbm_frac": byts / (ms * 1e-3) / 1e9 / hbm_gbs,
                                    "note": "interpreter over the flat GraphEvaluator program; rotated reads of one column hit L2"}
    return out


class Draw:
    """create_proof's rng: blinding rows from a host stream; the vanishing argument's random polynomial from the library's
    device ChaCha20 stream when `device_poly` (spb_fr_random_chacha_dev: it never crosses PCIe), so two engines -- and the
    compiled driver -- given the same seeds draw the same values."""

    def __init__(self, torch, seed, device_poly=True):
        self.g, self.seed = np.random.default_rng(seed), seed
        self.chacha_seed = (0xb200 + seed).to_bytes(32, "little")
        if device_poly:
            self.device_rows = lambda E, count: E.random_chacha(self.chacha_seed, 0, count)

    def __call__(self, count):
        a = self.g.integers(0, 1 << 63, size=(count, 4), dtype=np.uint64); a[:, 3] &= np.uint64((1 << 60) - 1)
        return a


def make_case(torch, name, k, pin=True):
    from spectre_b200 import circuits
    inst = list(range(1, 15))
    t0 = time.perf_counter()
    if name == "aggregation_shape":
        cs = circuits.aggregation_shape()
        fixed_cols, adv, copies = circuits.aggregation_witness(cs, k, inst, min(19, k - 2), 2000, seed=1, dense=True)
        adv_cols = [adv]
    else:
        cs = circuits.halo2lib_shape()
        fixed_cols, adv_cols, copies = circuits.halo2lib_witness(cs, k, inst, min(16, k - 2), 500, seed=1)
    t_witness = time.perf_counter() - t0
    pinned = None
    if pin:   # witness buffers registered once (a prover keeps its synthesis buffers pinned): advice columns go up as plain DMA
        pinned = [torch.from_numpy(np.ascontiguousarray(c, dtype=np.uint64).view(np.int64)).pin_memory() for c in adv_cols]
    return cs, inst, fixed_cols, adv_cols, pinned, copies, t_witness


def prove_both(torch, halo2, be, args):
    from spectre_b200 import plonk
    from spectre_b200.transcript import EvmTranscriptWrite
    from tools import cpp_driver
    secret = plonk.fr_mont(0x5eed7a75)                        # any SRS secret: timings do not depend on it
    proofs = {}
    exe, exe_dir = None, tempfile.TemporaryDirectory()        # the compiled driver is built outside the tree, which may be read-only
    for name, k in (("sync_step_shape", args.prove_k_step), ("aggregation_shape", args.prove_k)):
        t0 = time.perf_counter()
        srs = halo2.ParamsKZG.setup(be, k, secret).precompute()
        torch.cuda.synchronize(); t_srs = time.perf_counter() - t0
        cs, inst, fixed_cols, adv_cols, pinned, copies, t_witness = make_case(torch, name, k)
        E = plonk.DeviceEngine(be, srs, k, cs.degree())
        t0 = time.perf_counter()
        pkey = plonk.keygen(E, cs, k, fixed_cols, copies, vk_digest=BENCH_VK_DIGEST)
        E.sync(); t_keygen = time.perf_counter() - t0
        runs = []
        for rep in range(3):                                  # the later passes are the warm ones (lazy kernel loading, allocator)
            stages = {}
            t0 = time.perf_counter()
            proof = plonk.create_proof(E, pkey, [inst], pinned, Draw(torch, 7), EvmTranscriptWrite(pkey.vk_digest), stages)
            E.sync(); runs.append((time.perf_counter() - t0, stages))
        best = min(runs[1:], key=lambda r: r[0])
        row = {"k": k, "advice_columns": cs.num_advice, "lookups": len(cs.lookups), "permutation_columns": len(cs.permutation), "degree": cs.degree(),
               "create_proof_s": best[0], "first_create_proof_s": runs[0][0], "keygen_s": t_keygen, "srs_setup_and_tables_s": t_srs,
               "synthetic_witness_python_s": t_witness, "proof_bytes": len(proof), "stages_s": {a: round(b, 4) for a, b in best[1].items()}}
        # the compiled driver (include/spectre_b200_prover.hpp) on the same circuit, witness and RNG stream: host draws only
        if not args.no_cpp:
            try:
                host = Draw(torch, 9, device_poly=False)
                rec = cpp_driver.RecordingRng(host, chacha_poly=host.chacha_seed)
                t0 = time.perf_counter()
                ref_proof = plonk.create_proof(E, pkey, [inst], pinned, rec, EvmTranscriptWrite(pkey.vk_digest))
                E.sync(); t_py_host_rng = time.perf_counter() - t0
                del E, pkey, srs
                torch.cuda.empty_cache()
                exe = exe or cpp_driver.build_main_against_the_real_library(out_dir=exe_dir.name)
                with tempfile.TemporaryDirectory() as d:
                    head = "shape aggregation" if name == "aggregation_shape" else "shape halo2lib 15 2"
                    cpp_driver.dump_case(d, head, k, BENCH_VK_DIGEST, inst, copies, rec.counts, fixed_cols, adv_cols, rec.rows, secret, chacha_poly=host.chacha_seed)
                    rc, log, cproof, ms, kg = cpp_driver.run(exe, d, repeat=3, tables=True)
                row["compiled_driver"] = {"returncode": rc, "create_proof_s": (min(ms[1:]) / 1e3) if len(ms) > 1 else None, "first_create_proof_s": (ms[0] / 1e3) if ms else None,
                                          "keygen_s": kg / 1e3 if kg else None, "python_driver_same_rng_s": t_py_host_rng,
                                          "proof_equals_python_driver": bool(cproof is not None and cproof == ref_proof),
                                          "note": "C++17 header-only driver over the same C ABI, CudaMemory on the context stream; same host blinding rows and the same "
                                                  "device ChaCha20 random polynomial (spb_fr_random_chacha_dev) as the Python driver it is compared with"}
                if rc != 0:
                    row["compiled_driver"]["log"] = log[-400:]
            except Exception as e:
                row["compiled_driver"] = {"error": repr(e)}
        proofs[name] = row
        E = pkey = srs = None
        del fixed_cols, adv_cols, pinned
        torch.cuda.empty_cache()
    exe_dir.cleanup()
    proofs["sync_step_compressed_shape_total_s"] = proofs["sync_step_shape"]["create_proof_s"] + proofs["aggregation_shape"]["create_proof_s"]
    proofs["what"] = ("create_proof wall seconds, best warm pass of 2: pinned witness H2D, blinding, every commitment, evaluate_h, evaluations, SHPLONK, Keccak transcript; "
                      "host driver in Python over the C ABI (no torch synchronisation: everything is ordered on the library's stream); synthetic witnesses with full "
                      "columns; constraint-system shapes per SURVEY.md section 8 (aggregation: read off the committed verifier contract; sync-step: estimate from the pinning JSON)")
    return proofs


def prove_aggregation(torch, halo2, backends, k):
    """the aggregation-shaped proof on every backend of the list (first = one device, second = the N-device context), same witness
    and RNG streams: wall time per backend and byte equality"""
    from spectre_b200 import plonk
    from spectre_b200.transcript import EvmTranscriptWrite
    secret = plonk.fr_mont(0x5eed7a75)
    cs, inst, fixed_cols, adv_cols, pinned, copies, _ = make_case(torch, "aggregation_shape", k)
    out, proofs = {"k": k}, []
    for be_ in backends:
        nd = len(be_.devices)
        srs = halo2.ParamsKZG.setup(be_, k, secret).precompute()
        E = plonk.DeviceEngine(be_, srs, k, cs.degree())
        t0 = time.perf_counter()
        pkey = plonk.keygen(E, cs, k, fixed_cols, copies, vk_digest=BENCH_VK_DIGEST)
        E.sync(); t_keygen = time.perf_counter() - t0
        runs = []
        for rep in range(3):
            stages = {}
            t0 = time.perf_counter()
            proof = plonk.create_proof(E, pkey, [inst], pinned, Draw(torch, 7), EvmTranscriptWrite(pkey.vk_digest), stages)
            E.sync(); runs.append((time.perf_counter() - t0, stages))
        best = min(runs[1:], key=lambda r: r[0])
        out["devices_%d" % nd] = {"create_proof_s": best[0], "keygen_s": t_keygen, "stages_s": {a: round(b, 4) for a, b in best[1].items()}}
        proofs.append(proof)
        del E, pkey, srs
        torch.cuda.empty_cache()
    out["proof_equals_single_gpu"] = bool(proofs[0] == proofs[-1])
    out["speedup"] = out["devices_1"]["create_proof_s"] / out["devices_%d" % len(backends[-1].devices)]["create_proof_s"] if len(backends) > 1 else None
    out["what"] = ("one context over all N devices driven by rank 0: every commitment is an MSM sharded by point range (scalar ranges peer-copied), the quotient kernels "
                   "run on row ranges and the NTTs on whole polynomials spread over the devices, all reading the first device's HBM through NVLink peer access")
    return out


if __name__ == "__main__":
    main()
