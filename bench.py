#!/usr/bin/env python3
"""
bench.py -- headline benchmark of the hot path (BASELINE.json: "BN254 MSM points/s & NTT elems/s").

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the CPU restatement of the reference's path (oracle)
    python bench.py ... --dump-outputs DIR                   # also write the outputs of the last timed steps to DIR/*.npy

With the same arguments the inputs are the same from run to run (seeded generators on the device), so the files of
--dump-outputs from two builds can be compared array for array: msm, msm_witness, msm_e2e, msm_registered_pinned (the affine
result point of each MSM leg, x and y in 32-bit limbs; the identity is all zero) and ntt, ntt_e2e (the rows ntt_rows of the
device-resident and of the host-array NTT output, Montgomery form in 32-bit limbs).

A *step* is one pass of the hot path over one batch of synthetic input: one BN254 G1 MSM over
2^k points per GPU (k = 24 by default: BASELINE.json configs[3], the synthetic sweep; the other
configs need the Rust prover and are parity-test cases).  With N > 1 the MSM is sharded by point
range -- every rank owns 2^k points (weak scaling), computes its partial sum, the 224-byte partials
are all-gathered over NCCL and folded on the device.  After the MSM region the same K/W protocol
times the Fr NTT at 2^k per GPU; its numbers ride along in the "ntt" object of the same JSON line.

`value`  : whole-job MSM throughput, inputs resident in HBM, CUDA-event timed, max over ranks.
`e2e`    : the same metric through the reference-facing drop-in best_multiexp(coeffs, bases) = h2b_msm_bn254_g1 with
           PAGEABLE host arrays (what Rust Vecs are): every step uploads the scalars, re-verifies the digest of the
           caller's bases array against the resident copy (implicit SRS cache), runs, downloads the 96-byte result.
           `e2e_registered_pinned` is the friendlier variant (pinned scalars, explicitly registered SRS) for comparison.
`verified`: after the timed loops the device-timed result, the e2e result and the O(n) checksum [sum s_i z_i] G
           (field arithmetic only: h2b_msm_checksum_dev + one big-int scalar multiplication) must agree -- at every N.
`roofline`: dominant kernel (msm_accumulate_kernel) against the measured integer-pipe peak (SURVEY.md 8d).
`cpu_baseline`: the C++ restatement of halo2_proofs' best_multiexp/best_fft (oracle/) on the host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

IMADS_PER_POINT = 21760          # SURVEY.md 8(d): 16 windows x 10 Fq-muls x 136 MACs
MACS_PER_FR_MUL = 136


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--k", type=int, default=24, help="log2 of the points / elements per GPU")
    ap.add_argument("--scalars", default="uniform", choices=["uniform", "witness"])
    ap.add_argument("--sweep", action="store_true", help="also print a k=16..26 sweep (extra JSON lines on stderr)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-widened", action="store_true", help="skip the evaluate_h / SRS extras (SURVEY.md 8f) that ride along at N = 1")
    ap.add_argument("--plain", action="store_true", help="do not use the precomputed window tables of the registered SRS")
    ap.add_argument("--no-inprocess", action="store_true", help="N > 1: skip the in-process h2b_init(N) parity + strong-scaling leg (tools/multi_gpu_inprocess.py)")
    ap.add_argument("--strong-k", type=int, nargs="*", default=[24, 26], help="total sizes 2^k of the strong-scaling leg at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step of each leg returned "
                    "as DIR/<name>.npy (float64 32-bit limbs; the NTT outputs as a fixed, seeded sample of rows), rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def config_for(args, n_gpus):
    return {
        "workload": "synthetic BN254 G1 MSM (+ Fr NTT) at k=%d per GPU (BASELINE.json configs[3])" % args.k,
        "k": args.k,
        "points_per_gpu": 1 << args.k,
        "scalars": args.scalars,
        "parallelism": "point-range shard x%d, partial sums all-gathered + folded" % n_gpus if n_gpus > 1 else "single GPU",
        "l2": "inputs (%.1f GB per GPU) exceed the 126 MB L2; no flush needed" % ((96 << args.k) / 1e9),
    }


# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.25 and len(r) >= 9] or [r for (_, r) in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [float(r[1]) for r in rows]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][2]), "power_w_max": max(float(r[3]) for r in rows),
                "samples": len(rows), "reasons": sorted(reasons)}


DUMP_NTT_ROWS = 1 << 16        # --dump-outputs: rows of each 2^k NTT output written (4 MiB per array)
DUMP_SEED = 0xB2D0


def words_to_limbs(words):
    """(m, 4) u64 field elements -> (m, 8) float64 of their 32-bit halves, least significant first (exact)"""
    import numpy as np
    return np.ascontiguousarray(words, dtype=np.uint64).view(np.uint32).reshape(-1, 8).astype(np.float64)


def point_to_limbs(p):
    """affine (x, y) as canonical ints, None for the identity -> (2, 8) float64 of 32-bit limbs, least significant first.
    The identity is written as (0, 0), which is not on the curve."""
    import numpy as np
    x, y = p if p is not None else (0, 0)
    return np.array([[(c >> (32 * i)) & 0xFFFFFFFF for i in range(8)] for c in (x, y)], dtype=np.float64)


def omega_words(k):
    from halo2_scaffold_b200.domain import FR_MODULUS, FR_ROOT_OF_UNITY, FR_S, fr_to_words
    w = FR_ROOT_OF_UNITY
    for _ in range(k, FR_S):
        w = w * w % FR_MODULUS
    return fr_to_words(w)


# --------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own algorithm for this path on the host cores: oracle/h2_oracle.cpp, the C++ restatement of
    halo2_proofs v2023_02_02 best_multiexp / best_fft (the Rust original is un-vendored and there is no cargo here,
    so oracle/_ref cannot exist).  Each step is a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_c as oc
    oc.build()
    cores = oc.hardware_threads()
    ks = min(args.k, 22)          # the same bounded sample as the repo arm's own cpu_baseline leg
    n = 1 << ks
    scal = oc.random_fr(0xB2000000 + ks, n)
    pts = oc.gen_points(0xB2001000 + ks, n)
    for _ in range(args.warmup):
        oc.best_multiexp(scal, pts, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oc.best_multiexp(scal, pts, cores)
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    w = omega_words(ks)
    oc.best_fft(scal, w, ks, cores)
    t1 = time.perf_counter()
    for _ in range(args.steps):
        oc.best_fft(scal, w, ks, cores)
    ntt_value = n * args.steps / (time.perf_counter() - t1)
    sample = "best_multiexp over 2^%d of the 2^%d points per step (uniform scalars), %d threads" % (ks, args.k, cores)
    line = {
        "impl": "reference", "metric": "bn254_g1_msm_points_per_s", "value": value, "unit": "points/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32 limbs (254-bit modular integers)", "data": "synthetic", "config": config_for(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": cores, "kind": "port", "sample": sample,
                         "ntt_value": ntt_value, "ntt_unit": "elements/s", "ntt_sample": "best_fft at 2^%d" % ks},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "C++ restatement of halo2_proofs v2023_02_02 (oracle/h2_oracle.cpp); the Rust reference cannot be built here",
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import halo2_scaffold_b200 as h2
    from halo2_scaffold_b200 import verify as V

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this framework has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # N ranks share one host: give each rank its share of the cores for the pinned-staging and digest threads of the host-pointer
        # drop-in instead of 8 + 8 threads per rank (the e2e leg is host-memory bound at N = 8: 8 x (1 GiB digest + 0.5 GiB staging) per step)
        share = max(2, min(8, (os.cpu_count() or 16) // world))
        os.environ.setdefault("H2B_STAGE_THREADS", str(share))
        os.environ.setdefault("H2B_DIGEST_THREADS", str(share))
    L = h2.load()
    L.init_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        host_group = dist.new_group(backend="gloo")      # host-side waits that must not spin a kernel on the waiting GPUs

    k, n = args.k, 1 << args.k
    K, W = args.steps, args.warmup
    st = torch.cuda.current_stream().cuda_stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- synthetic inputs, generated on the device (each rank owns its own point range) ------------
    d_scal = torch.empty(n * 4, dtype=torch.int64, device=dev)
    d_base = torch.empty(n * 8, dtype=torch.int64, device=dev)
    d_block = torch.empty(28, dtype=torch.int64, device=dev)
    d_blocks = torch.empty(28 * world, dtype=torch.int64, device=dev)
    d_out = torch.empty(12, dtype=torch.int64, device=dev)
    d_chk = torch.empty(4, dtype=torch.int64, device=dev)
    d_chks = torch.empty(4 * world, dtype=torch.int64, device=dev)
    d_jac = torch.empty(12, dtype=torch.int64, device=dev)
    d_jacs = torch.empty(12 * world, dtype=torch.int64, device=dev)
    kind = 0 if args.scalars == "uniform" else 1
    seed_p = 0xB2001000 + k + 1000 * rank
    L.gen_scalars_dev(0, 0xB2000000 + k + 1000 * rank, n, kind, d_scal.data_ptr(), st)
    L.gen_points_dev(0, seed_p, n, d_base.data_ptr(), st)
    torch.cuda.synchronize()

    def expected_point(d_scalars):
        """[sum over all ranks of sum_i s_i z_i] G: the O(n) checksum of the (folded) MSM, field arithmetic only"""
        L.msm_checksum_dev(0, d_scalars.data_ptr(), seed_p, n, d_chk.data_ptr(), stream=st)
        if world > 1:
            dist.all_gather_into_tensor(d_chks, d_chk)
            cs = d_chks.cpu().numpy().view(np.uint64).reshape(world, 4)
        else:
            cs = d_chk.cpu().numpy().view(np.uint64).reshape(1, 4)
        return V.scalar_mul_generator(sum(V.words_to_int(c) for c in cs) % V.FR_MODULUS)

    # the SRS vector is registered once (ParamsKZG holds `g` / `g_lagrange` for the life of the prover): upload +
    # window tables, outside every timed region; its cost is reported as `srs_registration_ms`
    t0 = time.perf_counter()
    h_base = d_base.cpu()
    handle = L.register_bases(h_base.numpy().view(np.uint64))
    del h_base
    torch.cuda.synchronize()
    reg_ms = (time.perf_counter() - t0) * 1e3
    set_info = L.base_set_info(handle)
    if args.plain:
        del_handle, handle = handle, None
        L.unregister_bases(del_handle)

    def msm_step():
        if handle is not None:
            L.msm_dev_registered(0, d_scal.data_ptr(), handle, 0, n, d_block.data_ptr(), st)
        else:
            L.msm_dev_partial(0, d_scal.data_ptr(), d_base.data_ptr(), n, d_block.data_ptr(), st)
        if world > 1:
            dist.all_gather_into_tensor(d_blocks, d_block)
            L.msm_fold_partials_dev(0, d_blocks.data_ptr(), world, d_out.data_ptr(), st)
        else:
            L.msm_fold_partials_dev(0, d_block.data_ptr(), 1, d_out.data_ptr(), st)

    # integer-pipe peak, measured on this GPU right now (the MSM roofline denominator)
    imad_ms, imad_ops = L.imad_bench(0, 4096)
    imad_peak = imad_ops / imad_ms * 1e3          # IMAD/s
    mul_ms, mul_ops = L.imad_bench(2, 4096)
    fqmul_peak = mul_ops / mul_ms * 1e3

    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- MSM, device resident ------------------------------------------------------------------------------
    for _ in range(W):
        msm_step()
    barrier()
    L.profile_enable(True)
    launches0 = L.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record()
    for _ in range(K):
        msm_step()
    e1.record()
    barrier()
    t_wall1 = time.time()
    msm_ms = max_over_ranks(e0.elapsed_time(e1))
    launches = L.launch_count() - launches0
    prof = L.profile_read()
    L.profile_enable(False)
    # bucket accumulation = the pair pre-reduction passes (tag 10, batched affine additions) + the XYZZ accumulation (tag 5): together
    # they perform the per-point additions the algorithmic IMAD count stands for
    pair_total = sum(ms for (tag, ms) in prof if tag == 10)
    acc_ms = [ms for (tag, ms) in prof if tag == 5]
    if acc_ms:
        acc_ms = [ms + pair_total / len(acc_ms) for ms in acc_ms]
    phase_ms = {}
    for tag, ms in prof:
        phase_ms[tag] = phase_ms.get(tag, 0.0) + ms / K
    msm_value = world * n * K / (msm_ms / 1e3)
    result_host = d_out.cpu().numpy().view(np.uint64)
    expect = expected_point(d_scal)
    result_affine = V.jacobian_words_to_affine(result_host)
    checks = {"device_resident_equals_checksum": result_affine == expect}
    outputs = {"msm": point_to_limbs(result_affine)}          # what the last timed step of each leg returned (--dump-outputs)

    # ---- the same MSM over a witness-like column (SURVEY.md 8d: 50 % zero, 20 % one, 20 % < 2^19, 10 % r - small) ---------
    witness = None
    if args.scalars == "uniform":
        d_wit = torch.empty(n * 4, dtype=torch.int64, device=dev)
        L.gen_scalars_dev(0, 0xB2000000 + k + 1000 * rank + 77, n, 1, d_wit.data_ptr(), st)

        def wit_step():
            if handle is not None:
                L.msm_dev_registered(0, d_wit.data_ptr(), handle, 0, n, d_block.data_ptr(), st)
            else:
                L.msm_dev_partial(0, d_wit.data_ptr(), d_base.data_ptr(), n, d_block.data_ptr(), st)
        for _ in range(W):
            wit_step()
        barrier()
        e0.record()
        for _ in range(K):
            wit_step()
        e1.record()
        barrier()
        wit_ms = max_over_ranks(e0.elapsed_time(e1))
        if world > 1:
            dist.all_gather_into_tensor(d_blocks, d_block)
            L.msm_fold_partials_dev(0, d_blocks.data_ptr(), world, d_out.data_ptr(), st)
        else:
            L.msm_fold_partials_dev(0, d_block.data_ptr(), 1, d_out.data_ptr(), st)
        wit_affine = V.jacobian_words_to_affine(d_out.cpu().numpy().view(np.uint64))
        wit_ok = wit_affine == expected_point(d_wit)
        checks["witness_like_equals_checksum"] = wit_ok
        outputs["msm_witness"] = point_to_limbs(wit_affine)
        witness = {"value": world * n * K / (wit_ms / 1e3), "unit": "points/s", "ms_per_step": wit_ms / K,
                   "scalars": "50% zero, 20% one, 20% uniform < 2^19, 10% r - small", "verified": bool(wit_ok)}
        del d_wit

    # ---- MSM, end to end through the host-pointer drop-in ---------------------------------------------------
    # (a) the real drop-in: best_multiexp(coeffs, bases) = h2b_msm_bn254_g1 with PAGEABLE arrays, as a Rust prover holds them.
    #     Every call re-verifies the caller's bases array against the resident copy (implicit SRS cache); warm-up = upload,
    #     window tables, reuse.  With N ranks the N results are gathered and added on the host (north_star: "combined ... on the host").
    scal_np = d_scal.cpu().numpy().view(np.uint64).reshape(n, 4)      # pageable
    base_np = d_base.cpu().numpy().view(np.uint64).reshape(n, 8)      # pageable

    def e2e_step():
        r = L.msm(scal_np, base_np)
        if world == 1:
            return r
        d_jac.copy_(torch.from_numpy(r.view(np.int64)))
        dist.all_gather_into_tensor(d_jacs, d_jac)
        acc = None
        for j in d_jacs.cpu().numpy().view(np.uint64).reshape(world, 12):
            acc = V.affine_add(acc, V.jacobian_words_to_affine(j))
        return acc
    for _ in range(max(3, W)):
        r = e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        r = e2e_step()
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * n * K / e2e_s
    e2e_affine = V.jacobian_words_to_affine(r) if world == 1 else r
    checks["e2e_equals_checksum"] = e2e_affine == expect
    outputs["msm_e2e"] = point_to_limbs(e2e_affine)
    cache_stats = L.implicit_cache_stats()
    del base_np
    # (b) the friendlier variant of round 1: pinned scalars, explicitly registered SRS (what a patched ParamsKZG::commit does)
    h_scal = torch.empty(n * 4, dtype=torch.int64).pin_memory()
    h_scal.copy_(d_scal)
    if handle is None:
        L.set_msm_precomp(-1)
        h_base = d_base.cpu()
        handle = L.register_bases(h_base.numpy().view(np.uint64))       # plain mode: points only
        del h_base
    pin_np = h_scal.numpy().view(np.uint64).reshape(n, 4)
    for _ in range(2):
        r = L.msm_registered(pin_np, handle)
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        r = L.msm_registered(pin_np, handle)
    barrier()
    e2e_pinned_value = world * n * K / max_over_ranks(time.perf_counter() - t0)
    pinned_affine = V.jacobian_words_to_affine(r)            # at N > 1: this rank's share of the points
    if world == 1:
        checks["e2e_registered_pinned_equals_checksum"] = pinned_affine == expect
    outputs["msm_registered_pinned"] = point_to_limbs(pinned_affine)
    L.unregister_bases(handle)
    del scal_np

    # ---- NTT, device resident + end to end --------------------------------------------------------------------
    w_words = omega_words(k)
    d_ntt = d_scal          # reuse: 2^k Fr elements
    for _ in range(W):
        L.ntt_dev(0, d_ntt.data_ptr(), w_words, k, st)
    barrier()
    L.profile_enable(True)
    e0.record()
    for _ in range(K):
        L.ntt_dev(0, d_ntt.data_ptr(), w_words, k, st)
    e1.record()
    barrier()
    ntt_ms = max_over_ranks(e0.elapsed_time(e1))
    nprof = L.profile_read()
    L.profile_enable(False)
    pass_ms = [ms for (tag, ms) in nprof if tag >= 16]
    ntt_value = world * n * K / (ntt_ms / 1e3)
    # one more (untimed) step on the state the timed loop left behind, checked at 4 spot indices: out[i] = sum_j in[j] w^(i j),
    # evaluated by Horner on the device (h2b_fr_eval_polynomial_dev shares no code with the NTT passes)
    d_in = d_ntt.clone()
    L.ntt_dev(0, d_ntt.data_ptr(), w_words, k, st)
    torch.cuda.synchronize()
    from halo2_scaffold_b200.domain import FR_MODULUS, fr_to_words
    w_int = sum(int(w_words[i]) << (64 * i) for i in range(4)) * pow(1 << 256, -1, FR_MODULUS) % FR_MODULUS
    d_ev = torch.empty(4, dtype=torch.int64, device=dev)
    ntt_ok = True
    for idx in (0, 1, n // 2 + 3, n - 1):
        L.check(L.L.h2b_fr_eval_polynomial_dev(0, d_in.data_ptr(), n, fr_to_words(pow(w_int, idx, FR_MODULUS)).ctypes.data, d_ev.data_ptr(), st))
        torch.cuda.synchronize()
        ntt_ok = ntt_ok and bool((d_ev.cpu() == d_ntt[4 * idx: 4 * idx + 4].cpu()).all())
    checks["ntt_spot_values"] = ntt_ok
    ntt_rows = np.sort(np.random.default_rng(DUMP_SEED).choice(n, size=min(n, DUMP_NTT_ROWS), replace=False))
    outputs["ntt_rows"] = ntt_rows.astype(np.float64)
    outputs["ntt"] = words_to_limbs(d_in.view(n, 4)[torch.from_numpy(ntt_rows).to(dev)].cpu().numpy().view(np.uint64))
    del d_in
    a_np = np.empty((n, 4), dtype=np.uint64)                     # pageable, like the Vec<Fr> best_fft receives
    a_np[:] = h_scal.numpy().view(np.uint64).reshape(n, 4)
    L.ntt(a_np, w_words, k)
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        L.ntt(a_np, w_words, k)
    barrier()
    ntt_e2e_s = max_over_ranks(time.perf_counter() - t0)
    outputs["ntt_e2e"] = words_to_limbs(a_np[ntt_rows])
    sampler.stop()
    clocks = sampler.summary(t_wall0, t_wall1)

    # ---- CPU baseline: the oracle on the host cores, bounded sample (rank 0, N = 1 only) ------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle_c as oc
        oc.build()
        cores = oc.hardware_threads()
        ks = min(k, 22)
        m = 1 << ks
        s_s = d_scal[: 4 * m].cpu().numpy().view(np.uint64).reshape(m, 4)      # note: d_scal now holds NTT output = still uniform field elements
        b_s = d_base[: 8 * m].cpu().numpy().view(np.uint64).reshape(m, 8)
        t0 = time.perf_counter()
        cpu_msm_out = oc.best_multiexp(s_s, b_s, cores)
        cpu_msm = m / (time.perf_counter() - t0)
        kf = min(k, 22)
        t0 = time.perf_counter()
        cpu_ntt_out = oc.best_fft(s_s[: 1 << kf], omega_words(kf), kf, cores)
        cpu_ntt = (1 << kf) / (time.perf_counter() - t0)
        # the oracle as the checker (SURVEY.md 8d: full compare at k <= 22): the same sample through the C ABI, outside every timed region
        from halo2_scaffold_b200 import verify as V
        checks["msm_sample_equals_oracle"] = bool(V.jacobian_words_to_affine(L.msm(s_s, b_s)) == V.jacobian_words_to_affine(cpu_msm_out))
        checks["ntt_sample_equals_oracle"] = bool((L.ntt(np.array(s_s[: 1 << kf], copy=True), omega_words(kf), kf) == cpu_ntt_out).all())
        cpu_baseline = {"value": cpu_msm, "unit": "points/s", "cores": cores, "kind": "port",
                        "sample": "one best_multiexp over the first 2^%d of the 2^%d points, %d threads (C++ restatement of halo2_proofs v2023_02_02)" % (ks, k, cores),
                        "ntt_value": cpu_ntt, "ntt_unit": "elements/s", "ntt_sample": "one best_fft at 2^%d, %d threads" % (kf, cores)}

    # ---- N > 1: the modes ONE prover process uses (h2b_init(N)), outside every timed region, rank 0 only ------------------
    # parity of the in-library point-range sharding / round-robin columns against the oracle, and strong scaling of one MSM
    in_process = None
    if world > 1 and not args.no_inprocess:
        del d_scal, d_base, d_ntt
        torch.cuda.empty_cache()
        L.shutdown()                                   # this rank's resident sets and scratch: the subprocess owns the GPUs now
        dist.barrier(group=host_group)
        if rank == 0:
            try:
                cmd = [sys.executable, os.path.join(ROOT, "tools", "multi_gpu_inprocess.py"), str(world)] + [str(x) for x in args.strong_k]
                out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
                in_process = json.loads(out.stdout.strip().splitlines()[-1]) if out.returncode == 0 else {"error": out.stderr[-400:]}
            except Exception as ex:        # noqa: BLE001
                in_process = {"error": repr(ex)[:300]}
        dist.barrier(group=host_group)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        ncu = {}
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        except Exception:
            pass
        acc_avg = sum(acc_ms) / max(1, len(acc_ms))
        roofline = {
            "kernel": "msm_pair_reduce_kernel + msm_accumulate_kernel (bucket accumulation)" if pair_total else "msm_accumulate_kernel",
            "bound": "imad", "unit": "TIMAD/s",
            "achieved": IMADS_PER_POINT * n / (acc_avg / 1e3) / 1e12 if acc_avg else None,
            "peak": imad_peak / 1e12,
            "peak_source": "measured in this run: h2b_imad_bench, independent mad.lo.u32 chains on all SMs (MEASURED_PEAKS.json has no integer-pipe figure)",
            "frac": (IMADS_PER_POINT * n / (acc_avg / 1e3)) / imad_peak if acc_avg else None,
            "frac_whole_step": (IMADS_PER_POINT * n * K / (msm_ms / 1e3)) / imad_peak,
            "algorithmic_per_launch": "21760 IMAD x 2^%d points (SURVEY.md 8d canonical figure)" % k,
            "kernel_ms_avg": acc_avg, "kernel_share_of_step": acc_avg * K / msm_ms if msm_ms else None,
            "fq_mul_peak_gmul_s": fqmul_peak / 1e9,
            "traffic": ncu.get("msm_accumulate_kernel"),
        }
        pass_avg = sum(pass_ms) / max(1, len(pass_ms))
        passes_per_ntt = max(1, len(pass_ms) // max(1, K))
        ntt = {
            "metric": "bn254_fr_ntt_elements_per_s", "value": ntt_value, "unit": "elements/s", "k": k, "ms_per_step": ntt_ms / K,
            "verified": bool(checks["ntt_spot_values"]), "verified_how": "one extra step after the timed loop, 4 spot outputs against Horner evaluation on the device; N = 1: also a full compare of a 2^22 transform with the CPU oracle (checks.ntt_sample_equals_oracle)",
            "e2e": {"value": world * n * K / ntt_e2e_s, "unit": "elements/s", "h2d_bytes_per_step": 32 * n, "d2h_bytes_per_step": 32 * n},
            "roofline": {
                "kernel": "ntt_pass_kernel", "bound": "hbm", "unit": "GB/s",
                "achieved": 64.0 * n / (pass_avg / 1e3) / 1e9 if pass_avg else None, "peak": hbm_peak, "peak_source": hbm_src,
                "frac": (64.0 * n / (pass_avg / 1e3) / 1e9) / hbm_peak if pass_avg else None,
                "frac_whole_ntt": (64.0 * n / (ntt_ms / K / 1e3) / 1e9) / hbm_peak,
                "algorithmic_per_launch": "64 B x 2^%d elements per pass launch (each pass reads and writes the vector once); %d passes per NTT" % (k, passes_per_ntt),
                "kernel_ms_avg": pass_avg, "passes": passes_per_ntt,
                "imad_frac_whole_ntt": (MACS_PER_FR_MUL * (n / 2) * k * K / (ntt_ms / 1e3)) / imad_peak,
                "traffic": ncu.get("ntt_pass_kernel"),
            },
        }
        # ---- the widened rows (SURVEY.md 8f) ride along at N = 1: quotient evaluation and SRS point decompression -----------
        # guarded: whatever happens here cannot touch the headline numbers above
        widened = None
        if world == 1 and not args.no_widened:
            try:
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import evaluate_h_bench
                torch.cuda.empty_cache()
                eh = evaluate_h_bench.measure(L, 20, 22, 8, 2, reps=3, cpu_rows=(1 << 14) if not args.no_cpu_baseline else 0)
                m = 1 << 22
                d_pts = torch.empty(m * 8, dtype=torch.int64, device=dev)
                d_enc = torch.empty(m * 4, dtype=torch.int64, device=dev)
                L.gen_points_dev(0, 5, m, d_pts.data_ptr(), st)
                L.check(L.L.h2b_g1_encode_dev(0, d_pts.data_ptr(), m, d_enc.data_ptr(), st))
                L.check(L.L.h2b_g1_decode_dev(0, d_enc.data_ptr(), m, 0, d_pts.data_ptr(), None, st))
                torch.cuda.synchronize()
                e0.record()
                for _ in range(3):
                    L.check(L.L.h2b_g1_decode_dev(0, d_enc.data_ptr(), m, 0, d_pts.data_ptr(), None, st))
                e1.record()
                torch.cuda.synchronize()
                dec_ms = e0.elapsed_time(e1) / 3
                del d_pts, d_enc
                widened = {"evaluate_h": {"rows": 1 << 22, "columns": eh["device_columns"], "ms": eh["evaluate_h_ms"], "rows_per_s": eh["rows_per_s"],
                                          "custom_gates_ms": eh["custom_gates_ms"], "permutation_ms": eh["permutation_ms"], "lookups_ms": eh["lookups_ms"],
                                          "fr_mul_frac_of_peak": [eh["custom_gates_fr_mul_frac_of_peak"], eh["permutation_fr_mul_frac_of_peak"],
                                                                  eh["lookups_fr_mul_frac_of_peak"]],
                                          "parity_sample": eh.get("parity"), "cpu_rows_per_s_1_thread": eh.get("cpu_restatement_rows_per_s_1_thread")},
                           "srs_decompress": {"points": m, "ms": dec_ms, "points_per_s": m / dec_ms * 1e3}}
            except Exception as ex:        # noqa: BLE001
                widened = {"error": repr(ex)[:300]}
        # ---- one larger size beside the headline (N = 1, k = 24 only): 2^26 points, where the bucket costs are amortised and the tables are
        # spaced 22 bits (12 windows) -- device-resident, same roofline definition, verified against the O(n) checksum.  Guarded like the rows above.
        msm_large = None
        if world == 1 and not args.no_widened and k == 24:
            try:
                kl = 26
                nl = 1 << kl
                torch.cuda.empty_cache()
                d_sl = torch.empty(nl * 4, dtype=torch.int64, device=dev)
                d_bl = torch.empty(nl * 8, dtype=torch.int64, device=dev)
                d_ol = torch.empty(28, dtype=torch.int64, device=dev)
                d_cl = torch.empty(4, dtype=torch.int64, device=dev)
                seed_sl, seed_pl = 0xB2000000 + kl, 0xB2001000 + kl
                L.gen_scalars_dev(0, seed_sl, nl, 0, d_sl.data_ptr(), st)
                L.gen_points_dev(0, seed_pl, nl, d_bl.data_ptr(), st)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                h_bl = d_bl.cpu()
                del d_bl
                hl = L.register_bases(h_bl.numpy().view(np.uint64))
                del h_bl
                reg_l = (time.perf_counter() - t0) * 1e3
                info_l = L.base_set_info(hl)
                for _ in range(2):
                    L.msm_dev_registered(0, d_sl.data_ptr(), hl, 0, nl, d_ol.data_ptr(), st)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(3):
                    L.msm_dev_registered(0, d_sl.data_ptr(), hl, 0, nl, d_ol.data_ptr(), st)
                e1.record()
                torch.cuda.synchronize()
                ms_l = e0.elapsed_time(e1) / 3
                L.msm_checksum_dev(0, d_sl.data_ptr(), seed_pl, nl, d_cl.data_ptr(), stream=st)
                torch.cuda.synchronize()
                want_l = V.scalar_mul_generator(V.words_to_int(d_cl.cpu().numpy().view(np.uint64)) % V.FR_MODULUS)
                got_l = V.jacobian_words_to_affine(d_ol.cpu().numpy().view(np.uint64)[:12])
                L.unregister_bases(hl)
                del d_sl, d_ol, d_cl
                torch.cuda.empty_cache()
                msm_large = {"k": kl, "value": nl / ms_l * 1e3, "unit": "points/s", "ms_per_step": ms_l, "verified": bool(got_l == want_l),
                             "frac_whole_step": IMADS_PER_POINT * nl / (ms_l / 1e3) / imad_peak, "srs": dict(info_l, registration_ms=reg_l),
                             "note": "device-resident, 3 steps after 2 warm-up steps, CUDA events; roofline as for the headline (21760 IMAD per point against the measured integer-pipe peak)"}
            except Exception as ex:        # noqa: BLE001
                msm_large = {"error": repr(ex)[:300]}
        line = {
            "metric": "bn254_g1_msm_points_per_s", "value": msm_value, "unit": "points/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": msm_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 limbs (254-bit modular integers)", "data": "synthetic", "config": config_for(args, world),
            "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": 32 * n, "d2h_bytes_per_step": 96,
                    "call": "h2b_msm_bn254_g1(scalars, bases): pageable host arrays, implicit SRS cache (every call re-verifies the digest of "
                            "the caller's %d MiB bases array on host threads while the GPU runs)" % (n * 64 >> 20),
                    "implicit_cache": cache_stats,
                    "host": "%d host cores for %d ranks; per step every rank hashes its bases array (%d MiB) and stages its pageable scalars (%d MiB) "
                            "through pinned slots: at N = 8 this leg is bound by the host's memory bandwidth, not by the GPUs (compare e2e_registered_pinned)"
                            % (os.cpu_count() or 0, world, n * 64 >> 20, n * 32 >> 20)},
            "e2e_registered_pinned": {"value": e2e_pinned_value, "unit": "points/s", "call": "h2b_msm_bn254_g1_registered, pinned scalars"},
            "verified": bool(all(checks.values())), "checks": {kk: bool(v) for kk, v in checks.items()},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "ntt": ntt,
            "msm_phase_ms": {str(t): round(v, 4) for t, v in sorted(phase_ms.items())},
            "srs": dict(set_info, registration_ms=reg_ms, plain=bool(args.plain)),
            "result_x_limb0": int(result_host[0]),
        }
        if in_process is not None:
            line["in_process"] = in_process
            line["strong"] = in_process.get("strong")
            if "parity_ok" in in_process:
                line["checks"]["in_process_multi_gpu_parity_vs_oracle"] = bool(in_process["parity_ok"])
                line["checks"]["strong_scaling_results_equal_checksum"] = bool(all(x.get("verified") for x in in_process.get("strong", [])))
                line["verified"] = bool(all(line["checks"].values()))
        if widened:
            line["widened_rows"] = widened
        if msm_large is not None:
            line["msm_large"] = msm_large
        if witness:
            line["witness_like"] = witness
        if cpu_baseline:
            line["cpu_baseline"] = cpu_baseline
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
