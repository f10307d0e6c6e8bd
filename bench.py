#!/usr/bin/env python3
"""Benchmark of the hot path: BN254 G1 commitment MSM (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA, sm_100a)
    python bench.py --impl reference --gpus N ...            # the reference's CPU algorithm (oracle)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as .npy

A "step" is ONE multi-scalar multiplication of 2^LOG2N uniformly random BN254 scalars against a
resident commitment key (CE::commit with r = 0, benches/commit.rs:30,112-125).
  value   device-resident throughput: scalars already in HBM, K calls of b200_msm_dev timed with
          CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
  e2e     the same metric through the host-pointer C ABI (b200_commit for N=1): scalars start in
          PINNED HOST memory, the H2D copy and the D2H read of the 96-byte result are inside the
          timed region (wall clock around K blocking calls).
  N > 1   the (scalar, base) pairs are sharded by index range across ranks; every rank reduces its
          slice to one point, the partials are all-gathered over NCCL (96 B per rank) and summed on
          every rank (SURVEY.md §8e).  Total work is fixed => "scaling": "strong".
Inputs are synthetic: key bases[i] = (k0+i)*G built on the device, scalars from numpy's seeded
PRNG (32 random bytes masked below the modulus = a uniform Montgomery residue).
The GPU arm never touches oracle/; the cpu_baseline leg and --impl reference do (as the timed
CPU implementation, which is what they are for).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CURVE = 0  # BN254 G1
SCALAR_FIELD = 0  # BN254 Fr
R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
K0 = 0x5EED
METRIC = "MSM throughput (2^20 BN254 scalar*G1/s)"
UNIT = "pairs/s"
ALG_BYTES_PER_PAIR = 96  # 32 B scalar + 64 B affine base, each read once (SURVEY.md §8d)


def msm_config(log2n):
    """The workload description, identical in both arms (the driver compares the dicts)."""
    return {"workload": f"BN254 G1 Pippenger MSM, 2^{log2n} uniform scalars, resident key (BASELINE.json configs[1])",
            "log2n": log2n, "pairs_per_step": 1 << log2n,
            "l2": "GPU arm: working set (window tables 64*15*n B + sort buffers) >> 126 MB L2, no flush needed; "
                  "CPU arm: 96 MiB of inputs >> host caches"}


def synth_scalars(n, seed):
    """n x 32 B little-endian values uniform in [0, 2^253): every 32-byte string below the
    modulus is the Montgomery representation of exactly one field element, so this is a
    (near-)uniform scalar vector without any field arithmetic on the host."""
    import numpy as np
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 1 << 63, size=(n, 4), dtype=np.uint64) * 2 + rng.integers(0, 2, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 61) - 1)  # < 2^253 < r
    return a


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.first = 0

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self, wait_s=5.0):
        """Call right before the timed region: waits until nvidia-smi is up and sampling (its start-up
        must not fall inside the region: the fork and NVML initialisation stall kernel launches for
        milliseconds), then remembers where the region's samples begin."""
        if not self.proc:
            return
        t0 = time.time()
        while not self.lines and time.time() - t0 < wait_s:
            time.sleep(0.02)
        self.first = max(0, len(self.lines) - 1)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines[self.first:]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


def measured_peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def run_b200(args):
    import torch
    import torch.distributed as dist

    import nova_b200 as nb
    from nova_b200.native import check, lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    L = lib()
    check(L.b200_init(local_rank))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from nova_b200.sharding import shard_range

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    stream = torch.cuda.Stream()
    sp = ctypes.c_void_p(stream.cuda_stream)
    d_part = torch.zeros(96, dtype=torch.uint8, device="cuda")
    d_all = torch.zeros(96 * world, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(96, dtype=torch.uint8, device="cuda")

    peer_group = None
    if world > 1 and args.exchange == "fused":
        from nova_b200.sharding import PeerGroup
        peer_group = PeerGroup()  # exchange buffers mapped across the ranks (CUDA IPC); the only set-up collective

    def sharded_msm_step(ck_, d_sc_, n_):
        """One MSM of the whole vector: local Pippenger over this rank's index range; with N > 1 the reduction's
        last kernel writes the rank's partial sum into every peer's exchange buffer over NVLink, waits for the
        peers' and adds them (b200_msm_sharded_dev) -- no NCCL call per step.  --exchange nccl keeps the round-1
        form (all-gather of 96-byte partials + b200_jacobian_sum_dev) for A/B."""
        if world == 1:
            check(L.b200_msm_dev(ck_.handle, 0, d_sc_.data_ptr(), n_, d_part.data_ptr(), sp))
        elif peer_group is not None:
            peer_group.msm(ck_, 0, d_sc_.data_ptr(), n_, d_out.data_ptr(), sp)
        else:
            check(L.b200_msm_dev(ck_.handle, 0, d_sc_.data_ptr(), n_, d_part.data_ptr(), sp))
            dist.all_gather_into_tensor(d_all, d_part)
            check(L.b200_jacobian_sum_dev(CURVE, d_all.data_ptr(), world, d_out.data_ptr(), sp))

    def time_other_size(log2n, steps, warmup):
        """Same sharded MSM at another total size (BASELINE.json configs[3] names 2^22): device time
        per step, max over ranks.  Reported beside the headline, never instead of it."""
        nt = 1 << log2n
        lo_, hi_ = shard_range(nt, rank, world)
        n_ = hi_ - lo_
        ck_ = nb.CommitmentKey.setup_synthetic(nb.Curve(CURVE), n_, k0=K0 + lo_)
        d_sc_ = torch.from_numpy(synth_scalars(nt, seed=2)[lo_:hi_].view("uint8").reshape(-1)).cuda()
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                sharded_msm_step(ck_, d_sc_, n_)
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            for _ in range(steps):
                sharded_msm_step(ck_, d_sc_, n_)
            b.record(stream)
            barrier()
        tt = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ck_.release()
        del d_sc_
        torch.cuda.empty_cache()
        ms = float(tt.item()) / steps
        return {"log2n": log2n, "pairs_per_step": nt, "ms_per_step": round(ms, 4), "value": nt / (ms * 1e-3),
                "unit": UNIT, "steps": steps, "warmup": warmup}

    n_total = 1 << args.log2n
    lo, hi = shard_range(n_total, rank, world)  # this rank's index range of (scalar, base) pairs
    n = hi - lo
    ck = nb.CommitmentKey.setup_synthetic(nb.Curve(CURVE), n, k0=K0 + lo, window_bits=args.window_bits)
    sc_np = synth_scalars(n_total, seed=2)[lo:hi]
    d_sc = torch.from_numpy(sc_np.view("uint8").reshape(-1)).cuda()

    def step_device():
        sharded_msm_step(ck, d_sc, n)

    # ---------------- device-resident throughput ("value") --------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # started before the warm-up so that its start-up cost stays outside the timing
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step_device()
        barrier()
        check(L.b200_profile_enable(1))
        check(L.b200_profile_reset())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if rank == 0:
            sampler.mark()
        barrier()
        e0.record(stream)
        for _ in range(args.steps):
            step_device()
        e1.record(stream)
        barrier()
        clocks = sampler.stop() if rank == 0 else None
    ms_total = e0.elapsed_time(e1)
    stage_ms = (ctypes.c_double * 5)()
    msms, launches = ctypes.c_uint64(0), ctypes.c_uint64(0)
    check(L.b200_profile_read(stage_ms, 5, ctypes.byref(msms), ctypes.byref(launches)))
    check(L.b200_profile_enable(0))
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / args.steps
    value = n_total / (ms_per_step * 1e-3)

    # ---------------- end to end through the host-pointer C ABI ("e2e") -------------------------
    h_ptr = ctypes.c_void_p()
    check(L.b200_host_alloc(n * 32, ctypes.byref(h_ptr)))
    ctypes.memmove(h_ptr, sc_np.ctypes.data, n * 32)
    out_host = ctypes.create_string_buffer(96)
    h_pinned_t = None
    if world > 1:
        h_pinned_t = torch.empty(96, dtype=torch.uint8).pin_memory()

    def step_e2e():
        if world == 1:
            check(L.b200_commit(ck.handle, h_ptr, n, None, out_host))  # H2D + MSM + D2H, blocking
        else:
            with torch.cuda.stream(stream):
                check(L.b200_memcpy_h2d(d_sc.data_ptr(), h_ptr, n * 32))
                step_device()
                h_pinned_t.copy_(d_out, non_blocking=True)
                stream.synchronize()

    for _ in range(max(1, args.warmup)):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms_per_step = float(t.item()) / args.steps
    check(L.b200_host_free(h_ptr))

    # ---------------- the timed results are CHECKED (outside every timed region) -------------------
    # bases are P_i = (K0 + i) G, so the MSM must equal [sum_i s_i (K0 + i)] G: one scalar-mul on the oracle side
    result_check = None
    if rank == 0:
        device_result = (d_out if world > 1 else d_part).cpu().numpy().tobytes()
        e2e_result = out_host.raw if world == 1 else h_pinned_t.numpy().tobytes()
        result_check = closed_form_check(args.log2n, device_result, e2e_result)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"msm_device": device_result, "commit_e2e": e2e_result})

    # ---------------- the same sharded MSM at the other sizes north_star names -------------------
    other_sizes = [time_other_size(lg, steps=5, warmup=3) for lg in args.other_log2n if lg != args.log2n]

    if peer_group is not None:
        peer_group.status()  # B200_E_PEER if any exchange ever timed out
        peer_group.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (k_accumulate) ----------------------------
    peak, peak_src = measured_peak_hbm()
    acc_ms = stage_ms[2] / max(1, msms.value)  # average launch duration over the timed region
    alg_bytes = ALG_BYTES_PER_PAIR * n
    achieved = alg_bytes / (acc_ms * 1e-3) / 1e9 if acc_ms > 0 else 0.0
    stage_names = ["digits", "sort", "accumulate", "fixup", "reduce"]
    traffic = None
    tf = os.path.join(ROOT, "profiles", "accumulate_traffic_bytes.json")
    if os.path.exists(tf):
        try:
            traffic = json.load(open(tf)).get(f"log2n_{args.log2n}_gpus_{world}")
        except Exception:
            traffic = None
    cc, nt = ctypes.c_int(0), ctypes.c_int(0)
    check(L.b200_ck_len(ck.handle, None, ctypes.byref(cc), ctypes.byref(nt)))
    # the pipe that actually bounds the kernel: an XYZZ mixed addition (madd-2008-s: 8M + 2S) costs 9.5 full
    # Montgomery products here (y3 = r(q - x3) - y1 ppp shares ONE reduction between its two products), one addition
    # per non-zero digit; ceiling = the carry-chain multiplier's measured 64.2 G field-mul/s (tools/microbench.cu)
    fe_muls = 9.5 * n * nt.value * (1.0 - 2.0 ** -cc.value)
    mul_rate = fe_muls / (acc_ms * 1e-3) / 1e9 if acc_ms > 0 else 0.0
    roofline = {
        "kernel": "k_accumulate<BN254_FQ>", "bound": "hbm", "achieved": round(achieved, 2), "peak": peak,
        "unit": "GB/s", "frac": round(achieved / peak, 5), "traffic": traffic, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": round(acc_ms, 4),
        "note": "MSM is INT32-multiply bound, not HBM bound (DESIGN.md §Roofline); the HBM fraction is "
                "reported because north_star asks for it",
        "stage_ms_per_msm": {k: round(stage_ms[i] / max(1, msms.value), 4) for i, k in enumerate(stage_names)},
        "int_mul_pipe": {"achieved": round(mul_rate, 2), "peak": 64.2, "unit": "G field-mul/s",
                         "frac": round(mul_rate / 64.2, 4), "window_bits": cc.value, "windows": nt.value,
                         "peak_source": "measured fe_mul throughput of this multiplier (tools/microbench.cu)",
                         # ceilings that do not depend on this multiplier: wide 32x32+64 products issued per clock and
                         # SM, measured with tools/microbench.cu (61 without a carry flag, 30.5 with one), x 148 SMs x
                         # 1.965 GHz / 136 wide products per Montgomery product (64 + 64 + 8)
                         "hw_bounds": {"imad_wide_with_carry": {"peak": 65.2, "frac": round(mul_rate / 65.2, 4)},
                                       "imad_wide_full_rate": {"peak": 130.5, "frac": round(mul_rate / 130.5, 4),
                                                               "note": "unreachable with a carry chain; a carry-free "
                                                                       "formulation needs ~2x the instructions (DESIGN.md §4)"}}},
    }

    # ---------------- CPU baseline beside it (N = 1 only) ---------------------------------------
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_reference_run(args.log2n, steps=2, warmup=1, sc_np=sc_np)

    # ---------------- the prover workloads of BASELINE.json configs[2..4], each timed AND checked -----
    # (tools/workloads.py: prove_step replay vs the C oracle, HyperKZG 2^22 and ppsnark 2^18 proofs accepted by the
    #  restated verifiers).  `bench.py --workload X --gpus N` runs one of them alone, also over N GPUs.
    workloads_out = {}
    if world == 1 and not args.no_prove_step:
        ck.release()
        del d_sc
        torch.cuda.empty_cache()
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import workloads as wl
        for name, fn in (("prove_step", lambda: wl.prove_step(steps=5, warmup=2, check_parity=not args.no_cpu_baseline)),
                         ("hyperkzg_prove_2p22", lambda: wl.hyperkzg(log2n=22, steps=2, warmup=1)),
                         ("ppsnark_prove_2p18", lambda: wl.ppsnark(log2cons=18, steps=2, warmup=1))):
            try:
                workloads_out[name] = fn()
            except Exception as e:  # never let a side measurement take the headline down
                workloads_out[name] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u32 limbs (256-bit prime-field / curve integers)",
        "data": "synthetic",
        "config": msm_config(args.log2n),
        "sharding": f"index-range x{world}" + ("" if world == 1 else
                                                  (", partial sums exchanged by peer stores inside the reduction kernel"
                                                   if peer_group is not None else ", NCCL all-gather + local sum")),
        "clocks": clocks,
        "e2e": {"value": n_total / (e2e_ms_per_step * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms_per_step,
                "h2d_bytes_per_step": n * 32, "d2h_bytes_per_step": 96,
                "api": "b200_commit (host pointers, pinned)" if world == 1 else
                       ("b200_memcpy_h2d + b200_msm_sharded_dev + D2H" if peer_group is not None else
                        "b200_memcpy_h2d + b200_msm_dev + NCCL all_gather + b200_jacobian_sum_dev + D2H")},
        "gpu_launches": int(launches.value),
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
        "result_check": result_check,
        "parity_checked": bool(result_check and result_check["ok"]),
        "other_sizes": other_sizes,
        "workloads": workloads_out,
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def closed_form_check(log2n, device_result_jac, e2e_result_jac):
    """Checker (oracle side): expected = [sum_i s_i (K0 + i) mod r] G for the bench's scalars."""
    from nova_b200.provider import Curve, _jac_to_affine
    from oracle import coracle as co
    from oracle.pyref import CURVES
    c = CURVES[CURVE]
    sc = synth_scalars(1 << log2n, seed=2).tobytes()
    k = co.dot_index(SCALAR_FIELD, sc, K0)
    exp = c.affine_from_bytes(co.scalar_mul(CURVE, c.affine_bytes(c.gen), k))
    got_dev = _jac_to_affine(Curve(CURVE), device_result_jac)
    got_e2e = _jac_to_affine(Curve(CURVE), e2e_result_jac)
    return {"device_result_equals_closed_form": bool(got_dev == exp), "e2e_result_equals_closed_form": bool(got_e2e == exp),
            "ok": bool(got_dev == exp and got_e2e == exp),
            "checker": "oracle: [sum_i s_i (k0+i)] G by one scalar multiplication (bases are (k0+i) G)"}


def dump_outputs(out_dir, jacobian_results):
    """--dump-outputs: every MSM result of the last timed step as DIR/<name>.npy, float32 of shape (2, 32): the affine
    x and y in canonical (non-Montgomery) form, 32 little-endian bytes each, so every value is exact.  Affine because
    another build may return the same point with other Jacobian coordinates; the point at infinity is all zeros."""
    import numpy as np

    from nova_b200.provider import Curve, _jac_to_affine
    os.makedirs(out_dir, exist_ok=True)
    for name, jac in jacobian_results.items():
        point = _jac_to_affine(Curve(CURVE), jac) or (0, 0)
        raw = b"".join(v.to_bytes(32, "little") for v in point)
        np.save(os.path.join(out_dir, f"{name}.npy"), np.frombuffer(raw, dtype=np.uint8).reshape(2, 32).astype(np.float32))


def effective_cores():
    """Host threads actually available: min(visible CPUs, cgroup v2 CPU quota)."""
    n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def cpu_reference_run(log2n, steps, warmup, sc_np=None):
    """Time the CPU restatement of the reference's msm() (oracle/oracle.c, msm.rs:225-419 with the
    msm_best stand-in) with all host cores on the bench workload (or a bounded sample of it)."""
    from oracle import coracle as co
    cores = effective_cores()
    n_full = 1 << log2n
    if sc_np is None:
        sc_np = synth_scalars(n_full, seed=2)
    # bound the sample to a few seconds of work per step: probe at 2^16
    probe = 1 << min(16, log2n)
    bases_probe = co.gen_bases(CURVE, probe, K0)
    sc_probe = sc_np[:probe].tobytes()
    t0 = time.perf_counter()
    co.msm(CURVE, sc_probe, bases_probe, cores)
    t_probe = time.perf_counter() - t0
    est_full = t_probe * (n_full / probe)
    budget_s = 20.0
    n = n_full
    while n > probe and est_full * (n / n_full) * (steps + warmup) > budget_s:
        n //= 2
    bases = co.gen_bases(CURVE, n, K0)
    sc = sc_np[:n].tobytes()
    for _ in range(warmup):
        co.msm(CURVE, sc, bases, cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        co.msm(CURVE, sc, bases, cores)
    dt = (time.perf_counter() - t0) / steps
    return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port", "ms_per_step": round(dt * 1e3, 3),
            "sample": f"first 2^{n.bit_length() - 1} of the 2^{log2n} pairs, {steps} run(s), {dt * 1e3:.1f} ms each",
            "note": "C restatement of msm.rs (signed split + bit-width partition; halo2curves msm_best "
                    "restated as signed-digit Pippenger, c = ln(n)+2, (window x slice) jobs over all "
                    "cores), pthreads; Montgomery products on the mulx/adcx/adox path (inline assembly -- what halo2curves' "
                    "`asm` feature gives the reference) when the CPU has BMI2 + ADX, unsigned __int128 otherwise"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_reference_run(args.log2n, steps=args.steps, warmup=max(1, min(args.warmup, 2)))
    n_sample = cb["sample"]
    out = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u64 limbs (256-bit prime-field / curve integers)",
        "data": "synthetic",
        "config": msm_config(args.log2n),
        "sample": n_sample,
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


WORKLOAD_METRICS = {
    "hyperkzg": ("HyperKZG EvaluationEngine::prove time (BN254, BASELINE.json configs[3])", "ms"),
    "ppsnark": ("ppsnark RelaxedR1CSSNARK::prove time (BN254, BASELINE.json configs[4])", "ms"),
    "prove_step": ("RecursiveSNARK::prove_step kernel-sequence time (BN254/Grumpkin, BASELINE.json configs[2])", "ms"),
}


def workload_config(args):
    if args.workload == "hyperkzg":
        return {"workload": f"HyperKZG prove, 2^{args.log2n} uniform BN254 scalars", "log2n": args.log2n}
    if args.workload == "ppsnark":
        return {"workload": f"ppsnark prove, sha256-like synthetic shape, 2^{args.log2cons} constraints",
                "log2cons": args.log2cons}
    return {"workload": "prove_step kernel-sequence replay, MinRoot-sized shapes (2.07e5 / 1.05e4 constraints)"}


def run_workload(args):
    """bench.py --workload {hyperkzg, ppsnark, prove_step} [--gpus N]: one prover workload of BASELINE.json
    configs[2..4], timed and then checked by the restated verifier / the C oracle (tools/workloads.py)."""
    import torch
    import torch.distributed as dist

    from nova_b200.native import check, lib
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    L = lib()
    check(L.b200_init(local_rank))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import workloads as wl
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.mark()
    check(L.b200_profile_reset())
    if args.workload == "hyperkzg":
        res = wl.hyperkzg(log2n=args.log2n, steps=args.steps, warmup=args.warmup)
        ms, e2e_ms = res["ms_per_proof"], res["e2e_ms_per_proof"]
        h2d, d2h = res["h2d_bytes_per_proof"] // world, res["d2h_bytes_per_proof"]
    elif args.workload == "ppsnark":
        if world > 1:
            raise SystemExit("--workload ppsnark runs on one GPU (its multi-GPU pieces are covered by tests/test_ppsnark_sharded.py)")
        res = wl.ppsnark(log2cons=args.log2cons, steps=args.steps, warmup=args.warmup)
        ms = e2e_ms = res["ms_per_proof"]
        h2d, d2h = 0, 0
    else:
        if world > 1:
            raise SystemExit("--workload prove_step runs on one GPU (BASELINE.json configs[2]: 1xB200)")
        res = wl.prove_step(steps=args.steps, warmup=args.warmup)
        ms = e2e_ms = res["ms_per_step"]
        h2d, d2h = res["h2d_bytes_per_step"], res["d2h_bytes_per_step"]
    clocks = sampler.stop() if rank == 0 else None
    launches = ctypes.c_uint64(0)
    check(L.b200_profile_read(None, 0, None, ctypes.byref(launches)))
    if rank == 0:
        metric, unit = WORKLOAD_METRICS[args.workload]
        print(json.dumps({
            "metric": metric, "value": ms, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "u32 limbs (256-bit prime-field / curve integers)", "data": "synthetic",
            "config": workload_config(args), "clocks": clocks,
            "e2e": {"value": e2e_ms, "unit": unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches.value), "parity_checked": res["parity_checked"], "detail": res}))
    if world > 1:
        dist.destroy_process_group()


def run_workload_reference(args):
    """--impl reference --workload X: the same op sequence through the C restatement on the host cores."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    metric, unit = WORKLOAD_METRICS[args.workload]
    base = {"impl": "reference", "metric": metric, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "u64 limbs (256-bit prime-field / curve integers)", "data": "synthetic",
            "config": workload_config(args)}
    if args.workload == "hyperkzg":
        import hyperkzg_replay
        lg = min(args.log2n, 20)  # bounded sample: the 2^20 prover takes ~3 s on 16 cores; scaled linearly above
        cb = hyperkzg_replay.cpu(lg)
        v = cb["ms"]["total"] * (1 << (args.log2n - lg))
        cb = {"value": v, "unit": unit, "cores": cb["cores"], "kind": "port",
              "sample": f"whole prover at 2^{lg}, scaled x{1 << (args.log2n - lg)} to 2^{args.log2n}", "phases_ms": cb["ms"]}
    elif args.workload == "prove_step":
        import prove_step_replay as psr
        r = psr.cpu_replay(steps=max(1, min(args.steps, 3)))
        v = r["ms_per_step"]
        cb = {"value": v, "unit": unit, "cores": r["cores"], "kind": "port", "sample": "the full step"}
    else:
        print(json.dumps(dict(base, unavailable="the whole-prover CPU restatement of ppsnark is Python big-integer code "
                                                "(oracle/ppsnark_ref.py, the parity checker): not a timing baseline")))
        return
    print(json.dumps(dict(base, value=v, ms_per_step=v, cpu_baseline=cb,
                          e2e={"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 20, or 3 with --workload)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log2n", type=int, default=20)
    ap.add_argument("--window-bits", type=int, default=0)
    ap.add_argument("--other-log2n", type=lambda v: [int(x) for x in v.split(",") if x], default=[22, 24],
                    help="also time the sharded MSM at these total sizes (reported under other_sizes)")
    ap.add_argument("--workload", default="msm", choices=["msm", "hyperkzg", "ppsnark", "prove_step"],
                    help="msm = the headline (BASELINE.json configs[1]); the others time AND check one prover workload")
    ap.add_argument("--log2cons", type=int, default=18, help="--workload ppsnark: log2 of the constraint count")
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"],
                    help="N > 1: how the ranks' partial sums are combined (fused = peer stores inside the reduction kernel)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-prove-step", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the MSM results of the last timed step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.workload == "msm" else 3
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "msm" or args.impl != "b200"):
        ap.error("--dump-outputs writes the results of the MSM workload on --impl b200 only")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.workload != "msm":
        if args.workload == "hyperkzg" and "--log2n" not in sys.argv:
            args.log2n = 22
        (run_workload_reference if args.impl == "reference" else run_workload)(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
