#!/usr/bin/env python
"""bench.py - Groth16 proofs/sec (BN254, 2^20-constraint-domain circom squaring chain) on B200, next to the CPU path.

One "step" = one call of Groth16::<Bn254, CircomReduction>::create_proof_with_reduction_and_matrices
(ark-circom's benches/groth16.rs:69-84 times exactly this): proving key + matrices resident, witness given, fixed r, s.

  python bench.py [--gpus N --steps K --warmup W]        our arm (CUDA, through the C ABI)
  python bench.py --impl reference [...]                 the CPU restatement of the ark-groth16 0.5 path (oracle/cref.c)
  python bench.py [...] --dump-outputs DIR               also write the proof of the last timed step to DIR (dump_outputs)

Output: ONE JSON line (rank 0).  `value` = device-resident throughput (witness already in HBM), `e2e` = through
Groth16.create_proof_with_reduction_and_matrices with a pinned HOST witness (H2D 32 B x n_vars and D2H 256 B inside the
timed region), `roofline` = the dominant kernel (MSM bucket accumulation, G1) against measured HBM bandwidth,
`cpu_baseline` = oracle/cref.c on the host cores, same key / witness / (r, s), proof bytes asserted identical.
N > 1: the headline is N replicas (whole provers, weak scaling); `other_mode` is the same 2^20 proof base-sharded over the
N GPUs (strong scaling: latency), and `config4` is BASELINE.json config 4: a 2^22 chain, MSM bases sharded over the N GPUs.
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
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (it may be read-only)

R_FIX = 0x1234567890abcdef1234567890abcdef
S_FIX = 0xfedcba0987654321fedcba0987654321
METRIC = "groth16_proofs_per_sec_bn254_2p20"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.index, self.rows, self.proc, self.th = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.th = threading.Thread(target=self._read, daemon=True)
        self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace('.', '').isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith('active')})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def build_workload(log_n, kind):
    from circom_compat_b200 import synth
    t0 = time.time()
    if kind == 'chain':
        circ = synth.chain_circuit(1 << log_n)
        w = synth.chain_witness(1 << log_n, 3)
    else:
        circ, w = synth.circomlike_circuit(log_n)
    log(f"[bench] circuit {kind} 2^{log_n}: n_vars={circ.n_vars} m={circ.num_constraints} domain={circ.domain_size} ({time.time() - t0:.1f}s)")
    return circ, w


def oracle_key(pk, cm):
    import numpy as np
    za = dict(n_vars=pk.n_vars, n_public=pk.n_public, domain_size=pk.domain_size, num_constraints=cm.num_constraints, a_csr=cm.a, b_csr=cm.b)
    for name in ('alpha_g1', 'beta_g1', 'delta_g1', 'beta_g2', 'delta_g2', 'a_query', 'b_g1_query', 'b_g2_query', 'l_query', 'h_query'):
        za[name] = np.ascontiguousarray(getattr(pk, name), dtype=np.uint64)
    return za


def physical_cores():
    """hardware cores (not SMT threads): the OpenMP port runs ~3x slower oversubscribed on hyperthreads"""
    try:
        seen = set()
        phys = core = None
        for line in open('/proc/cpuinfo'):
            if line.startswith('physical id'):
                phys = line.split(':')[1].strip()
            elif line.startswith('core id'):
                core = line.split(':')[1].strip()
            elif not line.strip():
                if phys is not None and core is not None:
                    seen.add((phys, core))
                phys = core = None
        if seen:
            return len(seen)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def cpu_model():
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                return line.split(':', 1)[1].strip()
    except Exception:
        pass
    return 'unknown'


def pin_cpu_arm():
    """One OpenMP thread per physical core, packed: without this the same 64-thread run moved 2.5x between boxes (threads
    landing on SMT siblings / drifting across sockets).  Must be in the environment before libgomp is loaded (oracle/cref)."""
    os.environ.setdefault('OMP_PLACES', 'cores')
    os.environ.setdefault('OMP_PROC_BIND', 'close')
    os.environ.setdefault('OMP_DYNAMIC', 'false')


def cpu_setup(circ):
    """proving key from the CPU oracle only (reference arm: none of our kernels anywhere)"""
    from circom_compat_b200 import synth
    from oracle import cref

    nt = physical_cores()           # explicit: torchrun exports OMP_NUM_THREADS=1

    class CpuFixedBase:
        def fixed_base_g1(self, s): return cref.fixed_base_g1(s, nt)
        def fixed_base_g2(self, s): return cref.fixed_base_g2(s, nt)
    return synth.setup(CpuFixedBase(), circ)


def workload_config(args, circ):
    """names the WORKLOAD only - identical in both arms (how each arm runs it is reported beside it, not inside)"""
    return {"workload": f"circom squaring chain (reference bench family, test-vectors/complex-circuit), domain 2^{args.log_n}, "
                        f"n_vars={circ.n_vars}, constraints={circ.num_constraints}, BN254, synthetic trapdoor zkey seed 0xB200, fixed r,s",
            "witness": args.workload, "log_n": args.log_n,
            "l2": "inputs larger than L2 (proving-key tables ~6 GB per proof pass vs 126 MB L2)"}


def dump_outputs(out_dir, proof_bytes):
    """What the caller of the timed path receives from its last step: the 256-byte Proof (canonical little-endian affine
    coordinates), written as proof_a.npy (2, 32), proof_b.npy (2, 2, 32) and proof_c.npy (2, 32) in the order of Proof.a /
    Proof.b / Proof.c.  One float32 per byte: every value is exact, and a one-bit difference moves a value by at least 1.
    The inputs (synthetic key seed, witness, r, s) are fixed, so two builds given the same arguments must write the same files."""
    import numpy as np
    b = np.frombuffer(proof_bytes, dtype=np.uint8).astype(np.float32)
    assert b.size == 256, b.size
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (('proof_a', b[:64].reshape(2, 32)), ('proof_b', b[64:192].reshape(2, 2, 32)), ('proof_c', b[192:].reshape(2, 32))):
        np.save(os.path.join(out_dir, name + '.npy'), arr)
    log(f"[bench] last timed proof written to {out_dir}/proof_{{a,b,c}}.npy")


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    pin_cpu_arm()
    import numpy as np  # noqa: F401
    from oracle import cref
    from circom_compat_b200 import fr_to_mont
    cref.build()
    cores = physical_cores()        # OpenMP num_threads() clauses; OMP_NUM_THREADS (set to 1 by torchrun) does not apply
    circ, w = build_workload(args.log_n, args.workload)
    t0 = time.time()
    pk, _ = cpu_setup(circ)
    cm = circ.matrices()
    log(f"[bench] CPU setup {time.time() - t0:.1f}s on {cores} threads ({cpu_model()}, nproc={os.cpu_count()})")
    za, wm = oracle_key(pk, cm), fr_to_mont(w)
    for _ in range(args.warmup):
        cref.prove(za, R_FIX, S_FIX, wm, nthreads=cores)
    steps = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        t1 = time.perf_counter()
        proof = cref.prove(za, R_FIX, S_FIX, wm, nthreads=cores)
        steps.append(time.perf_counter() - t1)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, proof)
    val = args.steps / dt
    sample = f"{args.steps} full proofs of the {args.workload} 2^{args.log_n} workload, oracle/cref.c (C + OpenMP restatement of ark-groth16 0.5), {cores} threads pinned one per core"
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "proofs/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32x8 (254-bit Montgomery integers)",
           "data": "synthetic", "config": workload_config(args, circ), "parallelism": f"{cores} OpenMP threads on the host",
           "cpu_baseline": {"value": val, "unit": "proofs/s", "cores": cores, "kind": "port", "sample": sample, "phases_s": cref.last_phase_seconds(),
                            "best_step_value": 1.0 / min(steps), "step_seconds": steps, "cpu_model": cpu_model(), "nproc": os.cpu_count(),
                            "omp": {k: os.environ.get(k) for k in ('OMP_PLACES', 'OMP_PROC_BIND')}},
           "e2e": {"value": val, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit(out)


def static_kernel_profile():
    """per-launch DRAM traffic and IMAD.WIDE count of the dominant kernel come from an ncu capture, not from this run: the
    committed summary profiles/kernel_profile.json (written by tools/ncu_summary.py from the capture named inside it)."""
    p = os.path.join(ROOT, 'profiles', 'kernel_profile.json')
    try:
        return json.load(open(p))
    except Exception:
        return None


def run_ours(args):
    import numpy as np
    import torch
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        import datetime
        dist.init_process_group('nccl', device_id=torch.device('cuda', local), timeout=datetime.timedelta(seconds=300))
    from circom_compat_b200 import Context, Groth16, CircomReduction, fr_to_mont, fr_from_mont, synth, sharding, release_all
    from circom_compat_b200.zkey import Q_MOD
    dev = f'cuda:{local}'

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def threads(fn, n):
        ths = [threading.Thread(target=fn, args=(i,)) for i in range(n)]
        [t_.start() for t_ in ths]; [t_.join() for t_ in ths]

    setup_ctx = Context(local)

    class Workload:
        def __init__(self, log_n, kind, inflight):
            self.log_n = log_n
            self.circ, self.w = build_workload(log_n, kind)
            t0 = time.time()
            self.pk, self.td = synth.setup(setup_ctx, self.circ)
            self.cm = self.circ.matrices()
            log(f"[bench] rank {rank}: 2^{log_n} trapdoor setup + GPU fixed-base key generation {time.time() - t0:.1f}s")
            self.wm_np = fr_to_mont(self.w)
            self.pinned = [torch.empty(self.wm_np.shape, dtype=torch.int64).pin_memory() for _ in range(inflight)]
            self.wms = [p_.numpy().view(np.uint64) for p_ in self.pinned]
            for w_ in self.wms:
                w_[...] = self.wm_np

        def check_closed_form(self, proof):
            """the unique proof under the trapdoor, from a closed form that uses no h (synth.expected_proof_dlogs_independent):
            H term = (a(tau) b(tau) - c(tau)) / delta, so it checks the witness map, the five MSMs and the assembly"""
            da, db, dc = synth.expected_proof_dlogs_independent(self.td, self.circ, self.w, R_FIX, S_FIX)
            ea = setup_ctx.fixed_base_g1(synth._ints_to_limbs([da, dc])); eb = setup_ctx.fixed_base_g2(synth._ints_to_limbs([db]))
            qinv = pow(1 << 256, -1, Q_MOD)
            def canon(a): return [int.from_bytes(np.ascontiguousarray(a).tobytes()[i:i + 32], 'little') * qinv % Q_MOD for i in range(0, a.size * 8, 32)]
            exp = canon(ea[0]) + canon(eb[0]) + canon(ea[1])
            got = [int.from_bytes(proof.data[i:i + 32], 'little') for i in range(0, 256, 32)]
            assert exp == got, "proof does not match the trapdoor's closed-form expectation"
            # second, h-based form: additionally pins h . h_query == (ab - c)(tau) / delta for the GPU's own h
            h = fr_from_mont(CircomReduction.witness_map_from_matrices(self.cm, self.circ.num_inputs, self.circ.num_constraints, self.wms[0], setup_ctx))
            assert synth.expected_proof_dlogs(self.td, self.w, h, R_FIX, S_FIX, self.circ.num_inputs) == (da, db, dc), "witness map disagrees with the trapdoor"

    def measure(wl, mode, steps, warmup, want_inflight):
        """mode: 'single' / 'replicas' (whole proofs per GPU) or 'sharded' (MSM base ranges over the GPUs, partials exchanged
        through NVLink peer memory inside the captured proof graph, or with one NCCL all-gather)."""
        sharded = mode == 'sharded'
        pk, cm, circ = wl.pk, wl.cm, wl.circ
        # a sharded proof occupies every GPU for its whole duration; what sharding buys is latency, so one is in flight
        inflight = 1 if sharded else max(1, want_inflight)
        ctxs = [Context(local, rank if sharded else 0, world if sharded else 1) for _ in range(inflight)]
        fused = sharded and args.exchange == 'p2p'
        if fused:
            ctxs[0].prepare(pk, cm)                                # sizes the exchange arena (split witness map) before it is exported
            sharding.connect_p2p(ctxs[0], dist)                    # CUDA-IPC handles of the exchange arenas, once
            dist.barrier()

        def one_proof(i=0):
            if not sharded:
                return Groth16.create_proof_with_reduction_and_matrices(pk, R_FIX, S_FIX, cm, circ.num_inputs, circ.num_constraints, wl.wms[i], ctxs[i])
            if fused:
                return Groth16.prove_sharded_p2p(pk, cm, R_FIX, S_FIX, wl.wms[i], ctxs[i])
            return sharding.prove_sharded(ctxs[i], pk, cm, wl.wms[i], R_FIX, S_FIX, dist, dev, None)

        from concurrent.futures import ThreadPoolExecutor
        use_async = (not sharded) and args.host_driver == 'async'
        pool = ThreadPoolExecutor(max_workers=inflight)          # 'threads' driver: one host thread per in-flight proof

        def run_steps(total):
            if use_async:
                # ONE host thread keeps `inflight` proofs queued (b2g_prove_submit / b2g_prove_wait, one Context each):
                # every step still uploads its witness from pinned host memory and reads its 256 proof bytes back
                pend, submitted, done, last = [None] * inflight, 0, 0, None
                def submit(j):
                    return Groth16.submit(pk, R_FIX, S_FIX, cm, wl.wms[j], ctxs[j])
                for j in range(min(inflight, total)):
                    pend[j] = submit(j); submitted += 1
                while done < total:
                    j = done % inflight
                    last = pend[j].wait(); done += 1
                    if submitted < total:
                        pend[j] = submit(j); submitted += 1
                return last
            def worker(i):
                last = None
                for _ in range(total // inflight + (1 if i < total % inflight else 0)):
                    last = one_proof(i)
                return last
            res = list(pool.map(worker, range(inflight)))
            return res[0]

        t0 = time.time()
        proofs = [one_proof(i) for i in range(inflight)]                 # loads the key (tables) on first use
        log(f"[bench] rank {rank} {mode} 2^{wl.log_n}: key load + first proofs {time.time() - t0:.1f}s")
        assert all(p_.data == proofs[0].data for p_ in proofs)
        run_steps(max(warmup, inflight))
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        launches0 = ctxs[0].launch_count()
        t0 = time.perf_counter()
        proof = run_steps(steps)                                          # e2e: host witness in, proof bytes out, every step
        barrier()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        launches = ctxs[0].launch_count() - launches0
        res = {"mode": mode, "proof": proof, "launches": launches, "e2e_s": e2e_s, "ctxs": ctxs, "inflight": inflight,
               "host_driver": ("one host thread, b2g_prove_submit/wait" if use_async else f"{inflight} host threads, synchronous b2g_prove") + "; one captured CUDA graph launch per proof",
               "host_ms_last_proof": {k: v for k, v in ctxs[0].last_timings().items() if k.startswith('host_') or k in ('h2d', 'total')}}
        per_step = world if mode == 'replicas' else 1                    # replicas: every rank proves its own copy
        res["e2e_value"] = per_step * steps / e2e_s
        if not sharded:
            # device-resident: witness already in HBM, the same number of proofs in flight, every context's proofs queued back to
            # back.  Timed over ONE window common to all contexts - from an idle, synchronised device to an idle, synchronised
            # device - because per-context CUDA-event windows start and end at different moments and their maximum under-counts
            # the span (it produced rates above the multiplier-pipe bound with 6 contexts).
            per = [steps // inflight + (1 if i < steps % inflight else 0) for i in range(inflight)]
            barrier()
            t0 = time.perf_counter()
            for k in range(steps):                                        # round-robin over the contexts, like the e2e loop
                ctxs[k % inflight].bench_device(pk, cm, -1)               # enqueue only (one graph launch per proof), no wait
            torch.cuda.synchronize()
            dev_local = time.perf_counter() - t0
            dev_s = max_over_ranks(dev_local)
            log(f"[bench] rank {rank} {mode}: device-resident window {dev_local * 1e3:.1f} ms for {steps} proofs ({inflight} contexts)")
            barrier()
            res["value"] = per_step * steps / dev_s
            res["latency_ms"] = ctxs[0].bench_device(pk, cm, 5)
            barrier()
        else:
            res["value"] = res["e2e_value"]
            t0 = time.perf_counter()
            dev_lat = []
            for _ in range(5):
                one_proof(0)
                dev_lat.append(ctxs[0].last_timings()['total'])       # CUDA events: first upload byte -> proof bytes back, this rank
            barrier()
            res["latency_ms"] = max_over_ranks((time.perf_counter() - t0) / 5 * 1e3)     # host wall clock per proof (includes host jitter of the slowest rank)
            res["device_latency_ms"] = max_over_ranks(sorted(dev_lat)[len(dev_lat) // 2])  # on the device, median of 5, max over ranks
        res["clocks"] = sampler.stop() if rank == 0 else None
        pool.shutdown()
        if fused:
            # per-phase CUDA-event times of the same sharded proof issued WITHOUT the captured graph (the graph has no interior
            # events): a second context per rank, wired to its peers the same way; collective, so every rank takes part
            os.environ['B2G_GRAPH'] = '0'
            try:
                cx = Context(local, rank, world)
            finally:
                os.environ.pop('B2G_GRAPH', None)
            cx.prepare(pk, cm)
            sharding.connect_p2p(cx, dist)
            dist.barrier()
            for _ in range(3):
                Groth16.prove_sharded_p2p(pk, cm, R_FIX, S_FIX, wl.wms[0], cx)
            res["phase_ms_one_proof_alone"] = cx.last_timings()
            dist.barrier()
            cx.close()
        return res

    def phase_table(wl, sharded):
        """per-phase CUDA-event times of one proof issued WITHOUT the captured graph (the graph has no interior events)"""
        os.environ['B2G_GRAPH'] = '0'
        try:
            cx = Context(local, rank if sharded else 0, world if sharded else 1)
        finally:
            os.environ.pop('B2G_GRAPH', None)
        if sharded:
            Groth16.prove_partial(wl.pk, wl.cm, wl.wms[0], cx, R_FIX, S_FIX)
            Groth16.prove_partial(wl.pk, wl.cm, wl.wms[0], cx, R_FIX, S_FIX)
        else:
            for _ in range(2):
                Groth16.create_proof_with_reduction_and_matrices(wl.pk, R_FIX, S_FIX, wl.cm, wl.circ.num_inputs, wl.circ.num_constraints, wl.wms[0], cx)
        t = cx.last_timings()
        cx.close()
        return t

    inflight = max(1, args.inflight)
    wl = Workload(args.log_n, args.workload, inflight)
    main_mode = 'single' if world == 1 else args.mode
    main = measure(wl, main_mode, args.steps, args.warmup, inflight)
    proof = main["proof"]                                                 # the last step of the timed e2e loop
    ctx = main["ctxs"][0]
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, proof.data)

    if rank == 0 and not args.skip_check:
        wl.check_closed_form(proof)
        log("[bench] proof matches the trapdoor closed form (h-independent) and the witness map matches the trapdoor")

    roof, extra = None, {}
    if rank == 0:
        peak, how = measured_peaks()
        shard_div = world if main_mode == 'sharded' else 1
        pk, cm = wl.pk, wl.cm
        # dominant kernel group: the bucket accumulation of one G1 MSM (H query: n = domain bases / scalars), run alone
        msm_ms, acc_ms = ctx.bench_msm(pk, cm, 0, 5)
        alg = pk.domain_size // shard_div * 96.0
        prof = static_kernel_profile() or {}
        roof = {"bound": "hbm", "kernel": "G1 bucket accumulation (H query): " + prof.get("g1_kernels", "msm_accumulate_kernel<G1>"),
                "achieved": alg / (acc_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                "frac": alg / (acc_ms * 1e-3) / 1e9 / peak, "traffic": (prof.get("g1_dram_bytes_per_launch") or 0) / shard_div or None, "peak_source": how,
                "algorithmic_bytes": alg, "kernel_ms": acc_ms, "whole_msm_ms": msm_ms,
                "traffic_source": "static: " + prof.get("source", "no committed ncu summary (profiles/kernel_profile.json missing)"),
                "note": "254-bit Pippenger is bound by the IMAD.WIDE (fmaheavy) pipe, not by HBM (DESIGN.md section 5)"}
        if prof.get("g1_fmaheavy_pct") and args.log_n == prof.get("log_n") and shard_div == 1:
            # the binding roofline: the integer multiply-add ("fmaheavy") pipe.  Utilisation is a static ncu fact of the kernel
            # (sm__pipe_fmaheavy_cycles_active), rescaled by ncu-time / live CUDA-event time of this run
            frac = prof["g1_fmaheavy_pct"] / 100.0 * (prof["g1_time_us_ncu"] * 1e-3) / acc_ms
            roof["int_pipe"] = {"bound": "IMAD.WIDE issue (fmaheavy pipe)", "frac": frac, "static_pct_ncu": prof["g1_fmaheavy_pct"],
                                "static_kernel_us_ncu": prof["g1_time_us_ncu"], "source": "static: " + prof.get("source", "")}
        g2_ms, g2_acc = ctx.bench_msm(pk, cm, 4, 3)
        extra["msm_g2"] = {"whole_msm_ms": g2_ms, "kernel_ms": g2_acc, "algorithmic_gbs": (pk.n_vars - 1) / shard_div * 160.0 / (g2_acc * 1e-3) / 1e9}
        extra["single_proof_latency_ms"] = main["latency_ms"]
    for c_ in main["ctxs"]:
        c_.close()
    if rank == 0:
        extra["phase_ms_one_proof_alone"] = main.get("phase_ms_one_proof_alone") if main_mode == 'sharded' else phase_table(wl, False)

    other = None
    if world > 1 and not args.one_mode:
        other_mode = 'sharded' if main_mode == 'replicas' else 'replicas'
        o_ = measure(wl, other_mode, args.steps, args.warmup, inflight)
        assert o_["proof"].data == proof.data, "sharded and whole proofs differ"
        other = {"mode": other_mode, "value": o_["value"], "e2e_value": o_["e2e_value"], "unit": "proofs/s", "latency_ms": o_["latency_ms"],
                 "device_latency_ms": o_.get("device_latency_ms"),
                 "scaling": "strong" if other_mode == 'sharded' else "weak", "gpu_launches": o_["launches"], "in_flight": o_["inflight"],
                 "exchange": args.exchange if other_mode == 'sharded' else None}
        for c_ in o_["ctxs"]:
            c_.close()
        if other_mode == 'sharded':
            other["phase_ms_one_proof_alone"] = o_.get("phase_ms_one_proof_alone")

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:     # the CPU leg is reported at N = 1 only
        pin_cpu_arm()
        from oracle import cref
        cref.build()
        cores = physical_cores()
        za = oracle_key(wl.pk, wl.cm)
        t0 = time.perf_counter()
        ref = cref.prove(za, R_FIX, S_FIX, wl.wm_np, nthreads=cores)
        dt = time.perf_counter() - t0
        assert ref == proof.data, "GPU proof bytes differ from the CPU oracle's"
        log(f"[bench] CPU oracle proof identical to the GPU proof; {dt:.2f}s on {cores} threads")
        cpu = {"value": 1.0 / dt, "unit": "proofs/s", "cores": cores, "kind": "port",
               "sample": "1 full proof of the same workload (same key, witness, r, s), oracle/cref.c C+OpenMP restatement of the ark-groth16 0.5 CPU path, one pinned thread per core; proof bytes asserted identical",
               "phases_s": cref.last_phase_seconds(), "cpu_model": cpu_model(), "nproc": os.cpu_count()}

    cfg = workload_config(args, wl.circ)
    n_vars = wl.circ.n_vars

    # BASELINE.json config 4: 2^22-constraint chain, MSM bases sharded by range over the N GPUs
    config4 = None
    if world > 1 and not args.no_config4:
        release_all()
        del wl
        wl4 = Workload(22, 'chain', 1)
        m4 = measure(wl4, 'sharded', args.steps4, 2, 1)
        if rank == 0:
            if not args.skip_check:
                wl4.check_closed_form(m4["proof"])
                log("[bench] 2^22 sharded proof matches the trapdoor closed form (h-independent)")
            config4 = {"workload": "circom squaring chain, domain 2^22 (n_vars=4194304), MSM bases sharded by range over %d GPUs" % world,
                       "value": m4["value"], "unit": "proofs/s", "latency_ms": m4["latency_ms"], "device_latency_ms": m4.get("device_latency_ms"),
                       "steps": args.steps4, "in_flight": 1,
                       "exchange": args.exchange, "gpu_launches": m4["launches"], "scaling": "strong",
                       "checked": None if args.skip_check else "proof == trapdoor closed form (no h involved)"}
        for c_ in m4["ctxs"]:
            c_.close()
        if rank == 0:
            config4["phase_ms_one_proof_alone"] = m4.get("phase_ms_one_proof_alone")

    if rank == 0:
        sharded = main_mode == 'sharded'
        value = main["value"]
        per_step = world if main_mode == 'replicas' else 1
        parallelism = "single GPU" if world == 1 else (f"MSM base-range sharding over {world} GPUs; 768 B partials exchanged " + ("inside the proof graph over NVLink peer memory" if args.exchange == 'p2p' else "with one NCCL all-gather")
                                                       if sharded else f"{world} replicas (one whole prover per GPU)")
        out = {"metric": METRIC, "value": value, "unit": "proofs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": 1e3 / value * per_step, "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None,
               "dtype": "u32x8 (254-bit Montgomery integers)", "data": "synthetic", "config": cfg, "parallelism": parallelism, "in_flight": main["inflight"],
               "clocks": main["clocks"],
               "e2e": {"value": main["e2e_value"], "unit": "proofs/s", "h2d_bytes_per_step": n_vars * 32 + 64 + (768 * world if sharded and args.exchange != 'p2p' else 0),
                       "d2h_bytes_per_step": 256 + (768 * (world + 1) if sharded and args.exchange != 'p2p' else 0), "ms_per_step": 1e3 * main["e2e_s"] / args.steps,
                       "host_driver": main["host_driver"], "host_ms_last_proof": main["host_ms_last_proof"]},
               "gpu_launches": main["launches"], "roofline": roof, "cpu_baseline": cpu}
        out.update(extra)
        if other:
            out["other_mode"] = other
        if config4:
            out["config4"] = config4
        emit(out)
    release_all()
    setup_ctx.close()
    if dist is not None:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(obj):
    """the ONE JSON line, on the process's real stdout (libraries such as NCCL print banners to fd 1)"""
    line = (json.dumps(obj) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, line)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                       # anything else written to fd 1 goes to stderr
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=None)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--log-n', type=int, default=20)
    ap.add_argument('--workload', default='chain', choices=['chain', 'circomlike'])
    ap.add_argument('--mode', default='replicas', choices=['sharded', 'replicas'], help='N>1: headline mode (the other one is measured too, see other_mode)')
    ap.add_argument('--exchange', default='p2p', choices=['p2p', 'nccl'], help='sharded mode: partials folded from NVLink peer memory inside the kernels (p2p) or gathered with one NCCL all-gather (nccl)')
    ap.add_argument('--one-mode', action='store_true', help='N>1: measure only --mode')
    ap.add_argument('--no-config4', action='store_true', help='N>1: skip the 2^22 base-sharded leg (BASELINE.json config 4)')
    ap.add_argument('--steps4', type=int, default=5, help='timed proofs of the 2^22 leg')
    ap.add_argument('--inflight', type=int, default=3, help='proofs in flight per GPU (one Context + host thread each)')
    ap.add_argument('--host-driver', default='async', choices=['async', 'threads'], help="e2e loop: one host thread with b2g_prove_submit/wait (async) or one thread per in-flight proof")
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--skip-check', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the proof of the last timed step as DIR/proof_{a,b,c}.npy')
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 3 if args.impl == 'reference' else 20
    if args.warmup is None:
        args.warmup = 1 if args.impl == 'reference' else 3
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
