#!/usr/bin/env python
"""bench.py — field gates evaluated / second on BASELINE.json's headline config (C3):
a synthetic 2^24-gate Add/Mul/AssertZero circuit over the BLS12-381 scalar field (255-bit),
a batch of 4096 independent witnesses sharded across N B200s (one process per GPU).

One "step" = one satisfiability check of the whole batch against the relation.
  value : whole-job gate-evaluations / s with the witness batch already resident in HBM
  e2e   : the same through the C ABI call `zkb_evaluate` with HOST (pinned) witness buffers:
          H2D of the witnesses + all kernels + D2H of the verdicts inside the timed region
  --impl reference : the CPU restatement of the reference's evaluator (oracle/plaintext_flat.c;
          the Rust binary cannot be built in this image) on all host threads, bounded sample.
Relation flattening / levelization / program upload is one-off preparation, reported as prep_s.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2-gates", type=int, default=24)
    ap.add_argument("--witnesses", type=int, default=4096)
    ap.add_argument("--inputs", type=int, default=1024)
    ap.add_argument("--field", default="bls381", choices=["bls381", "bn254", "goldilocks", "p124", "m31"])
    ap.add_argument("--cpu-sample-log2-gates", type=int, default=0,
                    help="cap the CPU arms at the relation's first 2^k counted gates (0: the whole relation when the time budget allows)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-value-check", action="store_true", help="skip the sampled wire-value comparison with the oracle")
    ap.add_argument("--verdicts-only", action="store_true",
                    help="do not keep the live wires readable: slot re-use + dead-store elimination (not the headline)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float64): every witness's verdict and "
                         "the values of a fixed, seeded sample of wires x witnesses, so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    return args


FIELD = {"bls381": 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001,
         "bn254": 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001,
         "goldilocks": (1 << 64) - (1 << 32) + 1,
         "p124": 16249742125730185677094195492597105093,      # 4 limbs (the modulus of evaluator.rs:956)
         "m31": (1 << 31) - 1}                                 # 1 limb
SEED = 0x5EED0003


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.samples)}


def load_circuits():
    """the workload generator (numpy only), imported by path: the reference arm must not load libzkb.so"""
    import importlib.util
    if "zkb_circuits" in sys.modules:
        return sys.modules["zkb_circuits"]
    spec = importlib.util.spec_from_file_location("zkb_circuits", os.path.join(ROOT, "zkinterface-ir_b200", "circuits.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["zkb_circuits"] = mod
    spec.loader.exec_module(mod)
    return mod


def host_threads():
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        pass
    return max(1, min(n, 64))


def counted_prefix(circ_mod, circuit, n_counted_gates):
    """the first gates of the relation that hold `n_counted_gates` counted gates (Add / Mul / AssertZero)"""
    g = circuit.gates
    if n_counted_gates >= circuit.n_gates:
        return g, circuit.n_gates
    counted = np.isin(g["op"], [circ_mod.G_ADD, circ_mod.G_MUL, circ_mod.G_ASSERT_ZERO])
    cum = np.cumsum(counted)
    cut = int(np.searchsorted(cum, n_counted_gates, side="left")) + 1
    return g[:cut], int(cum[cut - 1])


def cpu_reference_run(circ_mod, flat, p, circuit, gates, n_counted, witnesses, n_threads):
    """one pass of the oracle (restatement of Evaluator<PlaintextBackend>, oracle/plaintext_flat.c) over `gates` for
    len(witnesses) witnesses on n_threads threads (the reference itself is single-threaded: one witness per thread is
    the data-parallel CPU figure); returns (gate-evals/s, seconds, results)"""
    eb = circ_mod.elem_bytes(p)
    n = len(witnesses)
    t0 = time.perf_counter()
    res = flat.eval_batch(gates, circuit.const_pool, p.to_bytes(eb, "little"), None, witnesses, n, n_threads=n_threads)
    dt = time.perf_counter() - t0
    return n_counted * n / dt, dt, res


DUMP_WIRES = 4096          # wire-value sample of --dump-outputs: 4096 wires x 16 witnesses, 4 MB at 8 limbs
DUMP_WITNESSES = 16


def dump_outputs(out_dir, be, circuit, ff, w_np, corrupt_local, eb, wires_readable):
    """--dump-outputs: the verdicts of the whole batch (first_fail_seq = -1 for a satisfied witness) and, when the wires are
    kept readable, the values of a seeded sample of wires for a seeded sample of this rank's satisfied witnesses, as
    little-endian u32 limbs [witness, wire, limb]; float64 holds every verdict and limb exactly"""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "verdict_ok.npy"), (ff >= (1 << 40)).astype(np.float64))
    np.save(os.path.join(out_dir, "first_fail_seq.npy"), np.where(ff >= (1 << 40), -1, ff).astype(np.float64))
    if not wires_readable:
        return
    rng = np.random.default_rng(SEED + 11)
    nw = circuit.n_wires
    wires = np.sort(rng.choice(nw, size=min(DUMP_WIRES, nw), replace=False))
    good = np.array([j for j in range(len(w_np)) if j not in corrupt_local])
    picks = np.sort(rng.choice(good, size=min(DUMP_WITNESSES, len(good)), replace=False))
    handles = [be.scope_lookup(int(i)) for i in wires]
    vals = np.zeros((len(picks), len(wires), eb), dtype=np.uint8)
    for r, j in enumerate(picks):
        vals[r] = [np.frombuffer(x.to_bytes(eb, "little"), np.uint8) for x in be.read_values(int(j), handles, eb)]
    np.save(os.path.join(out_dir, "wire_values.npy"), vals.view("<u4").astype(np.float64))


def workload_name(args):
    return (f"C3: 2^{args.log2_gates}-gate random Add/Mul/AssertZero circuit over {args.field}, "
            f"{args.witnesses} witnesses sharded over {args.gpus} GPU(s)")


def main():
    args = parse()
    # stdout carries exactly ONE line, the JSON: anything a library prints on fd 1 while the job runs (NCCL's version
    # banner, build chatter) is routed to stderr, and fd 1 is restored just before the line is printed
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    p = FIELD[args.field]
    n_gates = 1 << args.log2_gates

    import importlib
    if args.impl != "reference":
        import __graft_entry__ as ge
        import zkb_loader
        if world == 1:
            ge.build()

    if args.impl == "reference":
        if rank != 0:
            return
        # the reference's own CPU implementation of the path, timed on this box's host cores.  The Rust binary cannot
        # be built in this image (no cargo / rustc, crates not vendored), so this is the C restatement that keeps the
        # reference's structure (oracle/plaintext_flat.c).  libzkb.so is NOT loaded in this arm.
        circ_mod = load_circuits()
        from oracle import flat
        flat.build()
        circuit = circ_mod.random_circuit(n_gates, args.inputs, p, SEED)
        nt = host_threads()
        # every step = the relation's first 2^k counted gates x one witness per host thread; k is the largest that keeps
        # the whole (warmup + steps) run within ~3 minutes at ~2 M gates/s/thread (the full relation when it fits)
        budget_s = 170.0 / max(1, args.steps + args.warmup)
        k = args.log2_gates
        while k > 16 and (1 << k) / 2.0e6 > budget_s:
            k -= 1
        if args.cpu_sample_log2_gates:
            k = min(k, args.cpu_sample_log2_gates)
        gates, n_counted = counted_prefix(circ_mod, circuit, 1 << k)
        w = circ_mod.make_witnesses(circuit, nt, seed=SEED + 99)
        times = []
        for it in range(args.warmup + args.steps):
            rate, dt, res = cpu_reference_run(circ_mod, flat, p, circuit, gates, n_counted, w, nt)
            assert (res["status"] == 0).all(), "oracle found an unsatisfied witness in the baseline sample"
            if it >= args.warmup:
                times.append(dt)
        per_step = float(np.mean(times))
        rate = n_counted * nt / per_step
        sample = (f"{'the whole relation' if n_counted == circuit.n_gates else 'first ' + str(n_counted) + ' counted gates of the relation'}"
                  f" ({circuit.n_gates} gates) x {nt} witnesses, one per host thread, per step")
        line = {
            "impl": "reference", "metric": "field gates evaluated/sec", "value": rate, "unit": "gate-evals/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32x8 (255-bit field)",
            "data": "synthetic",
            "config": {"workload": workload_name(args), "gates": circuit.n_gates, "gate_histogram": circuit.hist,
                       "witnesses": args.witnesses, "witness_inputs": circuit.n_inputs},
            "cpu_baseline": {"value": rate, "unit": "gate-evals/s", "cores": nt, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "gate-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU restatement of zki_sieve 3.0.0 Evaluator<PlaintextBackend> (oracle/plaintext_flat.c: hash-map wire "
                    "store, heap big integers, generic long division), not the Rust binary; the reference is single-threaded, "
                    "this is one witness per host thread",
        }
        emit(line)
        return

    # keep stdout to the one JSON line: NCCL prints its version banner there when NCCL_DEBUG=VERSION
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        if rank == 0:          # one rank (re)builds if needed; the others load the library only afterwards
            ge.build()
        dist.barrier()
    z = zkb_loader.load()
    circ_mod = importlib.import_module("zkir_b200.circuits")

    # ---- one-off preparation: relation -> levelized device program ---------------------------
    # N > 1: the relation is recorded and levelized ONCE, on rank 0; the other ranks receive the device plan over NCCL
    # (zkb_comm_broadcast_program, include/zkb.h section 7) and never see the relation.
    t0 = time.perf_counter()
    circuit = circ_mod.random_circuit(n_gates, args.inputs, p, SEED)
    t_gen = time.perf_counter() - t0
    be = z.GpuBackend(local_rank)
    if world > 1:
        cid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            cid.copy_(torch.frombuffer(bytearray(z.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(cid, 0)                       # plumbing: the id reaches the peers through the launcher's group
        be.comm_init_rank(bytes(cid.cpu().numpy().tobytes()), world, rank)
        dist.barrier()
    t0 = time.perf_counter()
    if rank == 0:
        be.set_field(p)
        be.push_gates(circuit.gates, circuit.const_pool)
        be.finalize(keep_all_values=False, verdicts_only=args.verdicts_only)
    t_prep = time.perf_counter() - t0
    t_bcast = 0.0
    if world > 1:
        t0 = time.perf_counter()
        be.comm_broadcast_program(0)
        t_bcast = time.perf_counter() - t0
    st = be.stats()

    # ---- this rank's shard of the witness batch (contiguous block) ---------------------------
    total_w = args.witnesses
    shard = importlib.import_module("zkir_b200.sharding")
    lo, hi = shard.shard_range(total_w, rank, world)
    n_local = hi - lo
    # 1 % of the witnesses are corrupted; their first failing assertion is known by construction
    rng = np.random.default_rng(SEED + 1)
    bad = rng.choice(total_w, size=max(1, total_w // 100), replace=False)
    corrupt_global = {int(j): int(rng.integers(0, max(circuit.n_tracked, 1))) for j in bad} if circuit.n_tracked else {}
    corrupt_local = {j - lo: k for j, k in corrupt_global.items() if lo <= j < hi}
    w_np = circ_mod.make_witnesses(circuit, n_local, seed=SEED + 7 + rank, corrupt=corrupt_local)
    eb = circ_mod.elem_bytes(p)
    w_pinned = torch.empty(w_np.shape, dtype=torch.uint8, pin_memory=True)
    w_pinned.numpy()[...] = w_np
    w_host = w_pinned.numpy()
    expected = circ_mod.expected_first_fail(circuit, n_local, corrupt_local)

    def first_fail_vector(v):
        return np.where(v["ok"] == 1, np.int64(1) << 40, v["first_fail_seq"].astype(np.int64))

    def check(ff_local):
        got = np.where(ff_local >= (1 << 40), -1, ff_local)[:n_local]
        assert (got == expected).all(), f"rank {rank}: verdicts differ from the constructed expectation"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    gate_evals_local = circuit.n_gates * n_local
    gate_evals_total = circuit.n_gates * total_w

    def timed(fn, steps):
        """device time of a step = the library's CUDA events on its own stream: (H2D,) kernels, the verdict MIN all-reduce
        (ncclAllReduce inside libzkb, the path's only collective), verdict D2H; max over ranks."""
        barrier()
        dev_ms = 0.0
        lv_ms = 0.0
        t0 = time.perf_counter()
        for _ in range(steps):
            v = fn()
            tm = be.timing()
            dev_ms += tm["total_ms"]
            lv_ms += tm["levels_ms"]
        barrier()
        wall = time.perf_counter() - t0
        t = torch.tensor([dev_ms, wall * 1e3, lv_ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t[0].item(), t[1].item(), t[2].item(), first_fail_vector(v), v

    if world > 1:       # every rank receives the verdicts of the WHOLE batch
        run_resident = lambda: be.comm_run(lo, total_w)                                   # noqa: E731
        run_e2e = lambda: be.comm_evaluate(None, w_host, n_local, lo, total_w)            # noqa: E731
    else:
        run_resident = be.run
        run_e2e = lambda: be.evaluate(None, w_host, n_local)                              # noqa: E731

    # ---- value: inputs resident in HBM -----------------------------------------------------------
    be.upload_inputs(None, w_host, n_local)
    st = be.stats()
    for _ in range(args.warmup):
        run_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dev_ms, wall_ms, lv_ms, ff, v = timed(run_resident, args.steps)
    check(ff[lo:hi])
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, be, circuit, ff, w_np, corrupt_local, eb, not args.verdicts_only)
    launches = be.timing()["kernel_launches"] * args.steps
    level_launches = be.timing()["level_launches"]
    ms_per_step = dev_ms / args.steps
    value = gate_evals_total / (ms_per_step * 1e-3)

    # ---- e2e: host buffers through the C ABI --------------------------------------------------------
    for _ in range(min(args.warmup, 2)):
        run_e2e()
    e_dev_ms, e_wall_ms, _, ff2, v2 = timed(run_e2e, args.steps)
    sampler.stop_flag = True
    e2e_ms = max(e_dev_ms, 0.0) / args.steps
    e2e_value = gate_evals_total / (e2e_ms * 1e-3)
    check(ff2[lo:hi])
    if world > 1:
        n_false = int((ff2 < (1 << 40)).sum())
        assert n_false == len(corrupt_global), (n_false, len(corrupt_global))

    # ---- roofline of the dominant kernel (k_level<8,false>) ----------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    algo_bytes_step = st["algo_bytes_per_witness"] * n_local            # this rank
    lv_ms_step = lv_ms / args.steps
    achieved = algo_bytes_step / (lv_ms_step * 1e-3) / 1e9 if lv_ms_step > 0 else 0.0
    # launch_level's rule (csrc/kernels.cu): full 256-lane tiles of an 8-limb field take the bulk-copy ring kernel
    tma = eb == 32 and st["tile_witnesses"] == 256 and os.environ.get("ZKB_LEVEL_TMA", "1") != "0"
    kernel_name = "k_level_tma<8>" if tma else f"k_level_pipe<{max(1, eb // 4)}>"
    roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_bytes_step / max(level_launches, 1),
                "avg_launch_ms": lv_ms_step / max(level_launches, 1), "launches_per_step": level_launches,
                "bytes_per_gate_eval": st["algo_bytes_per_witness"] / circuit.n_gates}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            tj = json.load(open(prof))
            ratio = tj["traffic_over_algorithmic"]
            roofline["traffic"] = ratio * roofline["algorithmic_bytes_per_launch"]
            roofline["traffic_source"] = (f"profiles/traffic.json ({tj.get('capture', '?')}): dram__bytes_read+write of 3 captured "
                                          f"level launches = {ratio:.3f} x their algorithmic bytes, scaled to the average launch")
            roofline["dram_frac"] = roofline["frac"] * ratio
            roofline["note"] = ("frac counts ALGORITHMIC bytes (3E per two-input gate, E per assertion) and can exceed 1: "
                                f"{(1 - ratio) * 100:.1f} % of them never reach DRAM (operands read twice inside a wavefront hit L2, "
                                "fused-assert-only values are not stored); dram_frac = measured DRAM traffic / copy peak")
        except Exception:
            pass

    # ---- parity at the headline shape (every run): sampled wire values of three witnesses — the first, one across the
    # first tile boundary, the last — against the oracle's evaluation of the whole relation; the oracle is the checker here
    values_checked = 0
    value_witnesses = []
    if rank == 0 and not args.no_value_check and not args.verdicts_only:
        from concurrent.futures import ThreadPoolExecutor
        from oracle import flat
        tile_w = st["tile_witnesses"]
        good = [j for j in range(n_local) if j not in corrupt_local]
        picks = sorted({good[0], min((j for j in good if j >= tile_w), default=good[len(good) // 2]), good[-1]})
        nw = circuit.n_wires
        wires = np.unique(np.concatenate([np.linspace(0, nw - 1, 12000).astype(np.int64), np.arange(max(0, nw - 1000), nw),
                                          np.arange(min(64, nw))]))
        handles = [be.scope_lookup(int(i)) for i in wires]
        mod_le = p.to_bytes(eb, "little")
        with ThreadPoolExecutor(len(picks)) as ex:
            dumps = list(ex.map(lambda j: flat.eval_dump(circuit.gates, circuit.const_pool, mod_le, None, w_np[j], nw, stride=eb), picks))
        for j, (res, dump) in zip(picks, dumps):
            assert int(res["status"]) == flat.EV_TRUE, f"oracle: witness {j} is not satisfying"
            got = be.read_values(j, handles, eb)
            want = [int.from_bytes(dump[i].tobytes(), "little") for i in wires]
            bad_at = [int(wires[q]) for q in range(len(wires)) if got[q] != want[q]]
            assert not bad_at, f"witness {lo + j}: {len(bad_at)} wire values differ from the oracle, first at wire {bad_at[0]}"
            values_checked += len(wires)
            value_witnesses.append(lo + j)
        del dumps

    # ---- CPU baseline beside it (rank 0, N = 1): the oracle over the WHOLE relation, 1 core (the reference is
    # single-threaded) and one witness per host thread; its verdicts double as a check of ours for those witnesses
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import flat
        nt = host_threads()
        try:    # the restatement's hash-map wire store takes ~0.2 KB per live wire and thread
            avail = int([l for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0].split()[1]) * 1024
            nt = max(1, min(nt, int(avail * 0.6 / (circuit.n_wires * 200 + 1))))
        except Exception:
            pass
        gates_cpu, n_counted = counted_prefix(circ_mod, circuit, 1 << args.cpu_sample_log2_gates if args.cpu_sample_log2_gates else circuit.n_gates)
        whole = n_counted == circuit.n_gates
        rate1, dt1, res1 = cpu_reference_run(circ_mod, flat, p, circuit, gates_cpu, n_counted, w_np[:1], 1)
        rate, dt, res = cpu_reference_run(circ_mod, flat, p, circuit, gates_cpu, n_counted, w_np[:nt], nt)
        if whole:
            for j in range(min(nt, n_local)):
                ok_ref = int(res[j]["status"]) == flat.EV_TRUE
                assert ok_ref == (expected[j] < 0) and (ok_ref or int(res[j]["fail_assert_seq"]) == expected[j]), \
                    f"witness {j}: the oracle's verdict differs from the device's"
        what = "the whole relation" if whole else f"first {n_counted} counted gates of the relation"
        cpu_baseline = {"value": rate, "unit": "gate-evals/s", "cores": nt, "kind": "port",
                        "sample": f"{what} ({circuit.n_gates} gates) x {nt} witnesses, one per host thread, {dt:.1f} s",
                        "seconds": dt, "one_core": {"value": rate1, "seconds": dt1, "sample": f"{what} x 1 witness, 1 thread"},
                        "verdicts_checked_against_oracle": min(nt, n_local) if whole else 0,
                        "what": "C restatement of zki_sieve 3.0.0 Evaluator<PlaintextBackend> (oracle/plaintext_flat.c), gate loop only "
                                "(no .sieve parsing); the Rust binary cannot be built in this image"}

    if rank == 0:
        line = {
            "metric": "field gates evaluated/sec", "value": value, "unit": "gate-evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u32x8 (255-bit field, Montgomery)" if eb == 32 else f"u32x{eb // 4}",
            "data": "synthetic",
            "config": {"workload": workload_name(args),
                       "gates": circuit.n_gates, "gate_histogram": circuit.hist, "witnesses": total_w,
                       "witness_inputs": circuit.n_inputs, "levels": st["n_levels"], "tile_witnesses": st["tile_witnesses"],
                       "tiles_per_rank": st["n_tiles"], "wire_store_gb": st["n_slots"] * eb * st["tile_witnesses"] / 1e9,
                       "l2": "working set (wire store) is >> L2, no flush needed", "parallelism": f"witness-shard x{world}",
                       "wires_kept_readable": "none (verdicts only)" if args.verdicts_only else "all live top-scope wires"},
            "e2e": {"value": e2e_value, "unit": "gate-evals/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int(w_host.nbytes) * world, "d2h_bytes_per_step": (4 * total_w + 4) * world},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "clocks": sampler.summary(),
            "prep_s": {"generate_circuit": t_gen, "flatten_levelize_upload": t_prep, "program_broadcast": t_bcast,
                       "note": "levelized once on rank 0; the peers receive the device plan over NCCL (zkb_comm_broadcast_program)"},
            "wall_ms_per_step": wall_ms / args.steps,
            "verdicts": {"true": int((ff >= (1 << 40)).sum()), "false": int((ff < (1 << 40)).sum()),
                         "checked": "all, against the generator's expectation (1 % corrupted, first failing assertion known)"},
            "values_checked": values_checked,
            "values_checked_witnesses": value_witnesses,
        }
        emit(line)
    be.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
