#!/usr/bin/env python
"""bench.py -- benchmark of the B200-native Kaiju classification path.

Metric (BASELINE.json): read items/s (one item = one output line; a pair counts once) for 150 bp paired reads, MEM mode
-m 11 (default SEG on), against a viruses-scale .fmi, at N = 1/2/4/8 B200 -- next to the reference CPU `kaiju -z <best>`.

Headline workload (configs[1]): 10 M synthetic PE150 pairs per GPU per step (SURVEY.md 8d recipe, tools/kjgen.c, seeded) against the
"synth-viruses" stand-in (680 k proteins, ~2e8 letters; the real kaiju_db_viruses.fmi needs a download), whose .fmi is built here with
the reference's own kaiju-mkbwt/kaiju-mkfmi (-e 3).  A "step" is one pass of the hot path over the rank's batch.

  value      : whole-job items/s with reads resident in HBM (kj_classify_device2), CUDA-event timed, max over ranks
  e2e        : same metric through kj_classify2() with pinned HOST buffers (H2D of bases+offsets and D2H of results inside)
  roofline   : algorithmic bytes of the REFERENCE algorithm per launch (instrumented oracle on a sample of the same reads,
               SURVEY.md 8d) / kernel time, against the measured HBM peak in MEASURED_PEAKS.json
  cpu_baseline: the unmodified reference binary (oracle/_ref/kaiju) on a bounded sample, `-z` swept over {16, 32, 64, nproc},
               best point reported; its output on the sample is compared read by read with the GPU's (`parity`)
  configs    : (N = 1 only) the other BASELINE.json configurations in the same run, each with value / e2e / roofline / cpu_baseline / parity:
               greedy      = configs[2]: `-a greedy -e 3 -s 65` on the same 10 M pairs
               large_index = configs[3]: MEM on a refseq_ref-scale index (2.7e10 BWT rows, ~126 GB in HBM): the index of the collection
                             in which every synth-viruses protein occurs K times, built on the device by kj_create_scaled (the
                             reference's index builder cannot produce 2.7e10 rows inside a benchmark run; K-fold == what
                             kaiju-mkbwt builds for the K-fold FASTA, tests/test_gpu_build.py); results must equal the base index's

Multi-GPU: one process per GPU (torchrun), index replicated, reads sharded (weak scaling), ONE NCCL all-gather of the per-read dense
taxon indices (uint32) per step on a side stream, overlapped with the next step; `strong_scaling` = the 10 M-pair job split over N.
`--impl reference`: the CPU reference alone (no product library is loaded), same sweep, value = best `-z`.
"""
import argparse, json, os, subprocess, sys, tempfile, threading, time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="mem", choices=["mem", "greedy"], help="mode of the headline line (default: MEM)")
    ap.add_argument("--nprot", type=int, default=680000, help="synthetic DB size (680000 = viruses scale)")
    ap.add_argument("--reads", type=int, default=10_000_000, help="read pairs per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs for the CPU baseline sample (0 = auto)")
    ap.add_argument("--workdir", default=os.environ.get("KJ_BENCH_DIR", os.path.join(tempfile.gettempdir(), "kjbench")))
    ap.add_argument("--skip-cpu", action="store_true", help="no CPU legs (roofline numerator, cpu_baseline, parity)")
    ap.add_argument("--headline-only", action="store_true", help="skip the `configs` sub-runs (greedy, large_index)")
    ap.add_argument("--large-rows", type=float, default=2.7e10, help="target BWT rows of the large_index config (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline device-resident path returned in its last timed step to DIR/<name>.npy (float64, a seeded "
                         "sample of this rank's reads; with several GPUs also a sample of the all-gathered dense taxon indices of every rank)")
    return ap.parse_args()


DUMP_SAMPLE = 1 << 20          # reads in a --dump-outputs sample: at most 6 arrays x 8 bytes x 2^20 = 48 MB


def dump_outputs(R, directory):
    """Per-read results of the last timed device-resident step of the headline configuration (kj_classify_device2): taxon id, best
    match length/score and dense taxon index, for a fixed seeded sample of the reads (all of them if the batch is small enough), with
    the sampled read indices.  With several GPUs, also a seeded sample of the all-gathered dense indices of every rank's reads (the
    job's whole output).  float64 holds every value exactly (ids and indices < 2^53)."""
    os.makedirs(directory, exist_ok=True)
    def sample(n):
        return np.arange(n, dtype=np.int64) if n <= DUMP_SAMPLE else np.sort(np.random.default_rng(12345).choice(n, DUMP_SAMPLE, replace=False))
    idx = sample(R.n)
    out = {"read_index": idx, "taxon": R.kept["taxon"].cpu().numpy().view(np.uint64)[idx], "best": R.kept["best"].cpu().numpy().view(np.uint32)[idx],
           "dense_taxon_index": R.kept["dense_taxon_index"].cpu().numpy().view(np.uint32)[idx]}
    if R.kept["gathered"] is not None:
        g = R.kept["gathered"].cpu().numpy().view(np.uint32); gidx = sample(len(g))
        out.update({"all_ranks_read_index": gidx, "all_ranks_dense_taxon_index": g[gidx]})
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a.astype(np.float64))


def build_workload(args, rank):
    """DB + index (rank 0 builds, others wait); returns (SynthDB, fmi, nodes)."""
    from helpers import SynthDB, build_fmi
    d = os.path.join(args.workdir, "db_%d" % args.nprot); os.makedirs(d, exist_ok=True)
    fmi, nodes, done = d + "/db.fmi", d + "/nodes.dmp", d + "/.done"
    db = SynthDB(args.nprot, 1)
    if rank == 0 and not os.path.exists(done):
        db.write(d + "/db.faa", nodes)
        build_fmi(d + "/db.faa", d + "/db", threads=min(64, os.cpu_count() or 8))
        os.remove(d + "/db.faa")
        open(done, "w").write("ok")
    while not os.path.exists(done):
        time.sleep(0.5)
    return db, fmi, nodes


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True); self.index = index; self.rows = []; self.stop_flag = False

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=5).stdout.decode().strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(float(r[0])) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(len(r) > col and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(float(self.rows[0][1])) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------------- reference CPU legs
def ref_cmd(fmi, nodes, mode, a, b, z, out):
    from helpers import REF_DIR
    c = [os.path.join(REF_DIR, "kaiju"), "-t", nodes, "-f", fmi, "-i", a, "-j", b, "-a", mode, "-m", "11", "-z", str(z), "-o", out]
    return c + (["-e", "3", "-s", "65"] if mode == "greedy" else [])


def ref_timed(fmi, nodes, mode, fq, tiny, z, out):
    """Classification rate of the unmodified reference on the FASTQ pair `fq`; the index load is excluded with the two-size
    differential T(n) - T(tiny) (BASELINE.md section 3.4).  Returns seconds of classification."""
    t = time.time(); subprocess.check_call(ref_cmd(fmi, nodes, mode, tiny[0], tiny[1], z, out + ".tiny"), stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL); t_load = time.time() - t
    t = time.time(); subprocess.check_call(ref_cmd(fmi, nodes, mode, fq[0], fq[1], z, out), stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL); t_all = time.time() - t
    try:
        os.remove(out + ".tiny")
    except OSError:
        pass
    return max(t_all - t_load, 1e-3)


def z_points(cores):
    return sorted({z for z in (16, 32, 64, cores) if 1 <= z <= cores} or {cores})


def ref_sweep(db, fmi, nodes, mode, args, seed, n_full, keep_output):
    """BASELINE.md 3.3: `-z` swept (on a quarter of the sample), the best point re-run on the full sample.  Returns the cpu_baseline
    object and, if keep_output, the path of the reference's output for the full sample (first n_full pairs of stream `seed`)."""
    cores = os.cpu_count() or 1
    d = tempfile.mkdtemp(prefix="kjcpu_", dir=args.workdir)
    n_sw = max(20000, n_full // 4)
    fq = (d + "/r1.fq", d + "/r2.fq"); sw = (d + "/s1.fq", d + "/s2.fq"); tiny = (d + "/t1.fq", d + "/t2.fq")
    db.write_fastq(seed, 0, n_full, 150, True, fq[0], fq[1]); db.write_fastq(seed, 0, n_sw, 150, True, sw[0], sw[1]); db.write_fastq(seed, 0, 16, 150, True, tiny[0], tiny[1])
    points = {}
    for z in z_points(cores):
        points[z] = n_sw / ref_timed(fmi, nodes, mode, sw, tiny, z, d + "/sw.tsv")
    best_z = max(points, key=points.get)
    dt = ref_timed(fmi, nodes, mode, fq, tiny, best_z, d + "/out.tsv")
    for f in fq + sw + tiny + (d + "/sw.tsv",):
        try:
            os.remove(f)
        except OSError:
            pass
    cb = {"value": n_full / dt, "unit": "read pairs/s", "cores": cores, "threads_used": best_z, "kind": "reference",
          "sweep": {"-z %d" % z: round(v, 1) for z, v in sorted(points.items())}, "sweep_sample": n_sw,
          "sample": "first %d pairs of the same workload, oracle/_ref/kaiju -a %s -z %d (best of the sweep), %.1f s, index load excluded by differential" % (n_full, mode, best_z, dt)}
    out = d + "/out.tsv"
    if not keep_output:
        os.remove(out); out = None
    return cb, out


def parse_ref_output(path, n):
    """taxon id per read index from the reference's output file (lines `C/U <tab> r<i> <tab> taxid`)."""
    import pandas as pd
    df = pd.read_csv(path, sep="\t", header=None, usecols=[1, 2], names=["name", "tax"], dtype={"name": str, "tax": np.uint64}, engine="c")
    idx = df["name"].str.slice(1).astype(np.int64).to_numpy()
    tax = np.zeros(n, dtype=np.uint64); seen = np.zeros(n, dtype=bool)
    tax[idx] = df["tax"].to_numpy(); seen[idx] = True
    assert seen.all() and len(idx) == n, "reference output does not cover the sample"
    return tax


def emit(line):
    """The ONE JSON line of the contract goes to the real stdout; everything else printed by libraries (NCCL's version banner,
    build output) was diverted to stderr in main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def reference_arm(args):
    """--impl reference: the unmodified reference on the host cores; nothing of kaiju_b200/ is imported or loaded."""
    db, fmi, nodes = build_workload(args, 0)
    cores = os.cpu_count() or 1
    # a step = a bounded sample of the workload; all steps together ~10 M pairs of CPU work (about a minute at the reference's best -z on 128 vCPUs)
    n_sample = args.cpu_sample or max(20000, min(2560000, 20000 * cores, 10_000_000 // max(1, args.warmup + args.steps)))
    cb, _ = ref_sweep(db, fmi, nodes, args.mode, args, 1000, n_sample, False)          # untimed: finds the best -z
    z = cb["threads_used"]; vals = []
    for s in range(args.warmup + args.steps):
        d = tempfile.mkdtemp(prefix="kjref_", dir=args.workdir)
        fq = (d + "/r1.fq", d + "/r2.fq"); tiny = (d + "/t1.fq", d + "/t2.fq")
        db.write_fastq(1001 + s, 0, n_sample, 150, True, fq[0], fq[1]); db.write_fastq(1001 + s, 0, 16, 150, True, tiny[0], tiny[1])
        dt = ref_timed(fmi, nodes, args.mode, fq, tiny, z, d + "/out.tsv")
        for f in fq + tiny + (d + "/out.tsv",):
            try:
                os.remove(f)
            except OSError:
                pass
        if s >= args.warmup:
            vals.append(dt)
    v = n_sample * len(vals) / sum(vals)
    cb.update({"value": v, "sample": "%d pairs per step, kaiju -z %d (best of the sweep), index load excluded by differential" % (n_sample, z)})
    line = {"impl": "reference", "metric": "reads/sec (150 bp paired, %s mode, synth-viruses .fmi)" % args.mode.upper(), "value": v, "unit": "read pairs/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * sum(vals) / len(vals),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": "configs[1]: %s -m 11, synthetic PE150 pairs vs synth-viruses .fmi (%d proteins); bounded sample of %d pairs per step" % (args.mode.upper(), args.nprot, n_sample)},
            "cpu_baseline": cb, "e2e": {"value": v, "unit": "read pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ---------------------------------------------------------------------------------------------------- B200 arm
class Runner:
    """Reads of one rank (pinned host + device copies) and the timed loops over one Classifier."""

    def __init__(self, torch, dist, world, local, s1, o1, s2, o2):
        self.torch, self.dist, self.world = torch, dist, world
        self.n = len(o1) - 1; self.np_in = (s1, o1, s2, o2)
        pin = lambda a: torch.from_numpy(a.view(np.int64) if a.dtype == np.uint64 else a).pin_memory()
        self.h = [pin(x) for x in (s1, o1, s2, o2)]
        self.d = [x.cuda(non_blocking=True) for x in self.h]
        n = self.n
        self.d_tax = torch.zeros(n, dtype=torch.int64, device="cuda"); self.d_best = torch.zeros(n, dtype=torch.int32, device="cuda")
        self.h_tax = torch.zeros(n, dtype=torch.int64).pin_memory(); self.h_best = torch.zeros(n, dtype=torch.int32).pin_memory()
        # dense taxon indices (uint32 as int32 storage), double-buffered: the gather of step i overlaps the kernel of step i+1
        self.d_compact = [torch.zeros(n, dtype=torch.int32, device="cuda") for _ in range(2)]
        self.gathered = [torch.zeros(n * world, dtype=torch.int32, device="cuda") for _ in range(2)] if dist else None
        # the gather runs on a high-priority stream: when the classify kernel of step i retires, the few CTAs of the NCCL kernel must get their SM slots
        # before the persistent grid of step i+1 takes all of them (otherwise the gather sits behind that whole kernel and step i+2 waits for its buffer)
        self.stream = torch.cuda.current_stream(); self.side = torch.cuda.Stream(priority=-1) if dist else None
        self.gather_done = [None, None]; self.i = 0
        self.in_bytes = int(s1.nbytes + s2.nbytes + o1.nbytes + o2.nbytes)
        torch.cuda.synchronize()

    def _gather(self, k):
        torch = self.torch
        if os.environ.get("KJ_BENCH_GATHER_MAIN"):      # developer hook (A/B): the gather behind the kernel on the same stream
            self.dist.all_gather_into_tensor(self.gathered[k], self.d_compact[k])
            done = torch.cuda.Event(); done.record(self.stream); self.gather_done[k] = done
            return
        ev = torch.cuda.Event(); ev.record(self.stream)
        with torch.cuda.stream(self.side):
            self.side.wait_event(ev)
            self.dist.all_gather_into_tensor(self.gathered[k], self.d_compact[k])
            done = torch.cuda.Event(); done.record(self.side)
        self.gather_done[k] = done

    def step_device(self, clf):
        k = self.i & 1; self.i += 1; self.last_k = k
        if self.dist and self.gather_done[k] is not None:
            self.stream.wait_event(self.gather_done[k])                # buffer k is free again once its previous gather has finished
        d = self.d
        clf.classify_device2(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), self.n, self.d_tax.data_ptr(), self.d_best.data_ptr(),
                             self.d_compact[k].data_ptr(), 150, 150, self.stream.cuda_stream)
        if self.dist:
            self._gather(k)

    def step_host(self, clf):
        k = self.i & 1; self.i += 1
        if self.dist and self.gather_done[k] is not None:
            self.gather_done[k].synchronize()
        h = self.h
        clf.classify2_ptrs(h[0].data_ptr(), h[1].data_ptr(), h[2].data_ptr(), h[3].data_ptr(), self.n, self.h_tax.data_ptr(), self.h_best.data_ptr(), self.d_compact[k].data_ptr())
        if self.dist:
            self._gather(k)

    def timed(self, clf, fn, steps, warmup):
        torch, dist = self.torch, self.dist
        for _ in range(warmup):
            fn(clf)
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()
        ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
        l0 = clf.kernel_launches
        t0 = time.perf_counter(); ev0.record(self.stream)
        for _ in range(steps):
            fn(clf)
        if dist:
            self.stream.wait_stream(self.side)                         # the last gathers belong to the timed region
        ev1.record(self.stream); torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if dist:
            dist.barrier()
        ms = ev0.elapsed_time(ev1)
        if fn == self.step_host:
            ms = wall * 1000.0           # host-buffer path runs on the library's own streams: wall clock bracketed by synchronize
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), clf.kernel_launches - l0


def measure(R, clf, steps, warmup, world, keep=False):
    """value (device-resident) and e2e (host buffers) of one configuration on runner R, `steps` timed steps each.  keep: R.kept = the
    device outputs of the last device-resident step (untimed copies, taken before the e2e leg reuses the buffers)."""
    ms_dev, launches = R.timed(clf, R.step_device, steps, max(3, warmup))
    if keep:
        k = R.last_k
        R.kept = {"taxon": R.d_tax.clone(), "best": R.d_best.clone(), "dense_taxon_index": R.d_compact[k].clone(),
                  "gathered": R.gathered[k].clone() if R.dist else None}
        R.torch.cuda.synchronize()
    kernel_ms = clf.last_kernel_ms                                   # CUDA events around the last classify kernel, on its launch stream
    e2e_steps = steps
    ms_host, _ = R.timed(clf, R.step_host, e2e_steps, 1)
    clf.check_errors()
    assert R.torch.equal(R.h_tax, R.d_tax.cpu()), "host-buffer and device-buffer entry points disagree"
    total = R.n * world
    return {"value": total * steps / (ms_dev / 1000.0), "ms_per_step": ms_dev / steps, "kernel_ms": kernel_ms, "gpu_launches": int(launches),
            "e2e": {"value": total * e2e_steps / (ms_host / 1000.0), "unit": "read pairs/s", "h2d_bytes_per_step": R.in_bytes, "d2h_bytes_per_step": int(R.n * 12),
                    "note": "kj_classify2() with pinned host buffers, chunked H2D/kernel/D2H pipeline inside"}}


def peak_hbm():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        if "hbm_gbs" in peaks:
            return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        pass
    return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def cpu_legs(R, res, mode, db, fmi, nodes, args, n_or=20000):
    """Rank 0, N = 1: roofline numerator from the instrumented oracle, oracle check, reference sweep + parity on the CPU sample."""
    from helpers import Oracle, make_params, KoCounters
    s1, o1, s2, o2 = R.np_in; n = R.n; tax = R.h_tax.numpy().view(np.uint64)
    ctr = KoCounters(); orc = Oracle(fmi, nodes)
    t = time.time(); otax, _ = orc.classify_batch(make_params(mode), s1[:int(o1[n_or])], o1[:n_or + 1], s2[:int(o2[n_or])], o2[:n_or + 1], ctr); t_or = time.time() - t
    assert np.array_equal(otax, tax[:n_or]), "GPU result differs from the oracle on the bench workload (%s)" % mode
    c = ctr.as_dict()
    alg = (c["fmindex"] * 10 + c["scanned_bytes"] + c["lf_steps"] * 11 + c["get_suffix"] * 6 + c["bases"] + 8 * n_or) / n_or   # SURVEY.md 8d definition
    peak, peak_src = peak_hbm()
    ach = alg * n / (res["kernel_ms"] / 1000.0) / 1e9
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum per item from the latest `ncu --set full` capture (profiles/traffic.json)
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[mode]["dram_bytes_per_item"] * n
    except Exception:
        pass
    res["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                       "algorithmic_bytes_per_item": alg, "peak_source": peak_src,
                       "note": "numerator = reference algorithm's bytes (instrumented oracle, %d-pair sample) x items per launch; kernel time from CUDA events on the launch stream" % n_or}
    cores = os.cpu_count() or 1
    n_cpu = args.cpu_sample or max(20000, min(2560000 if mode == "mem" else 1280000, (20000 if mode == "mem" else 10000) * cores))
    n_cpu = min(n_cpu, n)
    cb, out = ref_sweep(db, fmi, nodes, mode, args, 7, n_cpu, True)
    rtax = parse_ref_output(out, n_cpu); os.remove(out)
    diffs = int((rtax != tax[:n_cpu]).sum())
    cb["oracle_port_value"] = n_or / t_or
    res["cpu_baseline"] = cb
    res["parity"] = {"parity_sample": n_cpu, "diffs": diffs, "against": "unmodified reference binary, read by read (= sort-equal, BASELINE.md 3.6)", "oracle_sample": n_or, "oracle_diffs": 0}
    assert diffs == 0, "GPU taxa differ from the reference binary on the CPU sample (%s): %d of %d" % (mode, diffs, n_cpu)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1); os.dup2(2, 1)          # fd 1 -> stderr for the rest of the process; emit() writes to the saved descriptor
    args = parse()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":                     # CPU only, rank 0 only; the product library is neither built nor loaded here
        if rank == 0:
            reference_arm(args)
        return

    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    import torch
    import kaiju_b200 as kb
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")      # NCCL's own stream as well (see Runner)
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    db, fmi, nodes = build_workload(args, rank)
    if dist:
        dist.barrier()
    clf = kb.Classifier(fmi, nodes, device=local, params=kb.make_params(args.mode, m=11))
    n = args.reads
    R = Runner(torch, dist, world, local, *db.reads(7, rank * n, n, 150, True))      # this rank's shard of the job: items [rank*n, (rank+1)*n)

    sampler = ClockSampler(local); sampler.start()
    res = measure(R, clf, args.steps, args.warmup, world, keep=bool(args.dump_outputs))
    sampler.stop_flag = True; sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(R, args.dump_outputs)
    # untimed: the kaiju2table-style summary -- per-taxon read counts in HBM, one all-reduce across the ranks (SURVEY.md 8e); and the
    # dense indices the ranks gathered map back to the 64-bit ids
    clf.counts_reset(); clf.counts_add_device(R.d_tax.data_ptr(), n); torch.cuda.synchronize()
    if dist:
        from kaiju_b200.sharding import all_reduce_counts
        all_reduce_counts(None, dist, clf); torch.cuda.synchronize()
    ids_c, cnt_c = clf.counts()
    assert int(cnt_c.sum()) == n * world, "per-taxon counts do not add up to the number of reads"
    cid = clf.compact_ids(); comp = R.d_compact[(R.i - 1) & 1].cpu().numpy().view(np.uint32)
    mapped = np.where(comp == 0xffffffff, np.uint64(0), cid[np.minimum(comp, len(cid) - 1)])
    assert np.array_equal(mapped, R.h_tax.numpy().view(np.uint64)), "dense taxon indices do not map back to the taxon ids"
    if dist:
        g = R.gathered[(R.i - 1) & 1].cpu().numpy().view(np.uint32)
        assert np.array_equal(g[rank * n:(rank + 1) * n], comp), "all-gathered taxon indices do not contain this rank's shard"

    strong = None
    if dist:   # strong scaling: the 10 M-pair job of ONE GPU split over the ranks (reads [0, n) of the same stream)
        lo, hi = rank * n // world, (rank + 1) * n // world
        RS = Runner(torch, dist, world, local, *db.reads(7, lo, hi - lo, 150, True))
        ms_s, _ = RS.timed(clf, RS.step_device, args.steps, 2)
        strong = {"value": n * args.steps / (ms_s / 1000.0), "unit": "read pairs/s", "total_pairs": n, "note": "fixed job of %d pairs split over %d GPUs, device-resident, gather included" % (n, world)}
        del RS

    line = None
    if rank == 0:
        line = {"metric": "reads/sec (150 bp paired, %s mode, synth-viruses .fmi)" % args.mode.upper(), "value": res["value"], "unit": "read pairs/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                "config": {"workload": "configs[1]: %s -m 11 (SEG on), %d synthetic PE150 pairs per GPU per step vs synth-viruses .fmi (%d proteins, bwtlen %d)" % (args.mode.upper(), n, args.nprot, clf.bwtlen),
                           "parallelism": "read-sharded x%d, index replicated, NCCL all-gather of uint32 dense taxon indices per step on a side stream" % world if world > 1 else "single GPU",
                           "l2": "inputs (%.1f GB/step) and index (%.2f GB) exceed the 126 MB L2" % (R.in_bytes / 1e9, clf.index_bytes / 1e9),
                           "launch": dict(zip(("grid", "block", "dyn_smem"), clf.launch_geometry)),
                           "index_build_ms": clf.index_build_ms,
                           "per_taxon_counts": "%d taxa with reads, counts sum to %d reads (untimed; all-reduce over %d rank(s))" % (len(ids_c) - 1, int(cnt_c.sum()), world)},
                "e2e": res["e2e"], "gpu_launches": res["gpu_launches"], "clocks": sampler.summary(), "kernel_ms": res["kernel_ms"]}
        if strong:
            line["strong_scaling"] = strong
    if world == 1 and not args.skip_cpu:
        cpu_legs(R, res, args.mode, db, fmi, nodes, args)
        for k in ("roofline", "cpu_baseline", "parity"):
            line[k] = res[k]

    # ------------------------------------------------------------------ the other BASELINE.json configurations (N = 1)
    if world == 1 and not args.headline_only:
        cfgs = {}
        other = "greedy" if args.mode == "mem" else "mem"
        mem_tax = R.h_tax.numpy().view(np.uint64).copy() if args.mode == "mem" else None
        try:
            clf.set_params(kb.make_params(other, m=11))
            sub = measure(R, clf, args.steps, 3, 1)
            sub.update({"workload": "configs[2]: %s -e 3 -s 65 -m 11 (E-value 0.01, SEG on), the same %d PE150 pairs vs synth-viruses .fmi" % (other.upper(), n) if other == "greedy" else "MEM -m 11"})
            if not args.skip_cpu:
                cpu_legs(R, sub, other, db, fmi, nodes, args)
            cfgs[other] = sub
            if other == "mem":
                mem_tax = R.h_tax.numpy().view(np.uint64).copy()
        except Exception as e:   # a failed sub-configuration must not take the headline line with it
            cfgs[other] = {"error": repr(e)}
        if args.large_rows > 0:
            try:
                alg = (line.get("roofline") or cfgs.get("mem", {}).get("roofline") or {}).get("algorithmic_bytes_per_item") if args.mode == "mem" else (cfgs.get("mem", {}).get("roofline") or {}).get("algorithmic_bytes_per_item")
                cfgs["large_index"] = large_index(kb, torch, R, clf, fmi, nodes, mem_tax, args, local, alg)
            except Exception as e:
                cfgs["large_index"] = {"error": repr(e)}
        line["configs"] = cfgs
    if rank == 0:
        emit(line)
    if dist:
        dist.destroy_process_group()


def large_index(kb, torch, R, clf_base, fmi, nodes, mem_tax, args, local, alg_base):
    """configs[3]: MEM against a refseq_ref-scale index resident in HBM (see the module docstring)."""
    clf_base.set_params(kb.make_params("mem", m=11))       # (a context that leaves Greedy mode returns its record buffers: HBM for the large index)
    free, total = torch.cuda.mem_get_info()
    copies = max(2, int(round(args.large_rows / clf_base.bwtlen)))
    per_row = 3.5 + 8.0 / 12 + 4.0 / 8 + 0.05                        # rank records + packed letters + taxon per sampled row (exponent 3) (+ slack)
    while copies > 2 and copies * clf_base.bwtlen * per_row > free - (6 << 30):
        copies -= 1
    t0 = time.time()
    big = kb.Classifier(fmi, nodes, device=local, params=kb.make_params("mem", m=11), copies=copies)
    t_create = time.time() - t0
    try:
        sub = measure(R, big, args.steps, 3, 1)
        tax = R.h_tax.numpy().view(np.uint64)
        diffs = int((tax != mem_tax).sum()) if mem_tax is not None else None
        peak, peak_src = peak_hbm()
        sub.update({"workload": "configs[3]: MEM -m 11, the same %d PE150 pairs vs a refseq_ref-scale index: synth-viruses x %d copies = %d BWT rows, %.1f GB resident in HBM (64-bit interval kernels, 192-row rank records)"
                                % (R.n, copies, big.bwtlen, big.index_bytes / 1e9),
                    "index": {"bwt_rows": big.bwtlen, "sequences": big.nseq, "hbm_bytes": big.index_bytes, "device_build_ms": big.index_build_ms, "create_s": t_create,
                              "built_by": "kj_create_scaled on the device from the 2e8-row .fmi (no host transcode, no suffix sort)"},
                    "parity": {"parity_sample": R.n, "diffs": diffs, "against": "results on the base index (every copy carries the taxon of its original, so MEM results must be identical); the base results are checked against the oracle and the reference binary"}})
        if alg_base:
            ach = alg_base * R.n / (sub["kernel_ms"] / 1000.0) / 1e9
            sub["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "algorithmic_bytes_per_item": alg_base, "peak_source": peak_src,
                               "note": "numerator = the reference algorithm's bytes per item on the BASE index (a lower bound: on the K-fold collection the reference resolves up to K times as many suffix-array rows per match)"}
        assert diffs in (0, None), "results on the scaled index differ from the base index: %s" % diffs
        return sub
    finally:
        big.close()


if __name__ == "__main__":
    main()
