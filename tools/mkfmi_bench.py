#!/usr/bin/env python
"""Index construction on the GPU (kaiju_b200.build_index) against the reference's kaiju-mkbwt + kaiju-mkfmi, on synthetic protein DBs.

    python tools/mkfmi_bench.py [--inputs small,large,dup] [--no-ref] [--out result.json]

Inputs (tools/kjgen.c, seeded): small = SynthDB(400000, 7), about 1.2e8 residues; large = about 1e9 residues; dup = SynthDB(100000, 7)
with every protein written 8 times under different taxa.  For each input one JSON line: the GPU build's wall time by stage, its sort
rounds with the suffixes sorted per round, the bytes the sort kernels moved over the sort time, and -- unless --no-ref -- the wall time
of `kaiju-mkbwt -n <cores> -e 3` + `kaiju-mkfmi` (oracle/_ref) on the same FASTA and whether the two .fmi files are byte-identical.
The first line names the GPU and its power limit.  Files go to a temporary directory (--workdir, default $TMPDIR)."""
import argparse, json, os, random, shutil, subprocess, sys, tempfile, time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
REF = os.path.join(ROOT, "oracle", "_ref")
SIZES = {"small": 400000, "large": 3300000}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,driver_version", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, driver = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "driver": driver}
    except Exception as e:          # noqa: BLE001 -- the numbers are still useful without the card's name
        return {"gpu": "unknown (%s)" % e}


def write_input(kind, d):
    from helpers import SynthDB
    faa, nodes = os.path.join(d, kind + ".faa"), os.path.join(d, kind + ".nodes.dmp")
    if kind in SIZES:
        SynthDB(SIZES[kind], 7).write(faa, nodes)
        return faa
    base = os.path.join(d, "dup_base.faa")
    SynthDB(100000, 7).write(base, nodes)
    taxa = [l.split("\t")[0] for l in open(nodes)]
    rnd = random.Random(8)
    with open(base) as f, open(faa, "w") as g:
        recs = f.read().split(">")[1:]
        for i, r in enumerate(recs):
            seq = r.split("\n", 1)[1]
            for k in range(8):
                g.write(">D%d_%d_%s\n%s" % (i, k, rnd.choice(taxa), seq))
    os.remove(base)
    return faa


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--inputs", default="small,large,dup")
    ap.add_argument("--no-ref", action="store_true")
    ap.add_argument("--threads", type=int, default=os.cpu_count())
    ap.add_argument("--exponent", type=int, default=3)
    ap.add_argument("--workdir", default=None)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import kaiju_b200 as kb
    lines = [dict(gpu_info(), host_cores=os.cpu_count())]
    print(json.dumps(lines[0]), flush=True)
    d = tempfile.mkdtemp(prefix="kjmkfmi_", dir=a.workdir)
    try:
        for kind in a.inputs.split(","):
            faa = write_input(kind, d)
            r = {"input": kind, "faa_bytes": os.path.getsize(faa)}
            kb.build_index(faa, os.path.join(d, "warm"), exponent=a.exponent)        # CUDA context + module load outside the timing
            t = time.perf_counter()
            st = kb.build_index(faa, os.path.join(d, "gpu"), exponent=a.exponent)
            r["gpu_wall_s"] = time.perf_counter() - t
            r.update(st)
            r["sort_GBps"] = st["sort_bytes"] / (st["sort_ms"] * 1e6) if st["sort_ms"] > 0 else None
            if not a.no_ref:
                t = time.perf_counter()
                subprocess.check_call([os.path.join(REF, "kaiju-mkbwt"), "-n", str(a.threads), "-e", str(a.exponent), "-a", "ACDEFGHIKLMNPQRSTVWY",
                                       "-o", os.path.join(d, "ref"), faa], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                r["ref_mkbwt_s"] = time.perf_counter() - t
                t = time.perf_counter()
                subprocess.check_call([os.path.join(REF, "kaiju-mkfmi"), os.path.join(d, "ref")], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                r["ref_mkfmi_s"] = time.perf_counter() - t
                r["ref_threads"] = a.threads
                r["fmi_identical"] = subprocess.call(["cmp", "-s", os.path.join(d, "gpu.fmi"), os.path.join(d, "ref.fmi")]) == 0
            for f in os.listdir(d):
                if not f.endswith(".nodes.dmp"):
                    os.remove(os.path.join(d, f))
            lines.append(r)
            print(json.dumps(r), flush=True)
    finally:
        shutil.rmtree(d, ignore_errors=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
