#!/usr/bin/env python
"""Turn the artefacts of tools/gpu_round2.sh (gpurun_out/) into the small tracked files under profiles/.

    python tools/collect_profiles.py r02b

Needs the `ncu` CLI (no GPU).  Writes <tag>_bench.json, <tag>_bench_reference.json, <tag>_launches.txt, <tag>_k_*.txt,
<tag>_k_pair_fast_lines.txt, <tag>_k_shell_grid_lines.txt, <tag>_k_pair_fast_sass.txt, <tag>_k_pair_fast_meta.json,
<tag>_files_timeline.{txt,json}, peaks_b200.json.
"""
import csv
import io
import json
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "gpurun_out")
PROF = os.path.join(ROOT, "profiles")


def run(cmd):
    return subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, cwd=ROOT).stdout


def raw(rep):
    rows = list(csv.reader(io.StringIO(run(["ncu", "-i", rep, "--page", "raw", "--csv"]))))
    return dict(zip(rows[0], rows[2]))


def last_json(path):
    for line in reversed(open(path).read().strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise ValueError(path)


def main(tag):
    cp = lambda a, b: shutil.copy(os.path.join(OUT, a), os.path.join(PROF, b))
    cp("bench_full.json", f"{tag}_bench.json")
    cp("bench_full_reference.json", f"{tag}_bench_reference.json")
    cp("peaks.json", "peaks_b200.json")
    cp("files_timeline.txt", f"{tag}_files_timeline.txt")
    cp("files_timeline.json", f"{tag}_files_timeline.json")
    open(os.path.join(PROF, f"{tag}_launches.txt"), "w").write(run([sys.executable, "tools/ncu_summary.py", "launches", "gpurun_out/launches.csv"]))
    for rep, name in (("prof_pair_fast", "k_pair_fast"), ("prof_pair", "k_pair_f64"), ("prof_msd", "k_msd_single"), ("prof_shell", "k_shell_grid"),
                      ("prof_fft", "k_fft_pass"), ("prof_flux", "k_charge_flux"), ("prof_dump", "k_dump_rows")):
        p = os.path.join(OUT, rep + ".ncu-rep")
        if os.path.exists(p):
            open(os.path.join(PROF, f"{tag}_{name}.txt"), "w").write(run([sys.executable, "tools/ncu_summary.py", "kernel", p]))
    for rep, name in (("prof_pair_fast", "k_pair_fast"), ("prof_shell", "k_shell_grid")):
        open(os.path.join(PROF, f"{tag}_{name}_lines.txt"), "w").write(run([sys.executable, "tools/ncu_lines.py", os.path.join(OUT, rep + ".ncu-rep")]))
    # SASS of the headline instantiation
    lib = os.path.join(ROOT, "mdproptools_b200", "libmdprop_b200.so")
    names = [l.split()[-1] for l in run(["cuobjdump", "-elf", lib]).splitlines() if ".text." in l and "k_pair_fast" in l]
    sym = sorted({n.split(".text.")[-1] for n in names if "ILb0ELb1ELb0EE" in n})
    if sym:
        sass = run(["cuobjdump", "-sass", "-fun", sym[0], lib])
        open(os.path.join(PROF, f"{tag}_k_pair_fast_sass.txt"), "w").write(sass)
    # instruction count per evaluated pair of the two captures (16 C2 frames per launch)
    fast, f64 = raw(os.path.join(OUT, "prof_pair_fast.ncu-rep")), raw(os.path.join(OUT, "prof_pair.ncu-rep"))
    bf, b64 = last_json(os.path.join(OUT, "ncu_pair_fast.log")), last_json(os.path.join(OUT, "ncu_pair.log"))
    num = lambda d, k: float(d[k].replace(",", ""))
    meta = {
        "kernel": "k_pair_fast<0,1,0>", "capture": "ncu --set full, bench.py --frames 16 (one launch = 16 C2 frames)", "frames": 16,
        "evaluated_pairs": bf["evaluated_pair_evals_per_step"], "inst_executed": num(fast, "smsp__inst_executed.sum"),
        "duration_ms": num(fast, "gpu__time_duration.sum") / (1e6 if num(fast, "gpu__time_duration.sum") > 1e4 else 1),
        "issue_active_pct": round(num(fast, "smsp__issue_active.avg.pct_of_peak_sustained_active"), 2),
        "warp_instr_per_32_pairs": round(num(fast, "smsp__inst_executed.sum") / (bf["evaluated_pair_evals_per_step"] / 32.0), 2),
        "all_fp64_kernel": {
            "kernel": "k_pair<0,0,1,0>", "evaluated_pairs": b64["evaluated_pair_evals_per_step"],
            "inst_executed": num(f64, "smsp__inst_executed.sum"),
            "duration_ms": num(f64, "gpu__time_duration.sum") / (1e6 if num(f64, "gpu__time_duration.sum") > 1e4 else 1),
            "warp_instr_per_32_pairs": round(num(f64, "smsp__inst_executed.sum") / (b64["evaluated_pair_evals_per_step"] / 32.0), 2)},
    }
    json.dump(meta, open(os.path.join(PROF, f"{tag}_k_pair_fast_meta.json"), "w"), indent=1)
    print(json.dumps(meta, indent=1))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "r02b")
