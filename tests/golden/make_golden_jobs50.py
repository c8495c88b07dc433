#!/usr/bin/env python
"""Whole-search counts of 50-job Taillard instances as the reference's own sequential C program prints them when it
is built with MAX_JOBS 50 (baselines/pfsp/lib/PFSP_node.h:10, the C twin of `config param MAX_JOBS`,
lib/pfsp/PFSP_node.chpl:7) -> tests/golden/pfsp_jobs50_counts.json.

oracle/Makefile keeps a scratch copy of the reference's PFSP sources with that one line rewritten under
oracle/_ref/jobs50/ (`make -C oracle ref`).  This script links those sources into the unmodified program in a
temporary directory and runs it with --ub 1, where the counts do not depend on the exploration order: the sequential
program's tree / solutions / optimum are also those of the offload driver, whatever its chunk sizes or GPU count.

Only searches that finish on a CPU are listed (most 50-job searches run for hours): ta032 / ta037 / ta038 with lb1
and lb2.  No lb1_d count: lb1_d reads min_heads, where the C program and the Chapel program differ (SURVEY.md
Appendix A.1) — with the Chapel statement ta031 / ta041 / ta051 prune every child of the root, with the C line the
same searches run for longer than ten minutes.
Run in the build container only (needs the reference):  make -C oracle ref && python tests/golden/make_golden_jobs50.py
"""
import json
import os
import re
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
J50 = os.path.join(ROOT, "oracle", "_ref", "jobs50")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pfsp_jobs50_counts.json")
SEARCHES = [(32, 1), (37, 1), (38, 1), (32, 2), (37, 2), (38, 2)]


def build(exe):
    pf = os.path.join(J50, "pfsp")
    src = [os.path.join(pf, "pfsp_c.c")] + [os.path.join(pf, "lib", f) for f in
                                            ("c_taillard.c", "c_bound_simple.c", "c_bound_johnson.c", "PFSP_node.c",
                                             "Pool.c")] + [os.path.join(J50, "commons", "util.c")]
    subprocess.run(["gcc", "-O3", "-w", "-o", exe] + src + ["-lm"], check=True)


def run(exe, inst, lb):
    txt = subprocess.run([exe, "--inst", str(inst), "--lb", str(lb), "--ub", "1"], capture_output=True, text=True,
                         cwd=tempfile.gettempdir(), timeout=300, check=True).stdout
    assert "n = 50)" in txt, txt
    g = lambda pat: int(re.search(pat, txt).group(1))  # noqa: E731
    return {"tree": g(r"explored tree: (\d+)"), "sol": g(r"explored solutions: (\d+)"), "best": g(r"makespan: (\d+)")}


def main():
    if not os.path.exists(os.path.join(J50, ".stamp")):
        raise SystemExit("oracle/_ref/jobs50 is missing: run `make -C oracle ref` first")
    out = {"_source": "the reference's sequential C program (baselines/pfsp/pfsp_c.c) built from oracle/_ref/jobs50, "
                      "i.e. with MAX_JOBS 50; --ub 1",
           "pfsp": {}}
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "pfsp_c50.out")
        build(exe)
        for inst, lb in SEARCHES:
            out["pfsp"][f"ta{inst:03d}_lb{lb}_ub1"] = run(exe, inst, lb)
    json.dump(out, open(OUT, "w"), indent=1)
    print("wrote", OUT, out["pfsp"])


if __name__ == "__main__":
    main()
