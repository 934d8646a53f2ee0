#!/usr/bin/env python3
"""Regenerate profiles/ptxas_and_sass_census.md (per-kernel registers / spills / smem from
`nvcc -Xptxas -v`, census of the interesting SASS mnemonics from `cuobjdump -sass`) AND the full
listings docs/sass/<file>.sm_100a.sass of the sources in LISTINGS, from one compile of every kernel
source with the Makefile's flags. Needs only the CUDA toolkit (no GPU)."""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = ["src/kernels/copy_kernels.cu", "src/kernels/update_kernels.cu", "src/kernels/update_rows_kernels.cu",
           "src/kernels/model_kernels.cu", "src/kernels/engine_kernels.cu"]
# update_rows_kernels.cu is summarised in the census only: its twelve instantiations would add a 1.6 MB
# listing (`cuobjdump -sass build/src/kernels/update_rows_kernels.o` prints it)
LISTINGS = {"src/kernels/copy_kernels.cu", "src/kernels/update_kernels.cu", "src/kernels/model_kernels.cu",
            "src/kernels/engine_kernels.cu"}
INTERESTING = re.compile(r"^(F2FP|LDG|STG|ST\.E|LD\.E|LDGMC|REDG|ATOMG|MEMBAR|MUFU\.(RCP|SQRT|EX2)|SYNCS|UBLKCP|UTMA|UTC)")
HEADER = (
    "# ptxas -v summary and SASS mnemonic census of every sm_100a kernel in src/kernels\n"
    "Generated on the build host (no GPU needed) by `scripts/sass_census.py` with "
    "`nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -Xptxas -v` and `cuobjdump -sass` (CUDA 12.9). "
    "No kernel spills; `UBLKCP.*`/`SYNCS.*` are the TMA bulk copy + mbarrier pipeline, `LDGMC.E.HPADD` is "
    "`multimem.ld_reduce`, `STG.E.*.STRONG.SYS` to a multicast address carries `multimem.st`, "
    "`ST.E.*.STRONG.SYS` / `MEMBAR.*.SYS` are the in-kernel completion signals (st.release.sys). The full "
    "listings are in `docs/sass/` (the row-sparse kernel of `update_rows_kernels.cu` has its census here only). "
    "Every flavour listed here has run on B200 (profiles/r2/).\n\n"
)


def demangle(name):
    out = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
    out = re.sub(r"\(anonymous namespace\)::", "", out)
    out = re.sub(r"^void ", "", out)
    out = re.sub(r"\(.*$", "", out)
    out = out.replace("(PsGradFmt)", "").replace("(PsOpt)", "")
    return out


def main():
    doc = [HEADER]
    for src in SOURCES:
        with tempfile.TemporaryDirectory() as tmp:
            obj = os.path.join(tmp, "k.o")
            cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
                   "-Iinclude", "-Isrc", "-Xptxas", "-v", "-c", src, "-o", obj]
            res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
            if res.returncode != 0:
                sys.exit(res.stderr)
            rows, cur = [], None
            for line in res.stderr.splitlines():
                m = re.search(r"Compiling entry function '(\S+)'", line)
                if m:
                    cur = {"name": demangle(m.group(1))}
                    rows.append(cur)
                    continue
                m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
                if m and cur is not None:
                    cur["spill"] = f"{m.group(1)} / {m.group(2)}"
                m = re.search(r"Used (\d+) registers", line)
                if m and cur is not None:
                    cur["regs"] = m.group(1)
                    s = re.search(r"(\d+) bytes smem", line)
                    cur["smem"] = s.group(1) if s else "0"
            sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
            if src in LISTINGS:
                listing = os.path.join(ROOT, "docs", "sass", os.path.basename(src).replace(".cu", ".sm_100a.sass"))
                with open(listing, "w") as lf:
                    lf.write(sass)
        census = collections.Counter()
        for line in sass.splitlines():
            m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
            if m and INTERESTING.match(m.group(1)):
                census[m.group(1)] += 1
        doc.append(f"\n## {src}\n| kernel | registers | spill stores / loads (B) | smem (B) |\n|---|---|---|---|\n")
        for r in rows:
            doc.append(f"| `{r['name']}` | {r.get('regs', '?')} | {r.get('spill', '?')} | {r.get('smem', '0')} |\n")
        doc.append("\nSASS census: " + ", ".join(f"`{k}` x{v}" for k, v in sorted(census.items())) + "\n")
    with open(os.path.join(ROOT, "profiles", "ptxas_and_sass_census.md"), "w") as f:
        f.write("".join(doc))
    print("wrote profiles/ptxas_and_sass_census.md")


if __name__ == "__main__":
    main()
