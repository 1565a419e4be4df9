#!/usr/bin/env python
"""Development tool: side-by-side variants of one kernel source for A/B timing in a single GPU call.

    python tools/build_variants.py mwa_sp.cu notma:-DMWA_SP_NO_TMA=1 nostore:-DMWA_SP_EPI_NOSTORE=1 ...

Each variant recompiles the named source with its defines, links it with the objects of the regular build and writes
build/variants/<name>.so (git-ignored; travels to the GPU box).  `tools/kbench.py --lib build/variants/<name>.so` times it.
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import importlib
B = importlib.import_module("deep-learning-based-rgba-image-compression-with-masked-window-based-attention_b200.build")


def main():
    src = sys.argv[1]
    B.build()
    outdir = os.path.join(ROOT, "build", "variants")
    os.makedirs(outdir, exist_ok=True)
    objdir = os.path.join(B.PKG_DIR, "build")
    procs = []
    for spec in sys.argv[2:]:
        name, _, defs = spec.partition(":")
        obj = os.path.join(outdir, name + ".o")
        cmd = [B._nvcc(), *B.ARCH, *B.COMMON, *B.EXTRA.get(src, []), *[d for d in defs.split(",") if d], "-Xptxas", "-v", "-c",
               os.path.join(B.CSRC, src), "-o", obj]
        procs.append((name, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for name, obj, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out)
            raise SystemExit(f"nvcc failed on variant {name}")
        spills = [l for l in out.splitlines() if "spill" in l and " 0 bytes spill stores, 0 bytes spill loads" not in l]
        objs = [obj if s == src else os.path.join(objdir, s.replace(".cu", ".o")) for s in B.SOURCES]
        lib = os.path.join(outdir, name + ".so")
        subprocess.run([B._nvcc(), *B.ARCH, "-shared", "--cudart", "static", "-o", lib, *objs], check=True)
        print(f"{lib}  ({len(spills)} functions with spills)")


if __name__ == "__main__":
    main()
