"""Instruction footprint of the eikonal kernels, from the compiler alone (no GPU needed).

    python tools/sass_footprint.py                      # compile csrc/eikonal.cu for sm_100a with the library's flags
    python tools/sass_footprint.py --src DIR            # ... from another source tree (DIR/mcmc_eq_b200/csrc/eikonal.cu)
    python tools/sass_footprint.py --cubin F.cubin      # read a cubin
    python tools/sass_footprint.py --so lib.so          # read the sm_100a cubin embedded in a built library
    options: --top N (source lines per kernel, default 8), --json

Per eikonal kernel: SASS instructions (the kernel's own code plus the out-of-line functions it calls, which the cubin
keeps inside the kernel's section), registers, stack frame, LDL/STL count (local memory) and which source files they come
from, and the source lines with the most instructions.  Line attribution needs -lineinfo, which the library build uses.
"""
from __future__ import annotations

import argparse
import collections
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_INSN = re.compile(r"^\s+/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;?\s*$")
_FILE = re.compile(r'^\s*//## File "([^"]+)", line (\d+)')
_SECTION = re.compile(r"^\.text\.(\S+):\s*$")
_SUB = re.compile(r"^\$(\S+?)\$(\S+):\s*$")
_PIPE = re.compile(r"eik_pipe_kernelILi(\d+)ELi(\d+)E")


def cuda_bin(tool: str) -> str | None:
    p = shutil.which(tool)
    if p:
        return p
    p = os.path.join("/usr/local/cuda/bin", tool)
    return p if os.path.exists(p) else None


def nvcc_flags() -> list[str]:
    """The library's nvcc flags (mcmc_eq_b200/build.py) without the ones that only concern linking a shared object."""
    sys.path.insert(0, ROOT)
    from mcmc_eq_b200 import build  # noqa: E402
    out, skip = [], False
    for f in build.NVCC_FLAGS:
        if skip:
            skip = False
            continue
        if f == "-Xcompiler":
            skip = True
            continue
        if f == "-shared":
            continue
        out.append(f)
    return out


def compile_cubin(src_root: str, out: str) -> str:
    nvcc = cuda_bin("nvcc")
    if nvcc is None:
        raise RuntimeError("nvcc not found")
    src = os.path.join(src_root, "mcmc_eq_b200", "csrc", "eikonal.cu")
    subprocess.run([nvcc, "-cubin"] + nvcc_flags() + [src, "-o", out], check=True, cwd=src_root)
    return out


def cubin_from_so(so: str, tmp: str) -> str:
    subprocess.run([cuda_bin("cuobjdump"), "-xelf", "all", os.path.abspath(so)], check=True, cwd=tmp,
                   stdout=subprocess.DEVNULL)
    for f in sorted(os.listdir(tmp)):
        if f.endswith(".cubin") and "sm_100a" in f:
            path = os.path.join(tmp, f)
            if "eik_pipe_kernel" in subprocess.run([cuda_bin("cuobjdump"), "-res-usage", path], capture_output=True,
                                                   text=True).stdout:
                return path
    raise RuntimeError(f"no sm_100a cubin with the eikonal kernels in {so}")


def resources(cubin: str) -> dict[str, dict[str, int]]:
    txt = subprocess.run([cuda_bin("cuobjdump"), "-res-usage", cubin], check=True, capture_output=True, text=True).stdout
    res, name = {}, None
    for line in txt.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = m.group(1)
            continue
        if name and "REG:" in line:
            res[name] = {k: int(v) for k, v in re.findall(r"(\w+):(\d+)", line)}
            name = None
    return res


def demangle(names: list[str]) -> dict[str, str]:
    tool = cuda_bin("cu++filt") or shutil.which("c++filt")
    if not tool or not names:
        return {n: n for n in names}
    out = subprocess.run([tool], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, out)) if len(out) == len(names) else {n: n for n in names}


def parse_sass(cubin: str) -> dict[str, dict]:
    """Per kernel section: instruction records (region, file, line, opcode)."""
    txt = subprocess.run([cuda_bin("nvdisasm"), "-g", "-c", cubin], check=True, capture_output=True, text=True).stdout
    kernels: dict[str, list] = {}
    cur, region, src = None, None, ("?", 0)
    for line in txt.splitlines():
        m = _SECTION.match(line)
        if m:
            cur = m.group(1)
            region, src = cur, ("?", 0)
            kernels[cur] = []
            continue
        if cur is None:
            continue
        m = _SUB.match(line)
        if m and m.group(1) == cur:
            region = m.group(2)
            continue
        if line.startswith("$__internal"):
            region = line.strip().rstrip(":")
            continue
        m = _FILE.match(line)
        if m:
            src = (m.group(1), int(m.group(2)))
            continue
        m = _INSN.match(line)
        if m:
            body = m.group(1)
            if body.startswith("@"):
                body = body.split(None, 1)[1] if " " in body else body
            op = body.split(None, 1)[0] if body else "?"
            kernels[cur].append((region, src[0], src[1], op))
    return kernels


def footprint(cubin: str, top: int = 8, match: str = "eik_") -> list[dict]:
    res = resources(cubin)
    sass = parse_sass(cubin)
    names = [k for k in sass if match in k and "kernel" in k]
    dm = demangle(names + sorted({r for k in names for r, *_ in sass[k] if r != k and not r.startswith("$")}))
    out = []
    for k in names:
        recs = sass[k]
        regions = collections.Counter(r for r, *_ in recs)
        local = [(f, ln) for _, f, ln, op in recs if op.startswith(("LDL", "STL"))]
        lines = collections.Counter((os.path.basename(f), ln) for _, f, ln, _ in recs)
        r = res.get(k, {})
        entry = {
            "kernel": dm.get(k, k), "mangled": k,
            "instructions": len(recs),
            "own_instructions": regions.get(k, 0),
            "functions": {dm.get(n, n): c for n, c in regions.most_common() if n != k},
            "registers": r.get("REG"), "stack": r.get("STACK"),
            "local_accesses": len(local),
            "local_by_file": dict(collections.Counter(os.path.basename(f) for f, _ in local)),
            "top_lines": [{"file": f, "line": ln, "instructions": c} for (f, ln), c in lines.most_common(top)],
        }
        m = _PIPE.search(k)
        if m:
            warps = int(m.group(2))
            entry["warps_per_cta"] = warps
            entry["register_limit"] = min(255, (65536 // (warps * 32)) // 8 * 8)
        out.append(entry)
    return out


def report(fp: list[dict]) -> str:
    rows = []
    for e in fp:
        lim = f" (limit {e['register_limit']} for {e['warps_per_cta']} warps)" if "register_limit" in e else ""
        rows.append(f"{e['kernel']}")
        rows.append(f"  instructions {e['instructions']} (kernel {e['own_instructions']}), registers {e['registers']}{lim}, "
                    f"stack {e['stack']} B, LDL/STL {e['local_accesses']} {e['local_by_file'] or ''}")
        for name, c in e["functions"].items():
            rows.append(f"    {c:7d}  {name}")
        for t in e["top_lines"]:
            rows.append(f"    {t['instructions']:7d}  {t['file']}:{t['line']}")
    return "\n".join(rows)


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    g = ap.add_mutually_exclusive_group()
    g.add_argument("--src", default=ROOT, help="source tree to compile (default: this repository)")
    g.add_argument("--cubin")
    g.add_argument("--so")
    ap.add_argument("--top", type=int, default=8)
    ap.add_argument("--json", action="store_true")
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        if a.cubin:
            cubin = a.cubin
        elif a.so:
            cubin = cubin_from_so(a.so, tmp)
        else:
            cubin = compile_cubin(os.path.abspath(a.src), os.path.join(tmp, "eikonal.cubin"))
        fp = footprint(cubin, a.top)
    print(json.dumps(fp, indent=1) if a.json else report(fp))


if __name__ == "__main__":
    main()
