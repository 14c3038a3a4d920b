r"""Instruction-for-instruction comparison of every kernel in two cubins (no GPU needed).

Usage: sass_compare.py [--map PATTERN=REPLACEMENT ...] OLD.cubin NEW.cubin
(cubins from nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -cubin ...)

Kernels are paired by demangled name.  --map rewrites NEW's demangled names (Python re.sub) before pairing, so that a kernel
that gained a template argument meets its old self, e.g. --map 'k_analyse<(\d+), (\w+), (\w+), false>=k_analyse<\1, \2, \3>';
with --map, a kernel only in NEW is reported as ADDED and is not an error.

For every kernel symbol of either cubin it prints one of
  identical      the same instruction stream
  immediates     the same instruction stream except hex immediates (shared-memory, parameter or branch offsets), followed
                 by the distinct old -> new pairs; a constant that ptxas loads as two fp16 halves (HFMA2 Rd, -RZ, RZ, hi, lo)
                 counts as one hex immediate
  DIFFERENT      anything else, with the first differing instruction
  MISSING        the symbol is in one cubin only
  ADDED          (with --map) the symbol is in NEW only
and exits with status 1 if any kernel is DIFFERENT or MISSING."""
import os
import re
import shutil
import struct
import subprocess
import sys

HEX = re.compile(r"0x[0-9a-fA-F]+")
# ptxas loads some 32-bit constants as "HFMA2 Rd, -RZ, RZ, hi, lo" with the halves printed as fp16 values: show the constant
HFMA2_MOV = re.compile(r"^HFMA2 (R\d+), -RZ, RZ, (\S+), (\S+)$")
# an anonymous namespace's mangled name carries a per-compilation hash: blank it so that its kernels pair up (same length)
ANON = re.compile(r"(_GLOBAL__N__)[0-9a-f]{8}")


def f16_bits(text):
    try:
        return struct.unpack("<H", struct.pack("<e", float(text)))[0]
    except (ValueError, OverflowError, struct.error):
        return None


def normalise(ins):
    m = HFMA2_MOV.match(ins)
    if m:
        hi, lo = f16_bits(m.group(2)), f16_bits(m.group(3))
        if hi is not None and lo is not None:
            return f"HFMA2.MOV {m.group(1)}, {(hi << 16) | lo:#x}"
    return ins


def kernels(cubin):
    tool = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    out = subprocess.run([tool, "-sass", cubin], capture_output=True, text=True, check=True).stdout
    fs, cur = {}, None
    for line in out.split("\n"):
        line = ANON.sub(r"\g<1>00000000", line)
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            fs[cur] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if m and cur:
            fs[cur].append(normalise(" ".join(m.group(1).split())))
    return fs


def demangle(names):
    if not names or shutil.which("c++filt") is None:
        return {n: n for n in names}
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.split("\n")
    return dict(zip(names, out))


def compare(a, b):
    if a == b:
        return "identical", ""
    if len(a) == len(b) and all(HEX.sub("#", x) == HEX.sub("#", y) for x, y in zip(a, b)):
        pairs = sorted({(u, v) for x, y in zip(a, b) for u, v in zip(HEX.findall(x), HEX.findall(y)) if u != v},
                       key=lambda p: (int(p[0], 16), int(p[1], 16)))
        return "immediates", ", ".join(f"{u} -> {v}" for u, v in pairs)
    i = next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
    old = a[i] if i < len(a) else "(end)"
    new = b[i] if i < len(b) else "(end)"
    return "DIFFERENT", f"{len(a)} -> {len(b)} instructions; first difference at {i}: {old!r} -> {new!r}"


def main():
    args, maps = sys.argv[1:], []
    while len(args) >= 2 and args[0] == "--map" and "=" in args[1]:
        maps.append(args[1].split("=", 1))
        args = args[2:]
    if len(args) != 2:
        sys.exit(__doc__)
    old, new = kernels(args[0]), kernels(args[1])
    pretty = demangle(sorted(set(old) | set(new)))
    old = {pretty[n]: v for n, v in old.items()}
    renamed = {}
    for n, v in new.items():
        name = pretty[n]
        for pat, rep in maps:
            name = re.sub(pat, rep, name)
        renamed[name] = (v, pretty[n])
    bad = False
    for name in sorted(set(old) | set(renamed)):
        if name not in renamed:
            verdict, detail = "MISSING", "only in OLD"
        elif name not in old:
            verdict, detail = ("ADDED", "") if maps else ("MISSING", "only in NEW")
        else:
            verdict, detail = compare(old[name], renamed[name][0])
        bad = bad or verdict in ("DIFFERENT", "MISSING")
        label = name
        if name in renamed and renamed[name][1] != name:
            label = f"{name} -> {renamed[name][1]}" if name in old else renamed[name][1]
        print(f"{verdict:<10} {label}" + (f": {detail}" if detail else ""))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
