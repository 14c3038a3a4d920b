"""Instruction-for-instruction comparison of every kernel in two cubins (no GPU needed).

Usage: sass_compare.py OLD.cubin NEW.cubin
(cubins from nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -cubin ...)

For every kernel symbol of either cubin it prints one of
  identical      the same instruction stream
  immediates     the same instruction stream except hex immediates (shared-memory, parameter or branch offsets), followed
                 by the distinct old -> new pairs; a constant that ptxas loads as two fp16 halves (HFMA2 Rd, -RZ, RZ, hi, lo)
                 counts as one hex immediate
  DIFFERENT      anything else, with the first differing instruction
  MISSING        the symbol is in one cubin only
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
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    names = sorted(set(old) | set(new))
    pretty = demangle(names)
    bad = False
    for n in names:
        if n not in old or n not in new:
            verdict, detail = "MISSING", "only in " + ("NEW" if n not in old else "OLD")
        else:
            verdict, detail = compare(old[n], new[n])
        bad = bad or verdict in ("DIFFERENT", "MISSING")
        print(f"{verdict:<10} {pretty[n]}" + (f": {detail}" if detail else ""))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
