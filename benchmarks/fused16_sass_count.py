"""Instruction count of the steady-state item path of the fp16 x 2 fused logistic gradient's epilogue, per instantiation
(KB = 1: dim <= 64, KB = 2: dim <= 128), from `cuobjdump -sass` of the built library (or of a cubin), split into the
floating-point arithmetic of half_item and everything else.  --cu compiles one source file to a cubin with the
Makefile's flags in a temporary directory and counts that: no library build or link is needed.

By default the path is the innermost loop of the kernel that holds a full work item (16 MUFU.EX2 per item), and the
count is per item (the loop runs two items per trip).  --ranges counts explicit half-open address ranges instead (for
builds without that loop), e.g. --ranges 2:0x15b0-0x1660,0x1ab0-0x29f0 --ranges 1:...; a static count of what lies in
the ranges.
    python benchmarks/fused16_sass_count.py [--lib aehmc_b200/lib/libb200hmc.so | --cu aehmc_b200/csrc/tc_gemm.cu]
                                            [--ranges KB:A-B,...]"""
import argparse, collections, os, re, subprocess, tempfile

ARITH = {"MUFU", "FMUL", "FADD", "FFMA", "FMUL2", "FADD2", "FFMA2", "FSETP", "FSEL", "F2FP", "HADD2", "FHADD", "FHFMA"}
KERNEL = "_ZN3b2h2tc26tc_logistic_fused16_kernelILi{}EEEv14CUtensorMap_stNS0_11Fused16ArgsE"
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")


def cubin(src, out_dir):
    out = os.path.join(out_dir, os.path.splitext(os.path.basename(src))[0] + ".cubin")
    subprocess.run([os.path.join(CUDA, "bin", "nvcc"), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                    "-lineinfo", "--expt-relaxed-constexpr", "-cubin", src, "-o", out], check=True)
    return out


def sass(lib, kb):
    cuobjdump = os.path.join(CUDA, "bin", "cuobjdump")
    txt = subprocess.run([cuobjdump, "-sass", "-fun", KERNEL.format(kb), lib], check=True, capture_output=True,
                         text=True).stdout
    ins = [(int(m.group(1), 16), m.group(2)) for m in re.finditer(r"/\*([0-9a-f]{4,})\*/\s+([^;]*?)\s*;", txt)]
    if not ins:
        raise SystemExit(f"no SASS for KB = {kb} in {lib}")
    return ins


def opcode(text):
    return re.sub(r"^@!?U?P\w+\s+", "", text).split()[0].split(".")[0]


def steady_loop(ins):
    """innermost backward-branch loop holding at least one full item; returns (ranges, items per trip)"""
    best = None
    for addr, text in ins:
        m = re.search(r"\bBRA\s+(?:`\()?(0x[0-9a-f]+)", text)
        if not m or int(m.group(1), 16) >= addr:
            continue
        lo = int(m.group(1), 16)
        ex2 = sum("MUFU.EX2" in t for a, t in ins if lo <= a <= addr)
        if ex2 >= 16 and (best is None or addr - lo < best[1] - best[0]):
            best = (lo, addr, ex2 // 16)
    if best is None:
        raise SystemExit("no loop holding a whole item: pass --ranges")
    return [(best[0], best[1] + 16)], best[2]


def main():
    ap = argparse.ArgumentParser()
    src = ap.add_mutually_exclusive_group()
    src.add_argument("--lib", default="aehmc_b200/lib/libb200hmc.so", help="library or cubin to disassemble")
    src.add_argument("--cu", help="source file to compile to a cubin and disassemble")
    ap.add_argument("--ranges", action="append", default=[], help="KB:A-B,C-D (half-open, hex)")
    a = ap.parse_args()
    given = {}
    for spec in a.ranges:
        kb, rs = spec.split(":")
        given[int(kb)] = [tuple(int(x, 16) for x in r.split("-")) for r in rs.split(",")]
    with tempfile.TemporaryDirectory() as tmp:
        lib = cubin(a.cu, tmp) if a.cu else a.lib
        ins_by_kb = {kb: sass(lib, kb) for kb in (1, 2)}
    for kb in (1, 2):
        ins = ins_by_kb[kb]
        if kb in given:
            ranges, items, how = given[kb], 1, "given ranges"
        else:
            ranges, items = steady_loop(ins)
            how = f"steady-state loop, {items} items per trip"
        body = [t for addr, t in ins if any(lo <= addr < hi for lo, hi in ranges)]
        ops = collections.Counter(opcode(t) for t in body)
        arith = sum(v for k, v in ops.items() if k in ARITH)
        other = {k: v / items for k, v in sorted(ops.items(), key=lambda kv: -kv[1]) if k not in ARITH}
        print(f"KB = {kb} ({how}: {', '.join(f'{lo:#x}-{hi:#x}' for lo, hi in ranges)})")
        print(f"  per item: {len(body) / items:g} instructions, {arith / items:g} half_item arithmetic, "
              f"{(len(body) - arith) / items:g} other")
        print("  other: " + ", ".join(f"{k} {v:g}" for k, v in other.items()))


if __name__ == "__main__":
    main()
