#!/usr/bin/env python3
"""IMAD-pipe budget of the Bandersnatch verify kernels, read from the SASS (no GPU needed).

The two kernels of an IETF verify, k_lincomb<BandCurve, 2, 0> (V = s*I - c*O) and k_lincomb<BandCurve, 1, 1> (U = s*G - c*Y),
spend nearly all their time in a few called functions (products, squares, point additions and doublings).  Every IMAD form
issues to the integer-multiply pipe, including the ones that multiply nothing: IMAD.MOV (a move or a negation), IMAD.IADD,
IMAD.SHL, and IMAD.X with an RZ multiplicand (a carry addition).  This tool

  1. disassembles the kernels (cuobjdump -sass) and splits each at the CALL.REL.NOINC targets into its called functions,
     named from the cubin's symbol table;
  2. counts each function's IMAD-pipe instructions by form, multiplying and non-multiplying apart;
  3. multiplies by the calls per item, derived below from the loop structure of lincomb.cuh and the formulas of te.cuh,
     and prints model cycles per 32 items (one warp): 4 cycles per warp instruction for IMAD.WIDE* / IMAD.HI*, 2 for the
     32-bit forms (plain IMAD, .X, .MOV, .IADD, .SHL).  Static counts: a function's both branches (want_t) are counted.

usage: tools/sass_imad_budget.py [LIB.so | KERNELS.cubin] [--json OUT]
(default: ark_ec_vrfs_b200/libvrfs_b200.so)
"""
import json
import os
import re
import shutil
import struct
import subprocess
import sys
import tempfile
from collections import Counter, defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KERNELS = {"<2,0>": "_Z9k_lincombIN4vrfs9BandCurveELi2ELi0EEvNS0_11LincombArgsE",
           "<1,1>": "_Z9k_lincombIN4vrfs9BandCurveELi1ELi1EEvNS0_11LincombArgsE"}


def cuobjdump():
    for c in (os.environ.get("CUOBJDUMP"), "/usr/local/cuda/bin/cuobjdump", shutil.which("cuobjdump")):
        if c and os.path.exists(c):
            return c
    return None


# ---- calls per item (lincomb.cuh lincomb_item / build_table, te.cuh) ------------------------------------------------------
WINDOWS = 32          # radix-16 windows of a 127-bit GLV half
FIX_WINDOWS = 16      # VRFS_FIX_BITS = 16
TBL_ODD, TBL_EVEN = 3, 4   # build_table: 3P, 5P, 7P by additions; 2P, 4P, 6P, 8P by doublings of entries read back


def calls_per_item(nv, nf):
    """dynamic calls of each called function per item, and the products / squares they make"""
    nt = 2 * nv                                   # GLV: two tables per variable base
    add_t = add_not = dbl_t = dbl_not = madd_t = madd_not = 0
    # variable bases: per base, two tables (B and psi(B)), one endomorphism, one GLV split
    add_t += nt * TBL_ODD
    dbl_t += nt * TBL_EVEN
    direct_mul = nv * (2 + 1) + nt * 9           # on-curve check (d * xx * yy), from_affine (T = xy), 9 to_entry per table (d * T)
    direct_sqr = nv * 2                           # on-curve check
    # Straus loop: WINDOWS windows, dbl4 between them (3 doublings without T, one with), NT additions per window; the last
    # addition of a window skips T unless fixed-base additions follow the last window
    dbl_not += (WINDOWS - 1) * 3
    dbl_t += (WINDOWS - 1) * 1
    add_t += WINDOWS * (nt - 1)
    if nf > 0:
        add_t += 1; add_not += WINDOWS - 1
    else:
        add_not += WINDOWS
    # fixed bases: FIX_WINDOWS mixed additions per term; only the very last one skips T
    madd_t += nf * FIX_WINDOWS - (1 if nf else 0)
    madd_not += 1 if nf else 0
    calls = {"te_add_cached": add_t + add_not, "te_dbl": dbl_t + dbl_not, "te_madd": madd_t + madd_not,
             "band_endo": nv, "band_glv_split": nv}
    # te_add_cached: 9 products (+1 for T); te_dbl: 4 squares, 3 products (+1 for T); te_madd: 7 products (+1); band_endo: 2 S + 8 M
    mul = direct_mul + 10 * add_t + 9 * add_not + 4 * dbl_t + 3 * dbl_not + 8 * madd_t + 7 * madd_not + 8 * nv
    sqr = direct_sqr + 4 * (dbl_t + dbl_not) + 2 * nv
    calls["mont_mul_call"] = mul
    calls["mont_sqr_call"] = sqr
    return calls


# ---- SASS -----------------------------------------------------------------------------------------------------------------
INSN = re.compile(r"^\s+/\*([0-9a-f]+)\*/\s+(.*?)\s*;")


def elf_func_symbols(cubin):
    """{(section symbol name of the kernel): {offset: local function name}} from the cubin's symbol table"""
    data = open(cubin, "rb").read()
    shoff, = struct.unpack_from("<Q", data, 0x28)
    shentsize, shnum = struct.unpack_from("<HH", data, 0x3A)
    secs = [struct.unpack_from("<IIQQQQIIQQ", data, shoff + i * shentsize) for i in range(shnum)]
    out = defaultdict(dict)
    for s in secs:
        if s[1] != 2:       # SHT_SYMTAB
            continue
        strtab = secs[s[6]]
        for off in range(s[4], s[4] + s[5], 24):
            name_off, info, _, _, value, _ = struct.unpack_from("<IBBHQQ", data, off)
            if info & 0xF != 2:   # STT_FUNC
                continue
            start = strtab[4] + name_off
            name = data[start:data.index(b"\0", start)].decode()
            if name.startswith("$") and name.count("$") >= 2:
                _, kern, callee = name.split("$", 2)
                out[kern][value] = callee
    return out


def short_name(mangled):
    m = re.search(r"vrfs(\d+)", mangled)
    if not m:
        return mangled
    i = m.end()
    name = mangled[i:i + int(m.group(1))]
    rest = mangled[i + int(m.group(1)):]
    t = re.match(r"INS0_(\d+)", rest)
    if t:
        name += "<" + rest[t.end():t.end() + int(t.group(1))] + ">"
    return name


def kernel_sass(sass_text, kernel):
    lines, on = [], False
    for ln in sass_text.splitlines():
        if "Function : " in ln:
            on = ln.split("Function : ")[1].strip() == kernel
            continue
        if on:
            m = INSN.match(ln)
            if m:
                lines.append((int(m.group(1), 16), m.group(2)))
    return lines


def split_functions(insns, names):
    targets = sorted({int(m.group(1), 16) for _, t in insns for m in [re.search(r"CALL\.REL\.NOINC\s+(0x[0-9a-f]+)", t)] if m})
    starts = [0] + targets
    funcs = {}
    for i, s in enumerate(starts):
        e = starts[i + 1] if i + 1 < len(starts) else float("inf")
        label = "(kernel body)" if s == 0 else short_name(names.get(s, "fn@0x%x" % s))
        funcs[label] = [t for a, t in insns if s <= a < e]
    return funcs


def classify(text):
    """None (not on the IMAD pipe) or (form, multiplies, model cycles)"""
    t = re.sub(r"^@!?U?P[T0-9]\s+", "", text)
    op = t.split()[0]
    if not op.startswith("IMAD"):
        return None
    srcs = [s.strip() for s in t[len(op):].split(",")]
    # operands: dst, [carry-out predicate,] a, b, c [, carry-in]
    srcs = [s for s in srcs[1:] if not re.fullmatch(r"!?U?P[T0-9]", s)]
    wide = ".WIDE" in op or ".HI" in op
    mult = not (".MOV" in op or ".IADD" in op or ".SHL" in op) and len(srcs) >= 2 and "RZ" not in srcs[:2] \
        and srcs[1] not in ("0x1", "1")
    return op, mult, 4 if wide else 2


def budget(funcs):
    rows = {}
    for name, body in funcs.items():
        forms = Counter()
        mult = nonmult = cyc_m = cyc_n = 0
        for t in body:
            c = classify(t)
            if c is None:
                continue
            op, is_m, cy = c
            forms[op + ("" if is_m else " (no multiply)")] += 1
            if is_m:
                mult += 1; cyc_m += cy
            else:
                nonmult += 1; cyc_n += cy
        rows[name] = {"instructions": len(body), "imad_mult": mult, "imad_nonmult": nonmult,
                      "cycles_mult": cyc_m, "cycles_nonmult": cyc_n, "forms": dict(sorted(forms.items()))}
    return rows


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_json = sys.argv[sys.argv.index("--json") + 1] if "--json" in sys.argv else None
    if out_json in args:
        args.remove(out_json)
    src = args[0] if args else os.path.join(ROOT, "ark_ec_vrfs_b200", "libvrfs_b200.so")
    tool = cuobjdump()
    if tool is None:
        sys.exit("cuobjdump not found")
    with tempfile.TemporaryDirectory() as tmp:
        if src.endswith(".cubin"):
            cubins = [src]
        else:
            subprocess.run([tool, "-xelf", "all", os.path.abspath(src)], cwd=tmp, check=True, stdout=subprocess.DEVNULL)
            cubins = [os.path.join(tmp, f) for f in os.listdir(tmp) if f.endswith(".cubin")]
        result = {"source": os.path.basename(src), "kernels": {}}
        for cubin in cubins:
            syms = elf_func_symbols(cubin)
            if not any(k in syms for k in KERNELS.values()):
                continue
            sass = subprocess.run([tool, "-sass", cubin], check=True, capture_output=True, text=True).stdout
            for label, kern in KERNELS.items():
                insns = kernel_sass(sass, kern)
                if not insns:
                    continue
                rows = budget(split_functions(insns, syms.get(kern, {})))
                nv, nf = (2, 0) if label == "<2,0>" else (1, 1)
                calls = calls_per_item(nv, nf)
                tot = Counter()
                for name, r in rows.items():
                    base = name.split("<")[0]
                    r["calls_per_item"] = calls.get(base, 0)
                    for k in ("imad_mult", "imad_nonmult", "cycles_mult", "cycles_nonmult"):
                        tot[k] += r[k] * r["calls_per_item"]
                tot_cyc = tot["cycles_mult"] + tot["cycles_nonmult"]
                result["kernels"][label] = {"functions": rows, "per_item": dict(tot),
                                            "model_cycles_per_32_items": tot_cyc,
                                            "nonmult_share_of_cycles": round(tot["cycles_nonmult"] / tot_cyc, 4) if tot_cyc else 0.0}
    if not result["kernels"]:
        sys.exit("no k_lincomb<BandCurve, 2, 0> / <1, 1> in %s" % src)
    for label, k in result["kernels"].items():
        print("k_lincomb<BandCurve,%s>" % label[1:-1])
        print("  %-26s %6s %6s %6s %6s  %s" % ("function", "insns", "mult", "nonm", "calls", "non-multiplying forms"))
        for name, r in k["functions"].items():
            nm = ", ".join("%d %s" % (v, f.replace(" (no multiply)", "")) for f, v in r["forms"].items() if "no multiply" in f)
            print("  %-26s %6d %6d %6d %6d  %s" % (name, r["instructions"], r["imad_mult"], r["imad_nonmult"], r["calls_per_item"], nm))
        p = k["per_item"]
        print("  per item: %d multiplying, %d non-multiplying IMAD-pipe instructions; model %.3f M cycles per 32 items, "
              "non-multiplying share %.1f %%" % (p["imad_mult"], p["imad_nonmult"], k["model_cycles_per_32_items"] / 1e6,
                                               100 * k["nonmult_share_of_cycles"]))
    if out_json:
        with open(out_json, "w") as f:
            json.dump(result, f, indent=1, sort_keys=True)
    return result


if __name__ == "__main__":
    main()
