#!/usr/bin/env python3
"""Emit ark_ec_vrfs_b200/csrc/gen/mont_chains.cuh: the carry-chain building blocks of the N-limb
(32-bit limbs) Montgomery multiplier, N = 8 and 12, each as ONE inline-PTX block (the carry flag never
leaves a block) plus a plain-C twin used only when the header is compiled for the host (the
`tests/host_emul` harness that lets the field / curve code be checked without a GPU).

The multiplier keeps the running sum in two interleaved accumulators so that every
`mad.lo.cc / madc.hi.cc` pair covers two adjacent, not-yet-touched columns; ptxas fuses each pair
into one IMAD.WIDE.U32(.X) (see DESIGN.md, "K1").
"""
import os

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "ark_ec_vrfs_b200", "csrc", "gen", "mont_chains.cuh")


def asm_block(lines, outs, ins):
    """outs: list of C lvalues bound "+r"; ins: list of C rvalues bound "r"."""
    body = " ".join(l + ";" for l in lines)
    o = ", ".join(f'"+r"({x})' for x in outs)
    i = ", ".join(f'"r"({x})' for x in ins)
    return f'    asm("{body}" : {o} : {i});'


def gen(N):
    L = []
    H = N // 2
    L.append(f"template <> struct MontChains<{N}> {{")

    # ---- mul_row: acc[0..N-1] = sum_{k=0..H-1} x[2k] * b  (two limbs each, no carries needed)
    L.append("  // acc[2k+1]:acc[2k] = x[2k] * b")
    L.append("  static HD_INLINE void mul_row(uint32_t* acc, const uint32_t* x, uint32_t b) {")
    L.append("#ifdef __CUDA_ARCH__")
    lines = []
    for k in range(H):
        lines.append(f"mul.lo.u32 %{2*k}, %{N+k}, %{N+H}")
        lines.append(f"mul.hi.u32 %{2*k+1}, %{N+k}, %{N+H}")
    o = ", ".join(f'"=r"(acc[{j}])' for j in range(N))
    i = ", ".join([f'"r"(x[{2*k}])' for k in range(H)] + ['"r"(b)'])
    L.append(f'    asm("{" ".join(l + ";" for l in lines)}" : {o} : {i});')
    L.append("#else")
    L.append(f"    for (int k = 0; k < {H}; k++) {{ uint64_t t = (uint64_t)x[2 * k] * b; acc[2 * k] = (uint32_t)t; acc[2 * k + 1] = (uint32_t)(t >> 32); }}")
    L.append("#endif")
    L.append("  }")

    # ---- mad_row: acc += x_even * b ; top += carry-out
    L.append("  // acc[0..N-1] += sum_k x[2k]*b*2^(64k) as one carry chain; the carry out of acc[N-1] is added to top")
    L.append("  static HD_INLINE void mad_row(uint32_t* acc, uint32_t& top, const uint32_t* x, uint32_t b) {")
    L.append("#ifdef __CUDA_ARCH__")
    lines = []
    for k in range(H):
        lo = "mad.lo.cc.u32" if k == 0 else "madc.lo.cc.u32"
        lines.append(f"{lo} %{2*k}, %{N+1+k}, %{N+1+H}, %{2*k}")
        lines.append(f"madc.hi.cc.u32 %{2*k+1}, %{N+1+k}, %{N+1+H}, %{2*k+1}")
    lines.append(f"addc.u32 %{N}, %{N}, 0")
    L.append(asm_block(lines, [f"acc[{j}]" for j in range(N)] + ["top"], [f"x[{2*k}]" for k in range(H)] + ["b"]))
    L.append("#else")
    L.append("    uint32_t c = 0;")
    L.append(f"    for (int k = 0; k < {H}; k++) {{")
    L.append("      unsigned __int128 t = (unsigned __int128)x[2 * k] * b + acc[2 * k] + ((uint64_t)acc[2 * k + 1] << 32) + c;")
    L.append("      acc[2 * k] = (uint32_t)t; acc[2 * k + 1] = (uint32_t)(t >> 32); c = (uint32_t)(t >> 64);")
    L.append("    }")
    L.append("    top += c;")
    L.append("#endif")
    L.append("  }")

    # ---- mad_row_last: same but the carry out is known to be zero (bounds) and is dropped
    L.append("  // same, for the accumulator that owns the top column: its carry out is zero by the size bound")
    L.append("  static HD_INLINE void mad_row_top(uint32_t* acc, const uint32_t* x, uint32_t b) {")
    L.append("#ifdef __CUDA_ARCH__")
    lines = []
    for k in range(H):
        lo = "mad.lo.cc.u32" if k == 0 else "madc.lo.cc.u32"
        hi = "madc.hi.cc.u32" if k < H - 1 else "madc.hi.u32"
        lines.append(f"{lo} %{2*k}, %{N+k}, %{N+H}, %{2*k}")
        lines.append(f"{hi} %{2*k+1}, %{N+k}, %{N+H}, %{2*k+1}")
    L.append(asm_block(lines, [f"acc[{j}]" for j in range(N)], [f"x[{2*k}]" for k in range(H)] + ["b"]))
    L.append("#else")
    L.append("    uint32_t c = 0;")
    L.append(f"    for (int k = 0; k < {H}; k++) {{")
    L.append("      unsigned __int128 t = (unsigned __int128)x[2 * k] * b + acc[2 * k] + ((uint64_t)acc[2 * k + 1] << 32) + c;")
    L.append("      acc[2 * k] = (uint32_t)t; acc[2 * k + 1] = (uint32_t)(t >> 32); c = (uint32_t)(t >> 64);")
    L.append("    }")
    L.append("#endif")
    L.append("  }")

    # ---- shift_mad_row: v0 += u[1]; u[j] = row(x,b)[j] + u[j+2] + carry chain (u[N], u[N+1] = 0)
    L.append("  // v0 += u[1] (carry into the chain); then u[j] = (x[0],x[2],..)*b row + u[j+2], j = 0..N-1, u[N] = u[N+1] = 0")
    L.append("  static HD_INLINE void shift_mad_row(uint32_t* u, uint32_t& v0, const uint32_t* x, uint32_t b) {")
    L.append("#ifdef __CUDA_ARCH__")
    lines = [f"add.cc.u32 %{N}, %{N}, %1"]
    for k in range(H):
        a_lo = f"%{2*k+2}" if 2 * k + 2 < N else "0"
        a_hi = f"%{2*k+3}" if 2 * k + 3 < N else "0"
        hi = "madc.hi.cc.u32" if k < H - 1 else "madc.hi.u32"
        lines.append(f"madc.lo.cc.u32 %{2*k}, %{N+1+k}, %{N+1+H}, {a_lo}")
        lines.append(f"{hi} %{2*k+1}, %{N+1+k}, %{N+1+H}, {a_hi}")
    L.append(asm_block(lines, [f"u[{j}]" for j in range(N)] + ["v0"], [f"x[{2*k}]" for k in range(H)] + ["b"]))
    L.append("#else")
    L.append("    uint64_t s = (uint64_t)v0 + u[1]; v0 = (uint32_t)s; uint32_t c = (uint32_t)(s >> 32);")
    L.append(f"    for (int k = 0; k < {H}; k++) {{")
    L.append(f"      uint32_t lo = 2 * k + 2 < {N} ? u[2 * k + 2] : 0, hi = 2 * k + 3 < {N} ? u[2 * k + 3] : 0;")
    L.append("      unsigned __int128 t = (unsigned __int128)x[2 * k] * b + lo + ((uint64_t)hi << 32) + c;")
    L.append("      u[2 * k] = (uint32_t)t; u[2 * k + 1] = (uint32_t)(t >> 32); c = (uint32_t)(t >> 64);")
    L.append("    }")
    L.append("#endif")
    L.append("  }")

    # ---- reduction rows for a modulus with p[0] = 1, p[1] = 2^32 - 1 (BLS12-381 Fr): the lowest pair of each chain is
    #      m*1 = (0 : m)  resp.  m*(2^32-1) = (m - [m != 0] : -m), i.e. two additions instead of one wide multiply
    L.append("  // mad_row with x[0] == 1: acc[1]:acc[0] += b, remaining pairs multiplied as usual")
    L.append("  static HD_INLINE void mad_row_lo1(uint32_t* acc, uint32_t& top, const uint32_t* x, uint32_t b) {")
    L.append("#ifdef __CUDA_ARCH__")
    no = N + 1
    lines = [f"add.cc.u32 %0, %0, %{no+H-1}", "addc.cc.u32 %1, %1, 0"]
    for k in range(1, H):
        lines.append(f"madc.lo.cc.u32 %{2*k}, %{no+k-1}, %{no+H-1}, %{2*k}")
        lines.append(f"madc.hi.cc.u32 %{2*k+1}, %{no+k-1}, %{no+H-1}, %{2*k+1}")
    lines.append(f"addc.u32 %{N}, %{N}, 0")
    L.append(asm_block(lines, [f"acc[{j}]" for j in range(N)] + ["top"], [f"x[{2*k}]" for k in range(1, H)] + ["b"]))
    L.append("#else")
    L.append("    mad_row(acc, top, x, b);")
    L.append("#endif")
    L.append("  }")
    L.append("  // mad_row_top with x[0] == 2^32-1: nb = -b, bm1 = b - (b != 0)")
    L.append("  static HD_INLINE void mad_row_top_loff(uint32_t* acc, const uint32_t* x, uint32_t b, uint32_t nb, uint32_t bm1) {")
    L.append("#ifdef __CUDA_ARCH__")
    no = N
    lines = [f"add.cc.u32 %0, %0, %{no+H}", f"addc.cc.u32 %1, %1, %{no+H+1}"]
    for k in range(1, H):
        hi = "madc.hi.cc.u32" if k < H - 1 else "madc.hi.u32"
        lines.append(f"madc.lo.cc.u32 %{2*k}, %{no+k-1}, %{no+H-1}, %{2*k}")
        lines.append(f"{hi} %{2*k+1}, %{no+k-1}, %{no+H-1}, %{2*k+1}")
    L.append(asm_block(lines, [f"acc[{j}]" for j in range(N)], [f"x[{2*k}]" for k in range(1, H)] + ["b", "nb", "bm1"]))
    L.append("#else")
    L.append("    (void)nb; (void)bm1; mad_row_top(acc, x, b);")
    L.append("#endif")
    L.append("  }")
    L.append("  // shift_mad_row with x[0] == 2^32-1")
    L.append("  static HD_INLINE void shift_mad_row_loff(uint32_t* u, uint32_t& v0, const uint32_t* x, uint32_t b, uint32_t nb, uint32_t bm1) {")
    L.append("#ifdef __CUDA_ARCH__")
    no = N + 1
    lines = [f"add.cc.u32 %{N}, %{N}, %1", f"addc.cc.u32 %0, %{no+H}, %2", f"addc.cc.u32 %1, %{no+H+1}, %3"]
    for k in range(1, H):
        a_lo = f"%{2*k+2}" if 2 * k + 2 < N else "0"
        a_hi = f"%{2*k+3}" if 2 * k + 3 < N else "0"
        hi = "madc.hi.cc.u32" if k < H - 1 else "madc.hi.u32"
        lines.append(f"madc.lo.cc.u32 %{2*k}, %{no+k-1}, %{no+H-1}, {a_lo}")
        lines.append(f"{hi} %{2*k+1}, %{no+k-1}, %{no+H-1}, {a_hi}")
    L.append(asm_block(lines, [f"u[{j}]" for j in range(N)] + ["v0"], [f"x[{2*k}]" for k in range(1, H)] + ["b", "nb", "bm1"]))
    L.append("#else")
    L.append("    (void)nb; (void)bm1; shift_mad_row(u, v0, x, b);")
    L.append("#endif")
    L.append("  }")
    # ---- the multiplier of such a row from its column value c0 (NINV = -1): m = -c0 and m - [m != 0] from one borrow chain
    #      (two ALU additions instead of a compare and a predicated negation, which ptxas issues as IMAD.MOV)
    L.append("  // m = -c0 (the reduction multiplier when NINV = -1) and bm1 = m - [m != 0]: the borrow of 0 - c0 is [c0 != 0]")
    L.append("  static HD_INLINE void neg_bm1(uint32_t& m, uint32_t& bm1, uint32_t c0) {")
    L.append("#ifdef __CUDA_ARCH__")
    L.append('    asm("sub.cc.u32 %0, 0, %2; subc.u32 %1, 0, %2;" : "=r"(m), "=r"(bm1) : "r"(c0));')
    L.append("#else")
    L.append("    m = 0u - c0; bm1 = m - (c0 != 0u ? 1u : 0u);")
    L.append("#endif")
    L.append("  }")

    # ---- merge: u[0..N-2] += v[1..N-1] with carry, u[N-1] += carry
    L.append("  // u[0..N-2] += v[1..N-1], carry into u[N-1]")
    L.append("  static HD_INLINE void merge(uint32_t* u, const uint32_t* v) {")
    L.append("#ifdef __CUDA_ARCH__")
    lines = []
    for j in range(N - 1):
        op = "add.cc.u32" if j == 0 else "addc.cc.u32"
        lines.append(f"{op} %{j}, %{j}, %{N+j}")
    lines.append(f"addc.u32 %{N-1}, %{N-1}, 0")
    L.append(asm_block(lines, [f"u[{j}]" for j in range(N)], [f"v[{j+1}]" for j in range(N - 1)]))
    L.append("#else")
    L.append("    uint32_t c = 0;")
    L.append(f"    for (int j = 0; j < {N-1}; j++) {{ uint64_t t = (uint64_t)u[j] + v[j + 1] + c; u[j] = (uint32_t)t; c = (uint32_t)(t >> 32); }}")
    L.append(f"    u[{N-1}] += c;")
    L.append("#endif")
    L.append("  }")

    # ---- add / sub with carry/borrow out
    for name, op0, opc, opl, expr in (("add", "add.cc.u32", "addc.cc.u32", "addc.u32", "+"), ("sub", "sub.cc.u32", "subc.cc.u32", "subc.u32", "-")):
        L.append(f"  // r = a {expr} b over N limbs; returns the carry (add) / borrow (sub) as 0 or 1")
        L.append(f"  static HD_INLINE uint32_t {name}(uint32_t* r, const uint32_t* a, const uint32_t* b) {{")
        L.append("#ifdef __CUDA_ARCH__")
        L.append("    uint32_t c;")
        lines = []
        for j in range(N):
            lines.append(f"{op0 if j == 0 else opc} %{j}, %{N+1+j}, %{2*N+1+j}")
        if name == "add":
            lines.append(f"addc.u32 %{N}, 0, 0")
        else:
            lines.append(f"subc.u32 %{N}, 0, 0")
        o = ", ".join([f'"=r"(r[{j}])' for j in range(N)] + ['"=r"(c)'])
        i = ", ".join([f'"r"(a[{j}])' for j in range(N)] + [f'"r"(b[{j}])' for j in range(N)])
        L.append(f'    asm("{" ".join(l + ";" for l in lines)}" : {o} : {i});')
        L.append("    return c & 1u;" if name == "sub" else "    return c;")
        L.append("#else")
        if name == "add":
            L.append(f"    uint32_t c = 0; for (int j = 0; j < {N}; j++) {{ uint64_t t = (uint64_t)a[j] + b[j] + c; r[j] = (uint32_t)t; c = (uint32_t)(t >> 32); }} return c;")
        else:
            L.append(f"    uint32_t c = 0; for (int j = 0; j < {N}; j++) {{ uint64_t t = (uint64_t)a[j] - b[j] - c; r[j] = (uint32_t)t; c = (uint32_t)(t >> 32) & 1u; }} return c;")
        L.append("#endif")
        L.append("  }")
    L += gen_sqr(N)
    L += gen_mul_wide(N)
    L.append("};")
    return L


def sqr_chains(N):
    """Triangular squaring a^2 = sum_i a_i * Q_i * 2^(64 i), Q_i = [a_i, 2a_{i+1} (no carry-in), limbs of 2a above i+1]:
    N(N+1)/2 wide products instead of N^2.  Products of row i land at columns 2i+k; even k go to the even-aligned
    accumulator e[], odd k to the odd-aligned accumulator o[] (both indexed by absolute column), so that every
    mad.lo.cc/madc.hi.cc pair covers one aligned 64-bit slot and fuses into IMAD.WIDE.U32(.X).
    Returns [(acc_name, first_col, [(multiplicand_expr)...], row, emit_carry_out)]"""
    chains = []
    touched = {"e": set(), "o": set()}
    for i in range(N):
        q = []
        for k in range(N - i):
            q.append(f"a[{i}]" if k == 0 else (f"s{i+1}" if k == 1 else f"d[{i+k}]"))
        for acc, par in (("e", 0), ("o", 1)):
            ks = [k for k in range(N - i) if k % 2 == par]
            if not ks:
                continue
            first = 2 * i + ks[0]
            top_hi = 2 * i + ks[-1] + 1
            carry = (top_hi in touched[acc]) and top_hi + 1 < 2 * N
            chains.append((acc, first, [q[k] for k in ks], i, carry))
            for k in ks:
                touched[acc].add(2 * i + k); touched[acc].add(2 * i + k + 1)
            if carry:
                assert top_hi + 1 not in touched[acc], "carry-out must land in an untouched column"
                touched[acc].add(top_hi + 1)
    return chains


def gen_sqr(N):
    L = []
    L.append("  // t[0..2N-1] = a^2 (a < 2^(32N-1)): N(N+1)/2 wide products (see tools/gen_mont_chains.py sqr_chains)")
    L.append("  static HD_INLINE void sqr_wide(uint32_t* t, const uint32_t* a) {")
    L.append("#ifdef __CUDA_ARCH__")
    L.append(f"    uint32_t d[{N}], e[{2*N}], o[{2*N}];")
    L.append(f"    for (int k = 0; k < {2*N}; k++) {{ e[k] = 0; o[k] = 0; }}")
    L.append(f"    d[0] = 0; for (int k = 1; k < {N}; k++) d[k] = __funnelshift_l(a[k - 1], a[k], 1);   // limbs of 2a")
    cur_row = -1
    for acc, first, mults, row, carry in sqr_chains(N):
        if row != cur_row:
            cur_row = row
            if row + 1 < N:
                L.append(f"    const uint32_t s{row+1} = a[{row+1}] << 1;")
        n = len(mults)
        outs = [f"{acc}[{first + j}]" for j in range(2 * n)] + ([f"{acc}[{first + 2*n}]"] if carry else [])
        no = len(outs)
        ins = mults + [f"a[{row}]"]
        lines = []
        for j in range(n):
            lo = "mad.lo.cc.u32" if j == 0 else "madc.lo.cc.u32"
            hi = "madc.hi.cc.u32" if (j < n - 1 or carry) else "madc.hi.u32"
            lines.append(f"{lo} %{2*j}, %{no+j}, %{no+n}, %{2*j}")
            lines.append(f"{hi} %{2*j+1}, %{no+j}, %{no+n}, %{2*j+1}")
        if carry:
            lines.append(f"addc.u32 %{2*n}, %{2*n}, 0")
        L.append(asm_block(lines, outs, ins))
    # merge t = e + o
    lines = []
    for c in range(1, 2 * N):
        op = "add.cc.u32" if c == 1 else ("addc.cc.u32" if c < 2 * N - 1 else "addc.u32")
        lines.append(f"{op} %{c-1}, %{c-1}, %{2*N-1+c-1}")
    L.append(asm_block(lines, [f"e[{c}]" for c in range(1, 2 * N)], [f"o[{c}]" for c in range(1, 2 * N)]))
    L.append(f"    for (int k = 0; k < {2*N}; k++) t[k] = e[k];")
    L.append("#else")
    L.append(f"    unsigned __int128 acc = 0;")
    L.append(f"    for (int c = 0; c < {2*N}; c++) {{")
    L.append(f"      unsigned __int128 nxt = 0;")
    L.append(f"      for (int i = 0; i < {N}; i++) {{ int j = c - i; if (j < 0 || j >= {N}) continue; uint64_t pr = (uint64_t)a[i] * a[j]; acc += (uint32_t)pr; nxt += pr >> 32; }}")
    L.append(f"      t[c] = (uint32_t)acc; acc = (acc >> 32) + nxt;")
    L.append("    }")
    L.append("#endif")
    L.append("  }")
    return L


def mul_chains(N):
    """Schoolbook 2N-limb product for the special-form fields (pseudo-Mersenne / Solinas reduction follows): row i adds
    a_k * b_i at column k+i; products whose column is even go to the even-aligned accumulator e[], the others to o[]."""
    chains = []
    touched = {"e": set(), "o": set()}
    for i in range(N):
        for acc, par in (("e", 0), ("o", 1)):
            ks = [k for k in range(N) if (k + i) % 2 == par]
            first = ks[0] + i
            top_hi = ks[-1] + i + 1
            carry = (top_hi in touched[acc]) and top_hi + 1 < 2 * N
            chains.append((acc, first, [f"a[{k}]" for k in ks], i, carry))
            for k in ks:
                touched[acc].add(k + i); touched[acc].add(k + i + 1)
            if carry:
                assert top_hi + 1 not in touched[acc]
                touched[acc].add(top_hi + 1)
    return chains


def gen_mul_wide(N):
    L = []
    L.append("  // t[0..2N-1] = a * b (any N-limb values): N^2 wide products on two column-aligned accumulators")
    L.append("  static HD_INLINE void mul_wide(uint32_t* t, const uint32_t* a, const uint32_t* b) {")
    L.append("#ifdef __CUDA_ARCH__")
    L.append(f"    uint32_t e[{2*N}], o[{2*N}];")
    L.append(f"    for (int k = 0; k < {2*N}; k++) {{ e[k] = 0; o[k] = 0; }}")
    for acc, first, mults, row, carry in mul_chains(N):
        n = len(mults)
        outs = [f"{acc}[{first + j}]" for j in range(2 * n)] + ([f"{acc}[{first + 2*n}]"] if carry else [])
        no = len(outs)
        ins = mults + [f"b[{row}]"]
        lines = []
        for j in range(n):
            lo = "mad.lo.cc.u32" if j == 0 else "madc.lo.cc.u32"
            hi = "madc.hi.cc.u32" if (j < n - 1 or carry) else "madc.hi.u32"
            lines.append(f"{lo} %{2*j}, %{no+j}, %{no+n}, %{2*j}")
            lines.append(f"{hi} %{2*j+1}, %{no+j}, %{no+n}, %{2*j+1}")
        if carry:
            lines.append(f"addc.u32 %{2*n}, %{2*n}, 0")
        L.append(asm_block(lines, outs, ins))
    lines = []
    for c in range(1, 2 * N):
        op = "add.cc.u32" if c == 1 else ("addc.cc.u32" if c < 2 * N - 1 else "addc.u32")
        lines.append(f"{op} %{c-1}, %{c-1}, %{2*N-1+c-1}")
    L.append(asm_block(lines, [f"e[{c}]" for c in range(1, 2 * N)], [f"o[{c}]" for c in range(1, 2 * N)]))
    L.append(f"    for (int k = 0; k < {2*N}; k++) t[k] = e[k];")
    L.append("#else")
    L.append("    unsigned __int128 acc = 0;")
    L.append(f"    for (int c = 0; c < {2*N}; c++) {{")
    L.append("      unsigned __int128 nxt = 0;")
    L.append(f"      for (int i = 0; i < {N}; i++) {{ int j = c - i; if (j < 0 || j >= {N}) continue; uint64_t pr = (uint64_t)a[i] * b[j]; acc += (uint32_t)pr; nxt += pr >> 32; }}")
    L.append("      t[c] = (uint32_t)acc; acc = (acc >> 32) + nxt;")
    L.append("    }")
    L.append("#endif")
    L.append("  }")
    return L


def main():
    L = ["// generated by tools/gen_mont_chains.py - do not edit", "#pragma once", "#include <stdint.h>",
         "template <int N> struct MontChains;"]
    for N in (8, 12):
        L += gen(N)
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    open(OUT, "w").write("\n".join(L) + "\n")
    print("wrote", OUT)


if __name__ == "__main__":
    main()
