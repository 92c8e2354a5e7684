#!/usr/bin/env python3
"""Generator (and CPU checker) of the straight-line PTX bodies in nim_blscurve_b200/csrc/fp_gen.cuh.

Emits, as single inline-asm blocks with block-local registers:
  fp_sqr_ptx     Montgomery squaring: the 66 off-diagonal products are taken once against the doubled operand
                 (78 product terms instead of 144) inside the same even/odd two-accumulator row structure as
                 fp_mul (fp.cuh); 234 IMADs instead of 300.
  fp_mulw_ptx    24-limb product a*b without reduction (144 IMAD.WIDE).
  fp_redc_ptx    Montgomery reduction of a 24-limb value T < p*2^384 to 12 limbs < 2p (156 IMADs).
The last two are the halves of a lazy-reduction Fp2 multiplication (3 wide products, 2 reductions).

`python tools/gen_fp_ptx.py --check` interprets the generated PTX on the CPU (registers + carry flag) against
big-integer arithmetic on random and edge inputs; `--write` (default) rewrites fp_gen.cuh.
The PTX subset used is: mov, add/addc/sub/subc(.cc), mad/madc.lo/.hi(.cc), mul.lo, shf.l.wrap, shl.
"""
import os
import random
import re
import sys

P = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
PL = [(P >> (32 * i)) & 0xffffffff for i in range(12)]
N0 = 0xfffcfffd
R = 1 << 384
M32 = 0xffffffff


class Asm:
    """Collects PTX lines; registers are block-local names, inputs/outputs are %k operands."""

    def __init__(self):
        self.lines = []
        self.regs = []
        self.n = 0

    def reg(self, hint="t"):
        self.n += 1
        nm = f"{hint}{self.n}"
        self.regs.append(nm)
        return nm

    def op(self, s):
        self.lines.append(s + ";")

    def zero(self, hint="z"):
        r = self.reg(hint)
        self.op(f"mov.u32 {r}, 0")
        return r


def lanes_chain(A, acc, pairs, first_cc_in=False, top=None):
    """acc[2L], acc[2L+1] += x*y for (L, x, y) in pairs (increasing L, contiguous), one carry chain.
    first_cc_in: the chain continues a pending carry; top: register that takes the carry out (else none expected)."""
    n = len(pairs)
    for k, (L, x, y) in enumerate(pairs):
        lo, hi = acc[2 * L], acc[2 * L + 1]
        first = k == 0 and not first_cc_in
        last = k == n - 1
        A.op(f"{'mad' if first else 'madc'}.lo.cc.u32 {lo}, {x}, {y}, {lo}")
        if last and top is None:
            A.op(f"madc.hi.u32 {hi}, {x}, {y}, {hi}")
        else:
            A.op(f"madc.hi.cc.u32 {hi}, {x}, {y}, {hi}")
    if top is not None and n:
        A.op(f"addc.u32 {top}, {top}, 0")


def imm(v):
    return "0x%08x" % v


def shift_rows(A, E, O, s_used=True):
    """T >>= 32 by renaming: new E = O (+ fresh top), new O = E >> 64.  Returns (newE, newO, stray)."""
    stray = E[1]
    # E[0] is exactly zero here (Montgomery step) -> reuse it as the fresh top limb of the new E
    newE = O[:12] + [E[0]]
    ztop = A.zero("z")
    newO = E[2:13] + [ztop]
    return newE, newO, stray


def gen_sqr():
    A = Asm()
    a = [f"%{12 + i}" for i in range(12)]
    out = [f"%{i}" for i in range(12)]
    d = [None] * 12      # limbs of 2a
    f = [None] * 12      # a_j << 1
    for j in range(1, 12):
        d[j] = A.reg("d")
        A.op(f"shf.l.wrap.b32 {d[j]}, {a[j - 1]}, {a[j]}, 1")
        f[j] = A.reg("f")
        A.op(f"shl.b32 {f[j]}, {a[j]}, 1")
    E = [A.zero("e") for _ in range(13)]
    O = [A.zero("o") for _ in range(12)]
    m = A.reg("m")

    def v(i, j):          # limb j of the row-i vector: a_i at i, (a_{i+1} << 1) at i+1, limbs of 2a above
        return a[i] if j == i else f[j] if j == i + 1 else d[j]

    for i in range(12):
        ev = [(j // 2, v(i, j), a[i]) for j in range(0, 12, 2) if j >= i]
        od = [((j - 1) // 2, v(i, j), a[i]) for j in range(1, 12, 2) if j >= i]
        if i == 0:
            lanes_chain(A, O, od)
            lanes_chain(A, E, ev, top=E[12])
            A.op(f"mul.lo.u32 {m}, {E[0]}, {imm(N0)}")
            lanes_chain(A, O, [(L, m, imm(PL[2 * L + 1])) for L in range(6)])
            lanes_chain(A, E, [(L, m, imm(PL[2 * L])) for L in range(6)], top=E[12])
        else:
            E, O, s = shift_rows(A, E, O)
            # E[0] is untouched by this row's products (their limbs start at i >= 1): reduce first, so that the carry of
            # the stray limb is absorbed by the full-width reduction chain
            A.op(f"add.cc.u32 {E[0]}, {E[0]}, {s}")
            A.op(f"mul.lo.u32 {m}, {E[0]}, {imm(N0)}")
            lanes_chain(A, O, [(L, m, imm(PL[2 * L + 1])) for L in range(6)], first_cc_in=True)
            lanes_chain(A, E, [(L, m, imm(PL[2 * L])) for L in range(6)], top=E[12])
            if od:
                lanes_chain(A, O, od)
            if ev:
                lanes_chain(A, E, ev, top=E[12])
    # result = O + (E >> 32)
    for k in range(12):
        opn = "add.cc" if k == 0 else ("addc.cc" if k < 11 else "addc")
        A.op(f"{opn}.u32 {out[k]}, {O[k]}, {E[k + 1]}")
    return A


def gen_mulw():
    """t[0..23] = a * b.  Row structure of fp_mul without the reduction: after row i the lowest limb is final."""
    A = Asm()
    out = [f"%{i}" for i in range(24)]
    a = [f"%{24 + i}" for i in range(12)]
    b = [f"%{36 + i}" for i in range(12)]
    E = [A.zero("e") for _ in range(13)]
    O = [A.zero("o") for _ in range(12)]
    for i in range(12):
        ev = [(L, a[2 * L], b[i]) for L in range(6)]
        od = [(L, a[2 * L + 1], b[i]) for L in range(6)]
        if i == 0:
            lanes_chain(A, O, od)
            lanes_chain(A, E, ev, top=E[12])
        else:
            # emit limb i-1 (= E[0]), then T >>= 32:  new E = O + stray, new O = E >> 64
            A.op(f"mov.u32 {out[i - 1]}, {E[0]}")
            stray = E[1]
            ztop, ztop2 = A.zero("z"), A.zero("z")
            E, O = O[:12] + [ztop2], E[2:13] + [ztop]
            A.op(f"add.cc.u32 {E[0]}, {E[0]}, {stray}")
            lanes_chain(A, O, od, first_cc_in=True)
            lanes_chain(A, E, ev, top=E[12])
    A.op(f"mov.u32 {out[11]}, {E[0]}")
    # high half = O + (E >> 32)
    for k in range(12):
        opn = "add.cc" if k == 0 else ("addc.cc" if k < 11 else "addc")
        A.op(f"{opn}.u32 {out[12 + k]}, {O[k]}, {E[k + 1]}")
    return A


def gen_redc():
    """r[0..11] = T / 2^384 mod p up to one subtraction (T = t[0..23] < p * 2^384): 12 Montgomery rows over a sliding
    13-limb window.  Limb 11+i of T enters at window limb 11 right after the i-th shift: the window is then below
    2^382 + 2^384, and below 2^414 after the row's m*p, so nothing is ever carried out of the 13 limbs."""
    A = Asm()
    out = [f"%{i}" for i in range(12)]
    t = [f"%{12 + i}" for i in range(24)]
    E = []
    for k in range(12):
        r = A.reg("e")
        A.op(f"mov.u32 {r}, {t[k]}")
        E.append(r)
    E.append(A.zero("e"))
    O = [A.zero("o") for _ in range(12)]
    m = A.reg("m")
    for i in range(12):
        if i > 0:
            E, O, s = shift_rows(A, E, O)
            A.op(f"add.cc.u32 {E[11]}, {E[11]}, {t[11 + i]}")
            A.op(f"addc.u32 {E[12]}, {E[12]}, 0")
            A.op(f"add.cc.u32 {E[0]}, {E[0]}, {s}")
            A.op(f"mul.lo.u32 {m}, {E[0]}, {imm(N0)}")
            lanes_chain(A, O, [(L, m, imm(PL[2 * L + 1])) for L in range(6)], first_cc_in=True)
        else:
            A.op(f"mul.lo.u32 {m}, {E[0]}, {imm(N0)}")
            lanes_chain(A, O, [(L, m, imm(PL[2 * L + 1])) for L in range(6)])
        lanes_chain(A, E, [(L, m, imm(PL[2 * L])) for L in range(6)], top=E[12])
    # result = O + (E >> 32) + t[23] * 2^352
    A.op(f"add.u32 {E[12]}, {E[12]}, {t[23]}")
    for k in range(12):
        opn = "add.cc" if k == 0 else ("addc.cc" if k < 11 else "addc")
        A.op(f"{opn}.u32 {out[k]}, {O[k]}, {E[k + 1]}")
    return A


# ---------------------------------------------------------------------------------------------------------------
# CPU interpreter of the PTX subset

def run_ptx(A, operands):
    regs = {}
    cf = 0

    def val(x):
        x = x.strip()
        if x.startswith("0x"):
            return int(x, 16)
        if x.isdigit():
            return int(x)
        if x.startswith("%"):
            return operands[int(x[1:])]
        return regs[x]

    def put(x, v):
        x = x.strip()
        assert 0 <= v <= M32
        if x.startswith("%"):
            operands[int(x[1:])] = v
        else:
            regs[x] = v

    for ln in A.lines:
        mm = re.match(r"(\S+)\s+(.*);", ln)
        opc, args = mm.group(1), [z.strip() for z in mm.group(2).split(",")]
        if opc == "mov.u32":
            put(args[0], val(args[1]))
        elif opc == "shl.b32":
            put(args[0], (val(args[1]) << val(args[2])) & M32)
        elif opc == "shf.l.wrap.b32":
            lo, hi, n = val(args[1]), val(args[2]), val(args[3]) & 31
            put(args[0], (((hi << 32) | lo) << n >> 32) & M32)
        elif opc == "mul.lo.u32":
            put(args[0], (val(args[1]) * val(args[2])) & M32)
        elif opc in ("add.cc.u32", "addc.cc.u32", "addc.u32", "add.u32"):
            s = val(args[1]) + val(args[2]) + (cf if opc.startswith("addc") else 0)
            put(args[0], s & M32)
            if ".cc" in opc:
                cf = s >> 32
            else:
                assert s >> 32 == 0, "carry lost by " + ln
        elif opc in ("mad.lo.cc.u32", "madc.lo.cc.u32", "madc.hi.cc.u32", "madc.hi.u32"):
            pr = val(args[1]) * val(args[2])
            part = (pr >> 32) if ".hi" in opc else (pr & M32)
            s = part + val(args[3]) + (cf if opc.startswith("madc") else 0)
            put(args[0], s & M32)
            if ".cc" in opc:
                cf = s >> 32
            else:
                assert s >> 32 == 0, "carry lost by " + ln
        else:
            raise ValueError("unknown op " + ln)
    return operands


def limbs(x, n=12):
    return [(x >> (32 * i)) & M32 for i in range(n)]


def unl(l):
    return sum(v << (32 * i) for i, v in enumerate(l))


def check():
    rng = random.Random(7)
    edge = [0, 1, 2, P - 1, P - 2, (P - 1) // 2, (1 << 381) - 1, (1 << 380), M32, (1 << 352) | M32, P - (1 << 200),
            int("55" * 47, 16) % P, int("aa" * 47, 16) % P, sum(M32 << (64 * i) for i in range(6)) % P]
    vals = edge + [rng.randrange(P) for _ in range(400)]
    rinv = pow(R, -1, P)
    S, W, Rd = gen_sqr(), gen_mulw(), gen_redc()
    for x in vals:
        ops = [0] * 12 + limbs(x)
        got = unl(run_ptx(S, ops)[:12])
        assert got < 2 * P and got % P == x * x * rinv % P, ("sqr", hex(x))
    for i, x in enumerate(vals):
        y = vals[(i * 7 + 3) % len(vals)]
        ops = [0] * 24 + limbs(x) + limbs(y)
        assert unl(run_ptx(W, ops)[:24]) == x * y, ("mulw", hex(x), hex(y))
        # operands up to 2^384 - 1 are legal for the wide product (unreduced sums in the lazy Fp2 product)
        x2, y2 = (x * 9 + 5) % R, (y * 11 + 1) % R
        ops = [0] * 24 + limbs(x2) + limbs(y2)
        assert unl(run_ptx(W, ops)[:24]) == x2 * y2, ("mulw-wide", hex(x2), hex(y2))
    tvals = [0, 1, P * R - 1, P * R - P, (P - 1) * (P - 1), 4 * (P - 1) * (P - 1) % (P * R), R - 1, R, R + 1, (R - 1) * (P - 1) % (P * R)]
    tvals += [rng.randrange(P * R) for _ in range(400)]
    # T = p (mod 2^384): every reduction multiplier is 0xffffffff and the sum before the final subtraction reaches p
    tvals += [P + k * R for k in [0, 1, P - 2, P - 1, (P - 1) // 2] + [rng.randrange(P) for _ in range(100)]]
    for T in tvals:
        ops = [0] * 12 + limbs(T, 24)
        got = unl(run_ptx(Rd, ops)[:12])
        assert got < 2 * P and got % P == T * rinv % P, ("redc", hex(T))
    cnt = lambda A: sum(1 for l in A.lines if l.startswith(("mad", "mul")))
    print("check OK: sqr %d mul-ops (%d lines), mulw %d (%d), redc %d (%d)" %
          (cnt(S), len(S.lines), cnt(W), len(W.lines), cnt(Rd), len(Rd.lines)))


def emit_fn(name, A, nout, nin_groups, doc):
    """C++ wrapper: outputs first (=r), then inputs (r), matching the %k numbering used by the generators."""
    body = ["    asm(\"{\\n\\t\"", "        \".reg .u32 " + ", ".join(A.regs) + ";\\n\\t\""]
    for ln in A.lines:
        body.append(f"        \"{ln}\\n\\t\"")
    body.append("        \"}\"")
    outs = ", ".join(f"\"=&r\"(r[{i}])" for i in range(nout))
    ins = []
    for nm, cnt in nin_groups:
        ins += [f"\"r\"({nm}[{i}])" for i in range(cnt)]
    params = ", ".join(f"const uint32_t *{nm}" for nm, _ in nin_groups)
    txt = f"// {doc}\nBLS_FN void {name}(uint32_t *r, {params}) {{\n" + "\n".join(body)
    txt += f"\n        : {outs}\n        : {', '.join(ins)});\n}}\n"
    return txt


def render():
    """the text of fp_gen.cuh"""
    hdr = """// fp_gen.cuh — GENERATED by tools/gen_fp_ptx.py (do not edit; rerun the generator).  Straight-line PTX bodies:
// every 32x32->64 partial product is a mad.lo.cc/madc.hi.cc pair on an aligned register pair (one IMAD.WIDE.U32.X),
// registers are block-local so the even/odd accumulator swap of each Montgomery row is a renaming, not a move.
// Checked on the CPU by `python tools/gen_fp_ptx.py --check` (PTX interpreter vs big integers) and on the GPU by
// tests/test_gpu_primitives.py against BLST.
#pragma once
#include <stdint.h>
#ifdef __CUDA_ARCH__
namespace bls {

"""
    out = hdr
    out += emit_fn("fp_sqr_ptx", gen_sqr(), 12, [("a", 12)],
                   "r (12 limbs, < 2p) = a*a / 2^384 mod p up to one subtraction of p; 78 + 144 + 12 IMADs")
    out += "\n"
    out += emit_fn("fp_mulw_ptx", gen_mulw(), 24, [("a", 12), ("b", 12)],
                   "r (24 limbs) = a * b, any 384-bit operands; 144 IMADs")
    out += "\n"
    out += emit_fn("fp_redc_ptx", gen_redc(), 12, [("t", 24)],
                   "r (12 limbs, < 2p) = t / 2^384 mod p up to one subtraction, t (24 limbs) < p * 2^384; 156 IMADs")
    out += "\n}  // namespace bls\n#endif  // __CUDA_ARCH__\n"
    return out


def write():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "nim_blscurve_b200", "csrc", "fp_gen.cuh")
    open(path, "w").write(render())
    print("wrote", os.path.normpath(path))


if __name__ == "__main__":
    if "--check" in sys.argv:
        check()
    else:
        check()
        write()
