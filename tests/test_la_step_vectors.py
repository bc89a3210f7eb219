"""Directed vectors for the LA step on step-shaped records (fs_la_step2.cuh, host build) against the oracle's
reference-shaped step (oracle/oracle_cpu.cpp): signed zeros in every operand, products that land in the subnormal range,
and the exponent gaps of the three aligned additions on both sides of 120 and 127.  The step evaluates the (re, im) halves
of each complex operation as one packed pair, with the signs of the rotated operands taken from exact sign flips; these
cases are where a sign or a rounding taken another way would show.  Whatever the step accepts must agree bit for bit --
the sign of a zero included wherever no addition drops an operand -- and what it refuses must be a case it is meant to
refuse."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HARNESS = r"""
#include "oracle_cpu.cpp"
#include "../fractalshark_b200/csrc/fs_la_step2.cuh"

namespace {
struct Counts { uint64_t cases = 0, accepted = 0, refused = 0, mismatches = 0, strict = 0; };

// One case: the oracle's step (LAKernel.cuh:91-127 as oracle_cpu.cpp restates it) and la2::step on the packed record.
void run_case(HC dz, HC Ref, HC ZC, HC CC, HC dc, HC nref, Counts &c) {
    c.cases++;
    HC newdz = mul(dz, add(mul(Ref, HF{1.0f, 1}), dz));
    Reduce(newdz);
    const HF cn = cheb(newdz);
    // threshold just above cheb(newdz) (usable), or the reduced value itself when it is not usable at all
    HF th = cn;
    if (!(th.mantissa >= 1.0f && th.mantissa < 2.0f)) th = HF{1.0f, cn.exp};
    th.exp += 1;
    const bool unusable = cmpPR(cn, th) >= 0;
    HC ndz = dz, z = dz;
    bool by_norm = false;
    int gap2 = 0, gap3 = 0;
    if (!unusable) {
        const HC p = mul(newdz, ZC), q = mul(dc, CC);
        gap2 = p.exp - q.exp;
        ndz = add(p, q);
        gap3 = nref.exp - ndz.exp;
        z = add(nref, ndz);
        HF n0 = cheb(z), nN = cheb(ndz);
        Reduce(n0);
        Reduce(nN);
        by_norm = cmpPR(n0, nN) < 0;
    }
    const int gap1 = (Ref.exp + 1) - dz.exp;
    const fs::la2::Rec rec = fs::la2::pack(fs::HdrC<float>{Ref.re, Ref.im, Ref.exp}, fs::HdrC<float>{ZC.re, ZC.im, ZC.exp},
                                           fs::HdrC<float>{CC.re, CC.im, CC.exp}, fs::Hdr<float>{th.mantissa, th.exp}, 1, 0,
                                           true, fs::HdrC<float>{nref.re, nref.im, nref.exp});
    uint4 qq[4];
    memcpy(qq, &rec, sizeof(rec));
    fs::la2::Out o;
    if (!fs::la2::step(qq[0], qq[1], qq[2], qq[3], dz.re, dz.im, dz.exp, dc.re, dc.im, dc.exp, o)) { c.refused++; return; }
    c.accepted++;
    // where an addition of the reference drops an operand (|gap| >= 120) it returns the other one untouched and the step
    // adds `dropped * 0`, which can turn -0 into +0; everywhere else the sign of a zero must match too
    const bool strict = gap1 > -120 && gap1 < 120 && gap2 > -120 && gap2 < 120 && gap3 > -120 && gap3 < 120;
    if (strict) c.strict++;
    auto same = [&](float a, float b) { return bits(a) == bits(b) || (!strict && a == 0.0f && b == 0.0f); };
    bool ok = o.unusable == unusable;
    if (ok && !unusable)
        ok = same(o.dre, ndz.re) && same(o.dim, ndz.im) && o.de == ndz.exp && same(o.zre, z.re) && same(o.zim, z.im) &&
             o.ze == z.exp && o.rebase == by_norm;
    if (!ok) c.mismatches++;
}
} // namespace

extern "C" void la2_vectors(uint64_t *out) {
    Counts c;
    const float m1 = 1.25f, m2 = -1.625f, m3 = 1.0625f;
    const float signed_vals[] = {0.0f, -0.0f, m1, m2};
    // signed zeros: every component of every complex operand takes +0, -0 or a normal mantissa (dz, dc, ZCoeff, CCoeff,
    // Ref, next Ref), exponents chosen so that no addition drops an operand
    for (float a : signed_vals)
        for (float b : signed_vals)
            for (int which = 0; which < 6; which++) {
                HC dz{m1, m2, -40}, Ref{m3, m2, -41}, ZC{m2, m1, 5}, CC{m1, m3, 3}, dc{m2, m3, -77}, nref{m1, m2, -75};
                HC *t[] = {&dz, &dc, &ZC, &CC, &Ref, &nref};
                t[which]->re = a;
                t[which]->im = b;
                run_case(dz, Ref, ZC, CC, dc, nref, c);
                // the same with the two products of Evaluate cancelling exactly: dc * CCoeff = -(newdz * ZCoeff) gives
                // exact zeros in dz' (and z = Ref' + 0)
                HC newdz = mul(dz, add(mul(Ref, HF{1.0f, 1}), dz));
                Reduce(newdz);
                const HC p = mul(newdz, ZC);
                run_case(dz, Ref, ZC, HC{1.0f, 0.0f, 0}, HC{-p.re, -p.im, p.exp}, nref, c);
            }
    // subnormal products: one component of an operand is tiny, so that ai*bi (or ar*bi) is subnormal or underflows to a
    // signed zero while the other component keeps the sums within [2^-60, 2^60)
    const float tiny[] = {0x1p-70f, -0x1p-70f, 0x1.8p-100f, -0x1.fffffep-126f, 0x1p-149f, -0x1p-149f};
    for (float s : tiny)
        for (int which = 0; which < 8; which++) {
            HC dz{m1, m2, -40}, Ref{m3, m2, -41}, ZC{m2, m1, 5}, CC{m1, m3, 3}, dc{m2, m3, -77}, nref{m1, m2, -75};
            float *f[] = {&dz.re, &dz.im, &dc.re, &dc.im, &ZC.re, &ZC.im, &CC.re, &CC.im};
            *f[which] = s;
            if (which < 2) { dz.re = which == 0 ? s : m1; dz.im = which == 1 ? s : m2; }
            run_case(dz, Ref, ZC, CC, dc, nref, c);
            CC.im = s * 0x1p-20f; // pairs of tiny factors: products below the smallest subnormal
            run_case(dz, Ref, ZC, CC, dc, nref, c);
        }
    // the three aligned additions at exponent gaps either side of the reference's cut (120) and the step's (127)
    const int gaps[] = {0, 1, 23, 24, 25, 118, 119, 120, 121, 126, 127, 128, 140};
    for (int g : gaps)
        for (int sign = -1; sign <= 1; sign += 2)
            for (int which = 0; which < 3; which++) {
                HC dz{m1, m2, -40}, Ref{m3, m2, -41}, ZC{m2, m1, 5}, CC{m1, m3, 3}, dc{m2, m3, -77}, nref{m1, m2, -75};
                if (which == 0) Ref.exp = dz.exp - 1 + sign * g; // 2 Ref against dz
                HC newdz = mul(dz, add(mul(Ref, HF{1.0f, 1}), dz));
                Reduce(newdz);
                const int pe = newdz.exp + ZC.exp;
                if (which == 1) dc.exp = pe - CC.exp - sign * g; // newdz * ZCoeff against dc * CCoeff
                if (which == 2) {
                    const HC nd = add(mul(newdz, ZC), mul(dc, CC));
                    nref.exp = nd.exp + sign * g; // Ref' against dz'
                }
                run_case(dz, Ref, ZC, CC, dc, nref, c);
            }
    out[0] = c.cases; out[1] = c.accepted; out[2] = c.refused; out[3] = c.mismatches; out[4] = c.strict;
}
"""


@pytest.fixture(scope="module")
def vectors_lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("la2_vectors")
    # built in pytest's temporary directory (the tree may be read-only), with the oracle and the product header included
    # by absolute path
    src = str(d / "la2_vectors.cpp")
    with open(src, "w") as f:
        f.write(HARNESS.replace('"oracle_cpu.cpp"', '"' + os.path.join(ROOT, "oracle", "oracle_cpu.cpp") + '"')
                .replace('"../fractalshark_b200/csrc/fs_la_step2.cuh"',
                         '"' + os.path.join(ROOT, "fractalshark_b200", "csrc", "fs_la_step2.cuh") + '"'))
    so = str(d / "libla2vectors.so")
    # the flags of oracle/liblockstep.so: x86 binary32 with explicit fmaf and no contraction is the GPU's IEEE arithmetic
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-mfma", "-ffp-contract=off", "-frounding-math", "-w",
                    "-I/usr/local/cuda/include", "-o", so, src], check=True)
    lib = C.CDLL(so)
    lib.la2_vectors.restype = None
    lib.la2_vectors.argtypes = [C.c_void_p]
    return lib


def test_step_shaped_la_step_directed_vectors(vectors_lib):
    out = (C.c_uint64 * 5)()
    vectors_lib.la2_vectors(out)
    st = dict(zip(("cases", "accepted", "refused", "strict", ), (out[0], out[1], out[2], out[4])), mismatches=out[3])
    assert st["mismatches"] == 0, st
    # most cases are accepted (refusals: exact zeros of a whole operand, the 120..126 gaps, out-of-range sums), and most
    # accepted ones are compared including the sign of zero
    assert st["accepted"] * 2 > st["cases"], st
    assert st["strict"] * 2 > st["accepted"], st
