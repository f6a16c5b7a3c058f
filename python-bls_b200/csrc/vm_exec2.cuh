// vm_exec2.cuh -- one instruction of the b200-bls field VM, executed by a PAIR of threads.
//
// Same instruction set and same programs as vm_exec.cuh (bls_b200/vm/isa.py); what changes is who
// computes what.  Two adjacent threads of a warp share one batch item: thread `role` (0 / 1) owns
// coefficient `role` of every Fq2 slot of the item's workspace -- fp cell c = 2 * slot + half
// belongs to the thread with role == half.  An Fq2 instruction is then one Fq-sized piece of work
// per thread with no communication:
//   MUL2   c0 = a0 b0 + (2q - a1) b1,  c1 = a1 b0 + a0 b1   one two-row Montgomery product each
//                                                            (fp.cuh: 444 limb products, lazily reduced)
//   SQR2   c0 = (a0 + a1)(a0 - a1 + 2q),  c1 = (2 a1) a0     one product each
//   ADD2 / SUB2 / TRI2 / CSEL2 / spills / fills              own coefficient only
// so a thread needs 12 + 12 operand registers and 24 accumulators instead of a whole Fq2 product's
// state, and an SM holds twice as many warps on the same per-item workspace (vm_kernel2.cuh).
// Operands of the partner are read from its shared-memory column, or -- for Tensor-Memory slots,
// whose lanes are private -- loaded by the partner and exchanged with shuffles (Env::ld_oth).
// Fq-granular instructions (hashing, roots, I/O conversions, flags) are computed by BOTH threads on
// the same operands (Env::ld_cell) and stored by the owner of the destination cell: the lanes of a
// warp instruction are paid for either way, and every flag is then known to both threads.
#pragma once
#include "vm_exec.cuh"

namespace b200bls {

// r = 2q - x as integers, for weakly reduced x: in (0, 2q]
FP_DEV void fp_neg_raw_2q(fp& r, const fp& x) {
  r.v[0] = sub_cc(Q2L(0), x.v[0]);
#pragma unroll
  for (int i = 1; i < NL - 1; i++) r.v[i] = subc_cc(Q2L(i), x.v[i]);
  r.v[NL - 1] = subc(Q2L(NL - 1), x.v[NL - 1]);
}

// own -/+ other: coefficient `role` of (x0 + x1 u)(1 + u) = (x0 - x1) + (x0 + x1) u
FP_DEV void fp_xi_coeff(fp& r, bool role, const fp& own, const fp& oth) {
  fp n, t;
  fp_neg_raw_2q(n, oth);
  fp_select(t, role, oth, n);
  fp_add(r, own, t);  // own < 2q, t <= 2q
}

// coefficient `role` of (own + oth u)^2 for role 0 (own = a0) / role 1 (own = a1):
// role 0: (a0 + a1)(a0 - a1 + 2q); role 1: (a1 + a1) a0 -- sums left unreduced (< 4q)
FP_DEV void fp_sqr2_coeff(fp& z, bool role, const fp& own, const fp& oth) {
  fp p, dd, x;
  fp_select(x, role, own, oth);
  fp_add_raw(p, own, x);
  fp_sub_raw_2q(dd, own, oth);
  fp_select(x, role, oth, dd);
  fp_mul(z, p, x);
  fp_cond_sub_2q(z, z);  // never fires: role 0 < 1.92 q ((a0 + a1)(a0 - a1 + 2q) <= (a0 + q)^2), role 1 < 1.82 q
}

// the second row's left operand of MUL2: role 0 computes a0 b0 + (2q - a1) b1, role 1 a1 b0 + a0 b1
FP_DEV void fp_mul2_oth(fp& r, bool role, const fp& oth) {
  fp n;
  fp_neg_raw_2q(n, oth);
  fp_select(r, role, oth, n);
}

template <class Env>
FP_DEV int vm_exec2(Env& env, uint32_t w0, uint32_t w1) {
  const int op = w0 & 0xff;
  const int aux = (w0 >> 8) & 0xff;
  const int d = (w0 >> 16) & 0xfff;
  const int a = w1 & 0xffff;
  const int b = w1 >> 16;
  const bool role = env.role() != 0;
  if ((unsigned)(op - OP_ADD2) <= (unsigned)(OP_SPILL2 - OP_ADD2)) {
    fp z;
    if (op <= OP_MUL2) {
      if (op <= OP_SUB2) {
        fp x, y;
        env.ld_own(a >> 1, x);
        env.ld_own(b >> 1, y);
        if (op == OP_ADD2)
          fp_add(z, x, y);
        else
          fp_sub(z, x, y);
      } else if (op == OP_SQR2) {
        fp own, oth;
        env.ld_own(a >> 1, own);
        env.ld_oth(a >> 1, oth);
        fp_sqr2_coeff(z, role, own, oth);
      } else {
        fp own, oth;
        env.ld_own(a >> 1, own);
        env.ld_oth(a >> 1, oth);
        fp_mul2_oth(oth, role, oth);
        // role 0: own * b_own + (2q - oth) * b_oth; role 1: own * b_oth + oth * b_own
        env.mul2(z, own, oth, b >> 1, role);
      }
    } else if (op <= OP_TRI2) {
      if (op == OP_MULXI2) {
        fp own, oth;
        env.ld_own(a >> 1, own);
        env.ld_oth(a >> 1, oth);
        fp_xi_coeff(z, role, own, oth);
      } else {
        fp x, y, u;
        env.ld_own(a >> 1, x);
        env.ld_own(b >> 1, y);
        if (aux)
          fp_add(u, x, y);
        else
          fp_sub(u, x, y);
        fp_add(u, u, u);
        fp_add(z, u, x);
      }
    } else if (op == OP_FILL2) {
      env.ld_cold_own(a, z);
      env.st_own(d >> 1, z);
      if (aux & 0x80) env.discard_cold_own(aux & 0x7f);   // after the store: the loaded registers have arrived
      return 0;
    } else {
      if (aux & 0x80) env.discard_cold_own(aux & 0x7f);   // a dead cold copy riding on this spill
      env.ld_own(a >> 1, z);
      env.st_cold_own(d, z);
      return 0;
    }
    const int post = w0 >> 28;
    if (post) {
      if (post <= POST_RSUB) {
        fp c;
        env.ld_own(aux >> 1, c);
        if (post == POST_ADD)
          fp_add(z, z, c);
        else if (post == POST_SUB)
          fp_sub(z, z, c);
        else
          fp_sub(z, c, z);
      } else if (post == POST_XI) {
        fp zo = z;
        env.xchg(zo);
        fp_xi_coeff(z, role, z, zo);
      } else {
        fp_add(z, z, z);
      }
    }
    env.st_own(d >> 1, z);
    return 0;
  }
  switch (op) {
    case OP_NEG2: {
      fp x, z;
      env.ld_own(a >> 1, x);
      fp_neg(z, x);
      env.st_own(d >> 1, z);
    } break;
    case OP_DBL2: {
      fp x, z;
      env.ld_own(a >> 1, x);
      fp_add(z, x, x);
      env.st_own(d >> 1, z);
    } break;
    case OP_CONJ2: {
      fp x, n, z;
      env.ld_own(a >> 1, x);
      fp_neg(n, x);
      fp_select(z, role, n, x);
      env.st_own(d >> 1, z);
    } break;
    case OP_MOV2: {
      fp x;
      env.ld_own(a >> 1, x);
      env.st_own(d >> 1, x);
    } break;
    case OP_MULFP2: {
      fp x, y, z;
      env.ld_own(a >> 1, x);
      env.ld_cell(b, y);
      fp_mul(z, x, y);
      env.st_own(d >> 1, z);
    } break;
    case OP_MUL1: {
      fp x, y, z;
      env.ld_cell(a, x);
      env.ld_cell(b, y);
      fp_mul(z, x, y);
      env.st_cell(d, z);
    } break;
    case OP_SQR1: {
      fp x, z;
      env.ld_cell(a, x);
      fp_sqr(z, x);
      env.st_cell(d, z);
    } break;
    case OP_ADD1: {
      fp x, y, z;
      env.ld_cell(a, x);
      env.ld_cell(b, y);
      fp_add(z, x, y);
      env.st_cell(d, z);
    } break;
    case OP_SUB1: {
      fp x, y, z;
      env.ld_cell(a, x);
      env.ld_cell(b, y);
      fp_sub(z, x, y);
      env.st_cell(d, z);
    } break;
    case OP_NEG1: {
      fp x, z;
      env.ld_cell(a, x);
      fp_neg(z, x);
      env.st_cell(d, z);
    } break;
    case OP_DBL1: {
      fp x, z;
      env.ld_cell(a, x);
      fp_add(z, x, x);
      env.st_cell(d, z);
    } break;
    case OP_MOV1: {
      fp x;
      env.ld_cell(a, x);
      env.st_cell(d, x);
    } break;
    case OP_LDC1: {
      fp x;
      env.ldc(a, x);
      env.st_cell(d, x);
    } break;
    case OP_LDC2: {
      fp x;
      env.ldc(a + (role ? 1 : 0), x);
      env.st_own(d >> 1, x);
    } break;
    case OP_FZERO1: {
      fp x;
      env.ld_cell(a, x);
      env.set_flag(d, fp_is_zero(x));
    } break;
    case OP_FZERO2: {
      fp x, y;
      env.ld_own(a >> 1, x);
      env.ld_oth(a >> 1, y);
      env.set_flag(d, fp_is_zero(x) && fp_is_zero(y));
    } break;
    case OP_FGTHALF: {
      fp x, s, h;
      env.ld_cell(a, x);
      fp_from_mont(s, x);
#pragma unroll
      for (int i = 0; i < NL; i++) h.v[i] = HALFQL(i);
      env.set_flag(d, fp_raw_gt(s, h));
    } break;
    case OP_INV1: {
      fp x;
      env.ld_cell(a, x);
      env.st_cell(d, fp_inv(x));
    } break;
    case OP_FSQR1: {
      fp x;
      env.ld_cell(a, x);
      env.set_flag(d, fp_is_square(x));
    } break;
    case OP_FEQ1: {
      fp x, y;
      env.ld_cell(a, x);
      env.ld_cell(b, y);
      env.set_flag(d, fp_eq(x, y));
    } break;
    case OP_FEQ2: {
      fp x, y;
      env.ld_own(a >> 1, x);
      env.ld_own(b >> 1, y);
      bool e = fp_eq(x, y);
      env.ld_oth(a >> 1, x);
      env.ld_oth(b >> 1, y);
      env.set_flag(d, e && fp_eq(x, y));
    } break;
    case OP_FAND:
      env.set_flag(d, env.get_flag(a) && env.get_flag(b));
      break;
    case OP_FOR:
      env.set_flag(d, env.get_flag(a) || env.get_flag(b));
      break;
    case OP_FXOR:
      env.set_flag(d, env.get_flag(a) != env.get_flag(b));
      break;
    case OP_FNOT:
      env.set_flag(d, !env.get_flag(a));
      break;
    case OP_FSET:
      env.set_flag(d, (a & 1) != 0);
      break;
    case OP_FBIT: {
      uint32_t byte = env.ld_byte(a, (aux ? aux : 31) - (b >> 3));  // aux = scalar bytes - 1 (0: 32-byte scalars)
      env.set_flag(d, ((byte >> (b & 7)) & 1) != 0);
    } break;
    case OP_FLDB:
      env.set_flag(d, env.ld_byte(a, b) != 0);
      break;
    case OP_FACTIVE:
      env.set_flag(d, env.active());
      break;
    case OP_CSEL2: {
      fp x, y, z;
      env.ld_own(a >> 1, x);
      env.ld_own(b >> 1, y);
      fp_select(z, env.get_flag(aux), x, y);
      env.st_own(d >> 1, z);
    } break;
    case OP_CSEL1: {
      fp x, y, z;
      env.ld_cell(a, x);
      env.ld_cell(b, y);
      fp_select(z, env.get_flag(aux), x, y);
      env.st_cell(d, z);
    } break;
    case OP_LDBE48: {
      fp raw, m;
      env.ld_be(a, b * 16, 12, raw);
      if (aux) raw.v[NL - 1] &= 0x1fffffffu;
      fp_to_mont(m, raw);
      env.st_cell(d, m);
    } break;
    case OP_LDBE32: {
      fp raw, m;
      env.ld_be(a, b * 16, 8, raw);
      fp_to_mont(m, raw);
      env.st_cell(d, m);
    } break;
    case OP_STBE48: {
      fp x, s;
      env.ld_cell(a, x);
      fp_from_mont(s, x);
      env.st_be48(d, b * 16, s, aux != 0, a & 1);
    } break;
    case OP_STFLAG:
      env.st_byte(d, b, env.get_flag(a) ? 1 : 0, aux != 0);
      break;
    case OP_LDRAW2: {
      fp x;
      env.ld_raw_own(a, b, x);
      env.st_own(d >> 1, x);
    } break;
    case OP_STRAW2: {
      fp x;
      env.ld_own(a >> 1, x);
      env.st_raw_own(d, b, x, false);
    } break;
    case OP_STRAWB2: {
      fp x;
      env.ld_own(a >> 1, x);
      env.st_raw_own(d, b, x, true);
    } break;
    case OP_SYNC:
      env.sync();
      break;
    case OP_XMOV2: {
      fp x;
      env.ld_lane_own(a >> 1, b, x);
      env.st_own(d >> 1, x);
    } break;
    case OP_DISCARD2:
      env.discard_cold_own(d);
      break;
    case OP_SKIPZ:
      return env.any_flag(d) ? 0 : a;
    case OP_END:
      return -1;
    default:
      break;
  }
  return 0;
}

}  // namespace b200bls
