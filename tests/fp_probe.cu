// fp_probe.cu -- the Fq primitives of csrc/fp.cuh, vm_exec.cuh and vm_exec2.cuh, one case per call.
//
// TEST INFRASTRUCTURE, never linked into the product library.  The same op switch is built twice:
//   * for the host by tests/hostsim/hostsim_fp.cpp (B200BLS_HOSTSIM: PTX emulated, carry flag included),
//   * for the device by tests/test_gpu_fp_probe.py with nvcc and the library's own flags
//     (-DB200BLS_MUL_CALL: fp_mul is the out-of-line fp_mul_call the kernels execute), one thread per case.
// tests/fp_exact.py states the exact integer every op returns; the op numbers are FP_OPS there.
//
// Record layout: in[4][12] and out[2][12] little-endian 32-bit limbs per case.  Predicates return 0 / 1 in
// out[0] limb 0.  Fq2 ops take a = (in[0], in[1]), b = (in[2], in[3]) and return (out[0], out[1]); the
// paired-executor ops return the coefficient computed by role 0 in out[0] and by role 1 in out[1].
#include "../python-bls_b200/csrc/vm_exec2.cuh"

namespace b200bls {

enum ProbeOp {
  P_MUL = 0,       // fp_mul(a, b): the product the executors call
  P_MUL_INLINE,    // fp_mul_inline(a, b)
  P_MUL_LOOPED,    // fp_mul_looped(a, b)
  P_MUL2_LOOPED,   // fp_mul2_looped(a, x, b, y) = (a x + b y) / R; in = a, x, b, y
  P_ADD,
  P_SUB,
  P_NEG,
  P_COND_SUB_2Q,
  P_CANONICAL,
  P_SUB_RAW_2Q,
  P_NEG_RAW_2Q,
  P_XI_COEFF,      // fp_xi_coeff(role, own = in[0], oth = in[1]), role = in[2] limb 0
  P_TO_MONT,
  P_FROM_MONT,
  P_IS_ZERO,
  P_EQ,
  P_RAW_GT,
  P_FP2_MUL,
  P_FP2_SQR,
  P_FP2_MUL_XI,
  P_PAIR_MUL2,     // vm_exec2 MUL2: fp_mul2_oth, then the two-row product with the operands env.mul2 streams
  P_PAIR_SQR2,     // vm_exec2 SQR2: fp_sqr2_coeff
  P_PAIR_XI,       // vm_exec2 MULXI2 and POST_XI: fp_xi_coeff with the partner's coefficient
  P_INV,
  P_IS_SQUARE,
  P_N_OPS
};

FP_DEV void probe_load(fp& x, const uint32_t* src) {
  for (int i = 0; i < NL; i++) x.v[i] = src[i];
}

FP_DEV void probe_one(int op, const uint32_t* in, uint32_t* out) {
  fp a, b, c, d, r, s;
  probe_load(a, in);
  probe_load(b, in + NL);
  probe_load(c, in + 2 * NL);
  probe_load(d, in + 3 * NL);
  fp_set_zero(r);
  fp_set_zero(s);
  switch (op) {
    case P_MUL: fp_mul(r, a, b); break;
    case P_MUL_INLINE: fp_mul_inline(r, a, b); break;
    case P_MUL_LOOPED: fp_mul_looped(r, a, b); break;
    case P_MUL2_LOOPED: fp_mul2_looped(r, a, b, c, d); break;
    case P_ADD: fp_add(r, a, b); break;
    case P_SUB: fp_sub(r, a, b); break;
    case P_NEG: fp_neg(r, a); break;
    case P_COND_SUB_2Q: fp_cond_sub_2q(r, a); break;
    case P_CANONICAL: fp_canonical(r, a); break;
    case P_SUB_RAW_2Q: fp_sub_raw_2q(r, a, b); break;
    case P_NEG_RAW_2Q: fp_neg_raw_2q(r, a); break;
    case P_XI_COEFF: fp_xi_coeff(r, (c.v[0] & 1u) != 0, a, b); break;
    case P_TO_MONT: fp_to_mont(r, a); break;
    case P_FROM_MONT: fp_from_mont(r, a); break;
    case P_IS_ZERO: r.v[0] = fp_is_zero(a); break;
    case P_EQ: r.v[0] = fp_eq(a, b); break;
    case P_RAW_GT: r.v[0] = fp_raw_gt(a, b); break;
    case P_FP2_MUL:
    case P_FP2_SQR:
    case P_FP2_MUL_XI: {
      fp2 x, y, z;
      x.c0 = a, x.c1 = b, y.c0 = c, y.c1 = d;
      if (op == P_FP2_MUL)
        fp2_mul(z, x, y);
      else if (op == P_FP2_SQR)
        fp2_sqr(z, x);
      else
        fp2_mul_xi(z, x);
      r = z.c0, s = z.c1;
    } break;
    case P_PAIR_MUL2: {
      // thread `role` owns a_role and b_role; env.mul2(z, own, oth', slot b, swap = role) streams x = b_own,
      // y = b_oth for role 0 and x = b_oth, y = b_own for role 1
      fp o;
      fp_mul2_oth(o, false, b);
      fp_mul2_looped(r, a, c, o, d);
      fp_mul2_oth(o, true, a);
      fp_mul2_looped(s, b, c, o, d);
    } break;
    case P_PAIR_SQR2:
      fp_sqr2_coeff(r, false, a, b);
      fp_sqr2_coeff(s, true, b, a);
      break;
    case P_PAIR_XI:
      fp_xi_coeff(r, false, a, b);
      fp_xi_coeff(s, true, b, a);
      break;
    case P_INV: r = fp_inv(a); break;
    case P_IS_SQUARE: r.v[0] = fp_is_square(a); break;
    default: r.v[0] = 0xdeadbeefu; break;
  }
  for (int i = 0; i < NL; i++) {
    out[i] = r.v[i];
    out[NL + i] = s.v[i];
  }
}

}  // namespace b200bls

#ifndef B200BLS_HOSTSIM
#include <cuda_runtime.h>

__global__ void fp_probe_kernel(const int* ops, const uint32_t* in, uint32_t* out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) b200bls::probe_one(ops[i], in + i * 4 * b200bls::NL, out + i * 2 * b200bls::NL);
}

// 0 on success, else the CUDA error code
extern "C" int fp_probe_run(long long n, const int* ops, const uint32_t* in, uint32_t* out) {
  const size_t b_ops = n * sizeof(int), b_in = n * 4 * b200bls::NL * 4, b_out = n * 2 * b200bls::NL * 4;
  int* d_ops = nullptr;
  uint32_t *d_in = nullptr, *d_out = nullptr;
  cudaError_t e = cudaMalloc(&d_ops, b_ops);
  if (e == cudaSuccess) e = cudaMalloc(&d_in, b_in);
  if (e == cudaSuccess) e = cudaMalloc(&d_out, b_out);
  if (e == cudaSuccess) e = cudaMemcpy(d_ops, ops, b_ops, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(d_in, in, b_in, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(d_out, 0xff, b_out);
  if (e == cudaSuccess) {
    fp_probe_kernel<<<(unsigned)((n + 127) / 128), 128>>>(d_ops, d_in, d_out, n);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(out, d_out, b_out, cudaMemcpyDeviceToHost);
  cudaFree(d_ops);
  cudaFree(d_in);
  cudaFree(d_out);
  return (int)e;
}
#endif
