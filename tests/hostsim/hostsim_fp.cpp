// Host build of the Fq primitive probe (tests/fp_probe.cu) with the PTX instructions emulated (carry flag
// included).  TEST INFRASTRUCTURE: lets the CPU-only box check the exact limb/carry sequences of csrc/fp.cuh,
// vm_exec.cuh and vm_exec2.cuh against tests/fp_exact.py.  Never linked into the product library.
#define B200BLS_HOSTSIM 1
#include "../fp_probe.cu"

extern "C" int hs_fp_probe_run(long long n, const int* ops, const uint32_t* in, uint32_t* out) {
  for (long long i = 0; i < n; i++) b200bls::probe_one(ops[i], in + i * 4 * b200bls::NL, out + i * 2 * b200bls::NL);
  return 0;
}
