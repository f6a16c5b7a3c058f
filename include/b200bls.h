/* b200bls.h -- C ABI of libb200bls.so, the B200 (sm_100a) engine for python-bls's
 * pairing / aggregation hot path.
 *
 * This is the drop-in boundary (SURVEY.md 8b).  The reference's own plugin seam is the set
 * of tuple-in / tuple-out functions that bls_py/fields_t.py:1218-1265 re-imports from the
 * Cython module extmod/bls_py/fields_t_c.pyx -- one field operation, one point operation or
 * one pairing per Python call.  A GPU needs batches, so every entry point here is the
 * *batched, byte-buffer* form of one of those functions; the citation on each declaration
 * names the reference function(s) it replaces (paths relative to /root/reference).
 *
 * Encoding = the reference's own serialize() bytes, so parity is a memcmp:
 *   Fq      48 bytes big-endian                       (bls_py/fields.py:87-88)
 *   Fq2/6/12  2/6/12 such coefficients in ZT order      (bls_py/fields.py:273-278)
 *   G1 affine  x || y            =  96 bytes, point at infinity = all zero bytes
 *   G2 affine  x.c0 x.c1 y.c0 y.c1 = 192 bytes, point at infinity = all zero bytes
 *   G1 / G2 compressed 48 / 96 bytes                  (bls_py/ec.py:94-111)
 *   scalars 32 bytes big-endian;  message hashes 32 bytes
 * Inputs are reduced mod q on load exactly like Fq(Q, int) does (bls_py/fields.py:59-61).
 *
 * Conventions: every function returns 0 on success and a negative B200BLS_E_* code on
 * failure (no exceptions cross the ABI; b200bls_last_error() describes the last failure of
 * the calling thread).  The caller owns every buffer; the library keeps no pointer after a
 * call returns.  Host-buffer entry points copy to the GPU, run, copy back and synchronise.
 * The *_dev variants take device pointers obtained from b200bls_malloc() and only enqueue
 * work on the library's stream (call b200bls_sync()).  One process drives one GPU
 * (b200bls_init(device)); a global mutex serialises calls.  There is NO CPU fallback: without
 * a CUDA device b200bls_init() fails and every compute call returns B200BLS_E_NOT_INIT.
 */
#ifndef B200BLS_H
#define B200BLS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200BLS_OK 0
#define B200BLS_E_NOT_INIT (-1)
#define B200BLS_E_CUDA (-2)
#define B200BLS_E_ARG (-3)
#define B200BLS_E_NOMEM (-4)
#define B200BLS_E_PROGRAM (-5)

/* ---- lifecycle ---------------------------------------------------------------------- */
int b200bls_init(int device);            /* select GPU `device`, upload the field programs */
void b200bls_shutdown(void);
const char* b200bls_last_error(void);
int b200bls_sm_count(void);              /* SMs of the initialised device, 0 if none */
int b200bls_sync(void);                  /* wait for the library stream */
/* The library owns 8 CUDA streams.  *_dev and *_async entry points enqueue on the stream
 * selected here (default 0); launches on different streams overlap, which removes the tail-wave
 * loss between back-to-back batches.  b200bls_sync() waits for all of them; the timer brackets
 * all of them.  Synchronous host-buffer entry points run on the selected stream.  The selection is per
 * calling thread (thread-local): host threads driving different streams do not interfere. */
int b200bls_set_stream(int idx);
int b200bls_stream_count(void);
/* Launch shape = CTAs of 128 threads per SM: 1 (18 shared + 21 Tensor-Memory Fq2 workspace slots
 * per thread), 2 (9 + 10) or 3 (6 + 5); 4 = the "wide" shape, ONE CTA of 384 threads per SM that
 * owns all 512 Tensor-Memory columns (6 + 7 slots per thread; programs without block-level
 * reductions only, the others fall back to 3).  More warps per SM = more throughput, but a
 * longer single pass.  5 = ONE CTA of 512 threads per SM (16 warps, 4 + 5 slots per thread): 0.97x
 * the throughput of 4 on whole waves, but 75,776 items in one pass -- what the automatic choice
 * takes for an isolated batch that is a little more than whole 384-item waves (65,536 pairings).
 * 0 (default, or environment variable B200BLS_CTAS_PER_SM) chooses per call
 * the shape that finishes an isolated batch soonest; pipelines that keep batches in flight on
 * several streams should select 4. */
int b200bls_set_ctas_per_sm(int n);
int b200bls_get_ctas_per_sm(void);

/* ---- device / pinned memory for resident-data pipelines and benchmarks ----------------- */
void* b200bls_malloc(size_t bytes);
void b200bls_free(void* dev_ptr);
void* b200bls_host_alloc(size_t bytes);  /* pinned host memory */
void b200bls_host_free(void* host_ptr);
int b200bls_h2d(void* dev_dst, const void* host_src, size_t bytes);   /* async on the stream */
int b200bls_d2h(void* host_dst, const void* dev_src, size_t bytes);   /* async on the stream */
/* CUDA-event timing on the library stream: tic, enqueue work, toc -> milliseconds */
int b200bls_timer_start(void);
int b200bls_timer_stop(float* ms_out);
/* kernels launched by this library since init (bench.py's gpu_launches) */
uint64_t b200bls_launch_count(void);

/* Integer-multiply roofline microbenchmark (SURVEY.md 8d).  variant 0: IMAD (mad.lo),
 * 1: IMAD.HI, 2: IMAD.WIDE.U32, 3: IMAD.WIDE.U32.X carry chains as in the Montgomery
 * product, 4: DFMA (FP64 pipe), 5: even warps variant 3 and odd warps variant 4 (do the two pipes
 * overlap?).  Launches blocks_per_sm x SMs CTAs of `threads` threads (<= 256); reports
 * multiply-add instructions per second (best of 4 timed launches, CUDA events). */
int b200bls_microbench_imad(int variant, int blocks_per_sm, int threads, int iters,
                            double* ops_per_second, float* ms_out);

/* ---- generic program launch (device pointers) ------------------------------------------ */
/* Runs the embedded field program `name` over n_items; bufs[i] / strides[i] (bytes per item)
 * are the program's numbered byte buffers.  Typed entry points below are thin wrappers. */
int b200bls_run_program_dev(const char* name, size_t n_items, void* const* bufs,
                            const int64_t* strides, int n_bufs);
int b200bls_program_info(const char* name, int* n_ins, int* n_slots, int* n_cold);

/* ---- field tower: level in {1, 2, 6, 12} coefficients -------------------------------------
 * op: 0 add, 1 sub, 2 mul, 3 sqr, 4 neg, 5 inv.  a, b, out: n x (48 * level) bytes.
 * Replaces the fq_ / fq2_ / fq6_ / fq12_ functions of bls_py/fields_t.py:47-554
 * (add, sub, neg, mul, invert)
 * and the operator methods of Fq/Fq2/Fq6/Fq12 (bls_py/fields.py:35-764). b is ignored for
 * unary ops.  Inverse of 0 is 0 as in fq_invert (fields_t.py:47-55). */
int b200bls_field_op_batch(int level, int op, const uint8_t* a, const uint8_t* b,
                           uint8_t* out, size_t n);
int b200bls_field_op_batch_dev(int level, int op, const void* a, const void* b, void* out,
                               size_t n);

/* x -> x^(q^i): fq2_qi_pow / fq6_qi_pow / fq12_qi_pow (fields_t.py:104-110, 203-212, 355-364, coefficient table
 * 1133-1216; pinned by tests.py:60-68).  level in {2, 6, 12}, 0 <= i < level.  a, out: n x (48 * level). */
int b200bls_field_frob_batch(int level, int i, const uint8_t* a, uint8_t* out, size_t n);
/* x -> x^e: fq_pow / fq2_pow / fq6_pow / fq12_pow (fields_t.py:58-68, 92-101, 344-352).  level in {1, 2, 6, 12};
 * e48: n exponents of 48 big-endian bytes (0 <= e < 2^384; e = 0 gives one). */
int b200bls_field_pow_batch(int level, const uint8_t* a, const uint8_t* e48, uint8_t* out, size_t n);
/* Fq.modsqrt (fields.py:199-205) / Fq2.modsqrt (fields.py:463-482, "complex method"): the reference's own root,
 * bit for bit.  level in {1, 2}.  ok[i] = 0 (and a zero root) where the reference raises
 * ValueError('No sqrt exists').  An Fq2 element with c1 = 0 goes through the Fq root as in the reference
 * (which then returns an Fq object): the root is in c0, c1 = 0. */
int b200bls_field_sqrt_batch(int level, const uint8_t* a, uint8_t* out, uint8_t* ok, size_t n);

/* ---- pairing ------------------------------------------------------------------------------
 * P: n x 96 (G1 affine), Q: n x 192 (G2 affine). */
/* fq_miller_loop + fq12_final_exp per pair (fields_t.py:1091-1128; pairing.py:76-81
 * ate_pairing).  out: n x 576. */
int b200bls_pairing_batch(const uint8_t* P, const uint8_t* Q, uint8_t* out, size_t n);
/* Asynchronous host-buffer form: enqueues H2D copy, kernel and D2H copy on the selected stream
 * and returns; call b200bls_sync() before reading `out`.  Use pinned host buffers
 * (b200bls_host_alloc) and alternate b200bls_set_stream() to overlap consecutive batches. */
int b200bls_pairing_batch_async(const uint8_t* P, const uint8_t* Q, uint8_t* out, size_t n);
int b200bls_pairing_batch_dev(const void* P, const void* Q, void* out, size_t n);
/* fq12_final_exp (fields_t.py:1124-1128; pairing.py:68-73).  in/out: n x 576. */
int b200bls_final_exp_batch(const uint8_t* in, uint8_t* out, size_t n);
int b200bls_final_exp_batch_dev(const void* in, void* out, size_t n);
/* Miller loop alone.  NOT byte-comparable with fq_miller_loop (fields_t.py:1091-1111): the
 * value differs from the reference's by a factor that the final exponentiation removes
 * (projective, denominator-free lines).  final_exp(out) is canonical. out: n x 576. */
int b200bls_miller_loop_batch(const uint8_t* P, const uint8_t* Q, uint8_t* out, size_t n);
int b200bls_miller_loop_batch_dev(const void* P, const void* Q, void* out, size_t n);

/* Product of Miller loops without the final exponentiation: stage one of
 * fq_ate_pairing_multi (fields_t.py:1114-1121).  out: 576 bytes.  This (non-canonical)
 * value is what ranks exchange in a multi-GPU ate_pairing_multi / aggregate verification:
 * multiply the per-rank values (b200bls_field_op_batch level 12, mul), then
 * b200bls_final_exp_batch once. */
int b200bls_miller_product(const uint8_t* P, const uint8_t* Q, uint8_t* out, size_t n);
int b200bls_miller_product_dev(const void* P, const void* Q, void* out, size_t n);
/* fq_ate_pairing_multi (fields_t.py:1114-1121; pairing.py:84-92 ate_pairing_multi):
 * prod_i miller(P_i, Q_i), one final exponentiation.  out: 576 bytes. */
int b200bls_pairing_multi(const uint8_t* P, const uint8_t* Q, uint8_t* out, size_t n);
int b200bls_pairing_multi_dev(const void* P, const void* Q, void* out, size_t n);
/* Many fq_ate_pairing_multi products in one device pass: n_groups products
 * prod_{j in [off[g], off[g+1])} e(P_j, Q_j), one final exponentiation each.
 * P: total x 96, Q: total x 192 (total = off[n_groups]); off: n_groups + 1 uint64, off[0] = 0, non-decreasing,
 * total <= 2^32 - 1, n_groups <= 2^31 - 1.
 * check = 0: out = n_groups x 576 canonical Fq12 bytes (an empty group gives one, as fields_t.py:1117);
 * check = 1: out = n_groups bytes, 1 iff the product is one (the cheaper final_exp_check).
 * Other offsets or check values return B200BLS_E_ARG; n_groups = 0 does nothing.  The host form checks the offsets
 * on the host.  The _dev form takes `off` in device memory as well: its offsets are checked on the device before any
 * pairing runs, and it synchronises the stream once to read that check and the chunk counts. */
int b200bls_pairing_multi_batch(int check, const uint8_t* P, const uint8_t* Q, const uint64_t* off,
                                size_t n_groups, uint8_t* out);
int b200bls_pairing_multi_batch_dev(int check, const void* P, const void* Q, const void* off,
                                    size_t n_groups, void* out);

/* ---- curve arithmetic (affine in, affine out; infinity = zero bytes) --------------------------
 * G1 points 96 bytes, G2 points 192 bytes, scalars 32 bytes big-endian (any value < 2^256;
 * the reference's `c % Q == 0 -> infinity` early-out, fields_t.py:710/729, only triggers for
 * c = 0 in that range and 0 * P is infinity anyway). */
/* fq_scalar_mult_jacobian / fq2_scalar_mult_jacobian + to_affine (fields_t.py:705-740,
 * 609-632; ec.py:365-391 scalar_mult_jacobian; keys.py:119-132 get_public_key / sign). */
int b200bls_g1_scalar_mul_batch(const uint8_t* pts, const uint8_t* scalars, uint8_t* out, size_t n);
int b200bls_g1_scalar_mul_batch_dev(const void* pts, const void* scalars, void* out, size_t n);
int b200bls_g2_scalar_mul_batch(const uint8_t* pts, const uint8_t* scalars, uint8_t* out, size_t n);
int b200bls_g2_scalar_mul_batch_dev(const void* pts, const void* scalars, void* out, size_t n);
/* fq_add_points_jacobian / fq2_add_points_jacobian + to_affine (fields_t.py:762-819;
 * ec.py:315-342).  P + P doubles for G1 too (the reference's TypeError at fields_t.py:781 is
 * a defect, not behaviour). */
int b200bls_g1_add_batch(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n);
int b200bls_g2_add_batch(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n);
/* Sum of n points -> one point: the folds of BLS.aggregate_pub_keys(secure=False)
 * (bls.py:204-223) and BLS.aggregate_sigs_simple (bls.py:13-26) as a strided per-thread
 * fold + CTA tree + one final CTA.  n = 0 gives infinity. */
int b200bls_g1_sum(const uint8_t* pts, uint8_t* out, size_t n);
int b200bls_g1_sum_dev(const void* pts, void* out, size_t n);
int b200bls_g2_sum(const uint8_t* pts, uint8_t* out, size_t n);
int b200bls_g2_sum_dev(const void* pts, void* out, size_t n);
/* Multi-scalar multiplication sum_i k_i * P_i -> one point: the secure aggregation folds
 * sum T_i * sig_i (bls.py:29-56, 132-144) and sum T_i * pk_i (bls.py:217-221), where the reference
 * runs one double-and-add ladder per point and a left fold.  pts: n affine points, scalars:
 * n x 32 big-endian bytes.  Bucket method (11-bit windows, counting sort, one thread per
 * bucket) from 65,536 points up, per-point ladders + reduction below.  n = 0 gives infinity. */
int b200bls_g1_msm(const uint8_t* pts, const uint8_t* scalars, uint8_t* out, size_t n);
int b200bls_g1_msm_dev(const void* pts, const void* scalars, void* out, size_t n);
int b200bls_g2_msm(const uint8_t* pts, const uint8_t* scalars, uint8_t* out, size_t n);
int b200bls_g2_msm_dev(const void* pts, const void* scalars, void* out, size_t n);
/* PublicKey.from_bytes (keys.py:29-40) / Signature.from_bytes (signature.py:22-38):
 * compressed 48 / 96 bytes -> affine 96 / 192 bytes.  ok[i] = 0 (and a zero point) where the
 * reference raises ValueError('No sqrt exists' / 'No y for point x'). */
int b200bls_g1_decompress_batch(const uint8_t* in, uint8_t* out, uint8_t* ok, size_t n);
int b200bls_g2_decompress_batch(const uint8_t* in, uint8_t* out, uint8_t* ok, size_t n);
/* AffinePoint.serialize (ec.py:94-111): affine -> compressed (x, top bit = lex_gt_neg). */
int b200bls_g1_compress_batch(const uint8_t* in, uint8_t* out, size_t n);
int b200bls_g2_compress_batch(const uint8_t* in, uint8_t* out, size_t n);
/* Prime-order subgroup membership, which the reference never checks: ok[i] = 1 iff affine point i
 * (g2 = 0: 96 bytes, G1; g2 = 1: 192 bytes, G2) lies on the curve and in G1 / G2.  Coordinates are
 * read mod q, as by every entry point taking affine points; infinity is the identity and counts as a
 * member, and it is every point whose coordinates reduce to (0, 0): zero bytes, but also q || 0, 0 || q
 * and q || q per coordinate.  Endomorphism tests (Scott 2021): psi(P) == [x]P on G2,
 * (beta x, y) == [-x^2]P on G1, about 1.1 k / 1.3 k Montgomery products per point. */
int b200bls_subgroup_check_batch(int g2, const uint8_t* pts, uint8_t* ok, size_t n);
int b200bls_subgroup_check_batch_dev(int g2, const void* pts, void* ok, size_t n);
/* The public-key rule of the strict verifications below (KeyValidate of the IETF BLS draft): ok[i] = 1
 * iff affine G1 point i (96 bytes) is in G1 and is not infinity, both decided on the coordinates
 * reduced mod q, as the pairing reads them. */
int b200bls_key_validate_batch(const uint8_t* pts, uint8_t* ok, size_t n);
int b200bls_key_validate_batch_dev(const void* pts, void* ok, size_t n);

/* The reference's Jacobian-coordinate functions on JACOBIAN inputs, the granularity of its plugin seam
 * (fields_t.py:1218-1265): a = n x (X, Y, Z), three coordinates of 48 (G1) / 96 (G2) bytes, infinity = Z = 0.
 * op 0: fq_/fq2_to_affine (fields_t.py:609-622); 1: fq_/fq2_double_point_jacobian (878-903); 2: fq_/fq2_
 * add_points_jacobian with b = n Jacobian points (762-819; equal points double -- for G1 too, the reference's
 * TypeError at 781 is a defect); 3: fq_/fq2_scalar_mult_jacobian with b = n x 32-byte big-endian scalars (705-740).
 * out = n affine points (96 / 192 bytes, zero = infinity): the normalised representative (x, y, 1) of the triple
 * the reference returns; the normalisation (two field inversions in the reference) runs on the device. */
int b200bls_jacobian_op_batch(int g2, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n);
/* fq2_untwist (fields_t.py:936-943; ec.py:402-418 untwist): points of the twist E'(Fq2), 192 bytes, ->
 * (x / w^2, y / w^3) on E(Fq12): x' || y', 2 x 576 bytes. */
int b200bls_g2_untwist_batch(const uint8_t* pts, uint8_t* out, size_t n);
/* fq12_twist (fields_t.py:1018-1031; ec.py:421-437 twist): (x, y) with Fq12 coordinates, 2 x 576 bytes, ->
 * (x w^2, y w^3), 2 x 576 bytes. */
int b200bls_fq12_twist_batch(const uint8_t* pts, uint8_t* out, size_t n);
/* psi (ec.py:440-444: twist(Frobenius(untwist(P)))) on affine points of the twist, 192 -> 192 bytes. */
int b200bls_g2_psi_batch(const uint8_t* pts, uint8_t* out, size_t n);

/* ---- hashing and verification ------------------------------------------------------------------ */
/* sw_encode for Fq2 (ec.py:449-507), the Shallue-van de Woestijne map both halves of hash_to_point_Fq2 go
 * through: t (Fq2, 96 bytes) -> affine point of the twist (192 bytes; t = 0 -> infinity = zero bytes). */
int b200bls_sw_encode_g2_batch(const uint8_t* t, uint8_t* out, size_t n);
/* hash_to_point_prehashed_Fq2 (ec.py:528-550): n x 32-byte message hashes -> n x 192 bytes. */
int b200bls_hash_to_g2_batch(const uint8_t* hashes, uint8_t* out, size_t n);
int b200bls_hash_to_g2_batch_dev(const void* hashes, void* out, size_t n);
/* PrivateKey.sign_prehashed (keys.py:128-132) for n (secret key, message hash) pairs: sig_i = sk_i * H(mh_i).
 * sk32: n x 32-byte big-endian secret keys (any value below 2^256; the signature is that of sk mod n), mh32: n x 32
 * bytes.  wire = 0: sig = n x 192 affine bytes; wire = 1: sig = n x 96 Signature.serialize() bytes.  The bytes are
 * those of the reference.  One device pass per batch: the SHA stage, a split of sk mod n into four base-|x| digits,
 * and one program that hashes to G2 and runs a 64-step ladder over the digits and the endomorphism psi (0.63x the
 * Montgomery products of b200bls_hash_to_g2_batch followed by b200bls_g2_scalar_mul_batch).  n = 0 does nothing.
 * Secret keys: the library's device copies -- the staged copy of sk32 in the host-buffer form and the digit buffer
 * in both forms -- are zeroed on the stream after their last reader, before the call returns.  The caller of the
 * _dev form owns its sk32 buffer and clears it.  Not constant-time: the inversion and the regions that warps skip
 * depend on the data, as in the scalar multiplications above. */
int b200bls_sign_batch(int wire, const uint8_t* sk32, const uint8_t* mh32, uint8_t* sig, size_t n);
int b200bls_sign_batch_dev(int wire, const void* sk32, const void* mh32, void* sig, size_t n);
/* PrivateKey.get_public_key (keys.py:119-121): pk_i = sk_i * G1, from the same digits with a table of multiples of
 * G1 fixed at build time (0.38x the products of b200bls_g1_scalar_mul_batch).  wire = 0: pk = n x 96 affine bytes;
 * wire = 1: n x 48 PublicKey.serialize() bytes.  Secret-key handling and timing as for b200bls_sign_batch. */
int b200bls_public_key_batch(int wire, const uint8_t* sk32, uint8_t* pk, size_t n);
int b200bls_public_key_batch_dev(int wire, const void* sk32, void* pk, size_t n);
/* hash_pks (util.py:36-50), the per-key part: out[i] = SHA256(uint32_be(first_index + i) ||
 * pk_hash) mod n as 32 big-endian bytes (the scalar format of the scalar-multiplication entry
 * points), pk_hash = SHA256(pk_1 || ... || pk_N) computed by the caller.  These are the
 * exponents T_i of secure aggregation (bls.py:29-56, 132-144, 217-221). */
int b200bls_hash_pks(const uint8_t* pk_hash32, uint32_t first_index, uint8_t* out, size_t n);
int b200bls_hash_pks_dev(const void* pk_hash32, uint32_t first_index, void* out, size_t n);
/* n independent single-message verifications, the data-parallel core of BLS.verify
 * (bls.py:154-201): ok[i] = (e(-G1, sig_i) * e(pk_i, H(mh_i)) == 1).
 * pk: n x 96, mh: n x 32, sig: n x 192 (affine), ok: n bytes. */
int b200bls_verify_batch(const uint8_t* pk, const uint8_t* mh, const uint8_t* sig, uint8_t* ok, size_t n);
int b200bls_verify_batch_dev(const void* pk, const void* mh, const void* sig, void* ok, size_t n);
/* The same from the wire formats: pk48 = n x 48-byte PublicKey.serialize() bytes, sig96 = n x 96-byte
 * Signature.serialize() bytes, decoded on the device (keys.py:29-40, signature.py:22-38).  A key or
 * signature that does not decode -- the reference raises ValueError -- gives ok[i] = 0. */
int b200bls_verify_batch_wire(const uint8_t* pk48, const uint8_t* mh, const uint8_t* sig96, uint8_t* ok, size_t n);
int b200bls_verify_batch_wire_dev(const void* pk48, const void* mh, const void* sig96, void* ok, size_t n);
/* Strict forms of b200bls_verify_batch / b200bls_verify_batch_wire: the same verdict AND-ed with
 * "pk_i is in G1 and is not infinity" and "sig_i is in G2" (b200bls_subgroup_check_batch).  The
 * reference accepts points outside the subgroups: the order-3 key (0, 2) verifies the infinity
 * signature for every message, pk + (0, 2) verifies pk's signatures, and the infinity key verifies
 * the infinity signature.  Rejecting the infinity key is the KeyValidate rule of the IETF BLS draft;
 * it is decided on the reduced coordinates, so a key encoded as q || 0 is infinity and rejected too. */
int b200bls_verify_batch_strict(const uint8_t* pk, const uint8_t* mh, const uint8_t* sig, uint8_t* ok, size_t n);
int b200bls_verify_batch_strict_dev(const void* pk, const void* mh, const void* sig, void* ok, size_t n);
int b200bls_verify_batch_wire_strict(const uint8_t* pk48, const uint8_t* mh, const uint8_t* sig96, uint8_t* ok,
                                     size_t n);
int b200bls_verify_batch_wire_strict_dev(const void* pk48, const void* mh, const void* sig96, void* ok, size_t n);
/* One aggregate signature over n distinct message hashes (bls.py:194-201):
 * *ok = (e(-G1, sig) * prod_i e(pk_i, H(mh_i)) == 1).  n + 1 Miller loops, one final
 * exponentiation.  pks are the per-message public-key sums the host-side grouping produced. */
int b200bls_aggregate_verify(const uint8_t* sig, const uint8_t* pks, const uint8_t* mhs, size_t n, uint8_t* ok);
/* The same, enqueued on the selected library stream without waiting: several aggregate
 * verifications overlap (b200bls_set_stream).  *ok is valid after b200bls_sync(); inputs must
 * stay untouched until then. */
int b200bls_aggregate_verify_async(const uint8_t* sig, const uint8_t* pks, const uint8_t* mhs, size_t n, uint8_t* ok);
/* One rank's partial of a sharded aggregate verification: [e(-G1, sig) *] prod_i miller(pk_i,
 * H(mh_i)) as 576 bytes, NOT final-exponentiated (sig = NULL where the rank does not own the
 * signature pair).  Ranks exchange these, multiply them (b200bls_field_op_batch, level 12) and run
 * b200bls_final_exp_batch once. */
int b200bls_aggregate_miller(const uint8_t* sig, const uint8_t* pks, const uint8_t* mhs, size_t n, uint8_t* out576);

/* ---- multi-GPU: one process per GPU, contiguous batch slices (SURVEY.md 8e) -----------------------------------
 * Independent units (pairing_batch, verify_batch) need no exchange.  The reductions exchange ONE tiny partial per
 * rank -- a 576-byte Miller product (stage one of fq_ate_pairing_multi, fields_t.py:1114-1121) or one affine point
 * -- with a single all-gather, and every rank finishes locally.  b200bls_comm_init joins the ranks of one node:
 * `key` names the rendezvous (e.g. the launcher's MASTER_PORT), nccl_lib_path the NCCL library to dlopen (NULL:
 * the system's libnccl.so.2; NCCL missing or failing leaves the shared-memory host gather, b200bls_comm_has_nccl
 * tells).  use_nccl selects the transport per call: ncclAllGather over NVLink on the library stream, or a host
 * gather through a POSIX shared-memory segment (north_star: measure both, keep the faster). */
int b200bls_comm_init(int rank, int world, const char* key, const char* nccl_lib_path);
void b200bls_comm_shutdown(void);
int b200bls_comm_has_nccl(void);
int b200bls_comm_world(void);
int b200bls_comm_rank(void);
/* The host gather on its own: `bytes` (<= 4096) per rank -> recv[world][bytes], in rank order, on every rank. */
int b200bls_allgather_host(const uint8_t* send, uint8_t* recv, size_t bytes);
/* bls.py:194-201 with the (pk_i, message hash_i) list sharded over the ranks: pks / mhs are this rank's slice
 * (n may be 0), sig is read on rank 0.  The same *ok on every rank. */
int b200bls_aggregate_verify_sharded(const uint8_t* sig, const uint8_t* pks, const uint8_t* mhs, size_t n, int use_nccl,
                                     uint8_t* ok);
/* bls.py:13-26 / 204-223 (plain sums) over device-resident slices: pts_dev = this rank's n affine points
 * (96 / 192 bytes each); out = the sum over all ranks' slices as 96 / 192 host bytes, on every rank. */
int b200bls_point_sum_sharded_dev(int g2, const void* pts_dev, size_t n, int use_nccl, uint8_t* out);

#ifdef __cplusplus
}
#endif
#endif /* B200BLS_H */
