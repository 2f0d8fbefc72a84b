/* fourq_b200.h -- C ABI of the B200-native batched Curve4Q engine (libfourq_b200.so).
 *
 * This is the drop-in boundary for the hot path of bifurcation/fourq.  The reference has no FFI: its boundary is the
 * set of Python functions in impl/curve4q.py, impl/fields.py and impl/curve25519.py.  Every entry point below names the
 * reference function it replaces; fourq_b200/ (Python, ctypes) mirrors those names in batched form.
 *
 * Conventions
 *   - all buffers are caller-owned, C-contiguous, little-endian byte rows:
 *       GF(p^2) element   32 B = LE128(re) | LE128(im)          (fields.py:125-132 packing, two halves)
 *       affine point      64 B = x | y                          (two GF(p^2) elements)
 *       encoded point     32 B                                   (curve4q.py:41-46)
 *       scalar            32 B  little-endian unsigned, no clamping (curve4q.py:558-559 limb order)
 *   - host entry points take HOST pointers (pageable or pinned) and run on `ndev` GPUs, rows split in contiguous
 *     slices (device i starts on rows [i*ceil(n/ndev), ...) and, once done, helps with the back of the slice that has the
 *     most rows left); there is no collective and no CPU fallback: with no CUDA device every call returns FQ_ERR_NO_DEVICE.
 *   - return value: 0 (FQ_OK) or a negative FQ_ERR_*; fq_last_error() gives the text (thread-local).
 *   - per-row outcome in status[n] (uint8): see FQ_ST_*.  Rows that fail are zero-filled in the output.
 *   - thread-safe: every GPU has its own lock and its own pair of host threads (one feeds chunks to the GPU, one retires
 *     them), so the slices of a call run concurrently and callers on disjoint GPUs do not wait for each other; calls that
 *     share a GPU are served in submission order.  Per-device contexts are created lazily.
 */
#ifndef FOURQ_B200_H
#define FOURQ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FQ_VERSION 200

#if defined(__GNUC__)
#define FQ_API __attribute__((visibility("default")))
#else
#define FQ_API
#endif

#define FQ_OK 0
#define FQ_ERR_NO_DEVICE (-1)   /* no CUDA device / driver: the engine has no CPU path */
#define FQ_ERR_CUDA (-2)        /* a CUDA call failed; see fq_last_error() */
#define FQ_ERR_ARG (-3)         /* null pointer, ndev out of range, ... */

/* per-row status codes */
#define FQ_ST_OK 0
#define FQ_ST_RESERVED_BIT 1    /* curve4q.py:52-53  "Malformed point: reserved bit is not zero" (bit 127 of y0) */
#define FQ_ST_NONCANONICAL 2    /* curve4q.py:61-62  y0 >= p or y1 >= p (same message in the reference) */
#define FQ_ST_QUIRK_T0 3        /* curve4q.py:76-77  the reference raises AttributeError (GFp.two) when t == 0 */
#define FQ_ST_NOT_ON_CURVE 4    /* curve4q.py:93-94, 447-448  "Point not on curve" */
#define FQ_ST_NEUTRAL 5         /* curve4q.py:459-460  "DH computation resulted in neutral point" */

FQ_API int fq_version(void);
FQ_API int fq_device_count(void);                 /* >= 0, or FQ_ERR_NO_DEVICE */
FQ_API const char* fq_last_error(void);
/* GPUs used by the host entry points are first .. first+ndev-1 (default 0).  One process per GPU sets its LOCAL_RANK. */
FQ_API int fq_set_device_base(int first);
/* device milliseconds of the last host call of this thread: CUDA-event time from the first kernel to the end of the last kernel of
 * a GPU's slice (its chunks overlap: copies of one run under the kernels of another), maximum over the GPUs used */
FQ_API float fq_last_kernel_ms(void);
/* rows[i] = rows GPU first+i processed in the last host call of this thread.  Every GPU starts on its own contiguous slice of
 * ceil(n/ndev) rows; one that runs out takes chunks from the back of the slice with the most rows left, so on a host whose GPUs
 * do not all reach memory equally fast the numbers differ from n/ndev. */
FQ_API int fq_last_rows_per_device(size_t* rows, int ndev);

/* Constant-time table selection of every scalar multiplication (csrc/dh.cuh).  In both modes every thread issues the loads
 * of ALL table entries from digit-independent addresses and there is no secret-dependent branch.
 *   1 (default)  strict scan: every lane loads every entry and keeps one with a predicated select per word, so not even the
 *                memory activity of a load depends on a digit: kernel time is flat across scalar distributions
 *                (profiles/r01_ct_timing.jsonl, r02_ct_timing.jsonl).  This is what draft-ladd-cfrg-4q.md:653-656, :753-755 ask for.
 *   0 (opt-in)   masked loads: the digit sets each load's predicate and a lane whose predicate is off transfers nothing; no
 *                select instructions at all, 1-2 % faster for variable-base DH and 8 % for the comb keygen.  The number of
 *                shared-memory wavefronts of a load then depends on how the digits are distributed over the 32 lanes of a warp:
 *                0.4 % of the ladder time between the extremes "all rows of every warp use the same scalar" and "all differ".
 *                Only for non-secret scalars (verification-style workloads, benchmarks).
 * Same outputs.  The environment variable FQ_STRICT_SELECT=0 selects 0 at start-up. */
FQ_API int fq_set_select_mode(int strict);
FQ_API int fq_get_select_mode(void);

/* ---- GF(p^2) field ops: fields.py GFp2.mul :167, sqr :176, inv :194, add :157, sub :162, neg :184, conj :189.
 * Inputs may be any 128-bit values per half (the reference reduces ints mod p); outputs are canonical. */
FQ_API int fq_fp2_mul(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int ndev);
FQ_API int fq_fp2_sqr(const uint8_t* a, uint8_t* out, size_t n, int ndev);
FQ_API int fq_fp2_inv(const uint8_t* a, uint8_t* out, size_t n, int ndev);
FQ_API int fq_fp2_add(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int ndev);
FQ_API int fq_fp2_sub(const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int ndev);
FQ_API int fq_fp2_neg(const uint8_t* a, uint8_t* out, size_t n, int ndev);
FQ_API int fq_fp2_conj(const uint8_t* a, uint8_t* out, size_t n, int ndev);
/* fields.py GFp2.invsqrt :201-230 (the reference marks it "not constant-time"; curve4q.py never calls it, fields.py:391 tests it).
 * Bit-compatible with the reference's control flow, including its two comparisons with -1 that can never be true: a row with
 * a[1] == 0 (raw value) takes the GF(p) branch :204-209, every other row the norm branch :214-230, whatever the
 * quadratic character of the input.  a, out are (n,32). */
FQ_API int fq_fp2_invsqrt(const uint8_t* a, uint8_t* out, size_t n, int ndev);
/* fields.py GFp.select :59-64 and GFp2.select :236-238:  out = y ^ ((mask * c) & (x ^ y)), i.e. c == 1 -> x, c == 0 -> y, bit for
 * bit (no reduction: x and y pass through as they are).  c is (n,) uint8, one condition per row; x, y, out are (n,16) for GF(p)
 * and (n,32) for GF(p^2) (the same c for both halves).  Other values of c behave as in the reference's expression:
 * the mask is (2^512 - 1) * c, i.e. -c modulo 2^128. */
FQ_API int fq_fp_select(const uint8_t* c, const uint8_t* x, const uint8_t* y, uint8_t* out, size_t n, int ndev);
FQ_API int fq_fp2_select(const uint8_t* c, const uint8_t* x, const uint8_t* y, uint8_t* out, size_t n, int ndev);

/* ---- GF(p) field ops on 16-byte rows (little-endian 128-bit values): fields.py GFp.mul :42, sqr :48, inv :67-106,
 * add :30, sub :36, neg :54, invsqrt :110-122.  a, b, out are (n,16); b is ignored by the unary ops (may be NULL).  Inputs may
 * be any 128-bit value (the reference reduces ints mod p); outputs are canonical. */
#define FQ_FP_MUL 0
#define FQ_FP_SQR 1
#define FQ_FP_INV 2
#define FQ_FP_ADD 3
#define FQ_FP_SUB 4
#define FQ_FP_NEG 5
#define FQ_FP_INVSQRT 6
FQ_API int fq_fp_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int ndev);

/* ---- GF(2^255-19) field ops on 32-byte rows (little-endian 256-bit values): fields.py GFp25519.add :267, sub :273, mul :279,
 * sqr :285, inv :293-362 -- the GFp25519 column of compare.py:14-49 (compare_fields).  op is FQ_FP_MUL, _SQR, _INV, _ADD or
 * _SUB; a, b, out are (n,32); b is ignored by the unary ops (may be NULL).  Inputs may be any 256-bit value (the reference
 * reduces ints mod p); outputs are canonical; inv(0) = 0 as the reference's chain gives. */
FQ_API int fq_fp25519_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t n, int ndev);

/* ---- point codec: curve4q.py decode :49-96 (enc (n,32) -> xy (n,64) + status), encode :41-46 (xy -> enc).
 * Unlike the reference, decode does not modify its input. */
FQ_API int fq_decode(const uint8_t* enc, uint8_t* xy, uint8_t* status, size_t n, int ndev);
FQ_API int fq_encode(const uint8_t* xy, uint8_t* enc, size_t n, int ndev);
/* curve4q.py PointOnCurve :23-29 on affine rows x | y (n,64): ok[i] = 1 if -x^2 + y^2 == 1 + d x^2 y^2, else 0 */
FQ_API int fq_point_on_curve(const uint8_t* xy, uint8_t* ok, size_t n, int ndev);
/* Opt-in, NOT bit-compatible with the reference on four inputs: decode as the draft specifies it (draft-ladd-cfrg-4q.md:841-888).
 * The reference raises AttributeError when t == 0 (curve4q.py:76-77, status 3 above); the draft continues with
 * t = 2 (t0 - t3), which decodes the encodings of the low-order points (0, 1), (0, -1), (i, 0), (-i, 0).  Every other input
 * gives exactly what fq_decode gives; status 3 never occurs. */
FQ_API int fq_decode_spec(const uint8_t* enc, uint8_t* xy, uint8_t* status, size_t n, int ndev);

/* ---- Diffie-Hellman
 * fq_dh:        encode(DH_windowed(k, decode(enc_pt)))            curve4q.py:49, 446-465, 41
 * fq_dh_affine: DH_windowed(k, (x, y)) on affine 64-byte points   curve4q.py:446-465
 * fq_dh_base:   encode(DH_windowed(k, G, table=T392)) = [392 k]G  curve4q.py:743-762
 * fq_mul_base:  encode(R1toAffine(MUL_windowed(k, G, table=table_windowed(G)))) = [k]G   curve4q.py:582-584 (no status:
 *               MUL_windowed has no failure path; k = 0 mod N gives the encoding of the neutral point) */
FQ_API int fq_dh(const uint8_t* k, const uint8_t* enc_pt, uint8_t* enc_out, uint8_t* status, size_t n, int ndev);
FQ_API int fq_dh_affine(const uint8_t* k, const uint8_t* xy, uint8_t* xy_out, uint8_t* status, size_t n, int ndev);
FQ_API int fq_dh_base(const uint8_t* k, uint8_t* enc_out, uint8_t* status, size_t n, int ndev);
FQ_API int fq_mul_base(const uint8_t* k, uint8_t* enc_out, size_t n, int ndev);
/* The same four with the reference's endomorphism algorithm: DH_endo / MUL_endo (curve4q.py:405-442, 467-468; phi, psi
 * :258-322; decompose, recode :339-380; table_endo :385-403).  Bit-identical outputs (curve4q.py:706-762), about 1.8x
 * fewer field multiplications. */
FQ_API int fq_dh_endo(const uint8_t* k, const uint8_t* enc_pt, uint8_t* enc_out, uint8_t* status, size_t n, int ndev);
FQ_API int fq_dh_endo_affine(const uint8_t* k, const uint8_t* xy, uint8_t* xy_out, uint8_t* status, size_t n, int ndev);
FQ_API int fq_dh_endo_base(const uint8_t* k, uint8_t* enc_out, uint8_t* status, size_t n, int ndev);
FQ_API int fq_mul_endo_base(const uint8_t* k, uint8_t* enc_out, size_t n, int ndev);

/* Fixed base with one precomputed table per digit ("comb"): the same results as fq_mul_base / fq_dh_base (the affine
 * point is canonical, curve4q.py:582-598 and :743-762 assert table == no table), computed as 62 mixed additions and no
 * doubling.  This is the fixed-base algorithm the draft recommends for key generation (draft-ladd-cfrg-4q.md:702-705,
 * :727-729: "FourQlib's fixed-base algorithm"); tables of G and [392]G are built on the device at context creation. */
FQ_API int fq_mul_base_comb(const uint8_t* k, uint8_t* enc_out, size_t n, int ndev);
FQ_API int fq_dh_base_comb(const uint8_t* k, uint8_t* enc_out, uint8_t* status, size_t n, int ndev);

/* ---- Fixed base for a point the caller registers: one public point, many scalars, on per-digit tables as above.
 * fq_base_create:  validates P once, exactly as the DH entry points do, on the GPU (one row):
 *                  affine = 0: pt is a 32-byte encoding, *status = that of fq_decode (1-4, including 3 at the reference's
 *                  t == 0 quirk, curve4q.py:49-96); affine = 1: pt is 64-byte x | y, each half reduced mod p, *status = 4
 *                  if P is not on the curve (curve4q.py:447-448).
 *                  Valid P: *status = 0 and *out = a new handle.  Invalid P: returns FQ_OK with *status != 0 and *out = NULL.
 *                  A pure-torsion P is valid: fq_dh_fixed then gives status 5 on every row, as fq_dh does.
 *                  Each GPU builds the tables of P and [392]P (2 x 48,384 B) on the first call that uses the handle there.
 * fq_dh_fixed:     per row, exactly fq_dh(k, enc(P)) for an encoded registration, and encode(DH_windowed(k, P)) for an affine
 *                  one (the bytes of fq_encode(fq_dh_affine(k, P))): DH_core (curve4q.py:446-462) computes Q = [392]P and
 *                  MUL_windowed(m, Q) = [r]Q with r = m mod N, plus N if that is even (curve4q.py:216-219).  Status 0 or 5.
 * fq_mul_fixed:    per row, encode(R1toAffine(MUL_windowed(k, P))) (curve4q.py:188-235) = encode([r]P) with the same r; no
 *                  status, k = 0 mod N gives the encoding of the neutral point.  For a P with a small-order component this is
 *                  NOT [k]P (r differs from k by a multiple of N, which does not kill the torsion part) and not what
 *                  MUL_endo would give; for P in the prime-order subgroup it is [k]P, and a handle of G gives fq_mul_base.
 * fq_base_destroy: frees the handle and its tables on every GPU (NULL is a no-op).  The handle must not be in use by a call
 *                  in flight on any thread.  fq_trim keeps the tables (multiples of a public point).
 * A handle may be used by several threads at once, on the same or on different GPUs. */
typedef struct fq_base fq_base;
FQ_API int fq_base_create(const uint8_t* pt, int affine, uint8_t* status, fq_base** out);
FQ_API int fq_base_destroy(fq_base* base);
FQ_API int fq_dh_fixed(const fq_base* base, const uint8_t* k, uint8_t* enc_out, uint8_t* status, size_t n, int ndev);
FQ_API int fq_mul_fixed(const fq_base* base, const uint8_t* k, uint8_t* enc_out, size_t n, int ndev);

/* ---- X25519 (RFC 7748): impl/curve25519.py:88-91 x25519(k, u) -> 32 bytes; k, u, out are (n,32) */
FQ_API int fq_x25519(const uint8_t* k, const uint8_t* u, uint8_t* out, size_t n, int ndev);

/* Frees the staging and scratch buffers the engine keeps per GPU between calls (up to ~0.5 GB per stream slot for the DH
 * ops) and trims the scratch pool of the stream entry points (up to ~4.9 GB per GPU, fq_stream_run) to zero; contexts,
 * streams and the fixed-base tables stay.  The next call allocates what it needs again. */
FQ_API int fq_trim(void);

/* ---- pinned host memory for zero-staging transfers (optional; any host pointer is accepted above) */
FQ_API int fq_host_alloc(void** p, size_t bytes);
FQ_API int fq_host_free(void* p);
/* Page-locked array of `rows` rows of `row_bytes` bytes for a batch that will run on `ndev` GPUs: the bytes of slice i (rows
 * [i*ceil(rows/ndev), ...), the way the host entry points cut a batch) are placed on the NUMA node of GPU i before the pages
 * are locked, so that every GPU copies from and to its own socket's memory.  Falls back to an ordinary page-locked allocation
 * where the platform gives no NUMA information or does not permit the placement.  Free with fq_host_free. */
FQ_API int fq_host_alloc_sliced(void** p, size_t rows, size_t row_bytes, int ndev);
FQ_API int fq_device_numa_node(int dev);          /* the NUMA node of a GPU, -1 if the platform does not say */

/* ---- device-resident variants, for measurement with inputs already in HBM (bench.py `value`, ncu).
 * op: one of FQ_DEVOP_*; pointers are device pointers on GPU `dev`; the kernel is launched `iters` times back to back on
 * the context's stream and *ms receives the average CUDA-event time of one launch. */
#define FQ_DEVOP_FP2_MUL 0
#define FQ_DEVOP_FP2_SQR 1
#define FQ_DEVOP_FP2_INV 2
#define FQ_DEVOP_FP2_ADD 3
#define FQ_DEVOP_FP2_SUB 4
#define FQ_DEVOP_FP2_NEG 5
#define FQ_DEVOP_FP2_CONJ 6
#define FQ_DEVOP_FP2_INVSQRT 7
#define FQ_DEVOP_FP2_SELECT 8  /* a = x, b = y, c = cond (1 byte per row), out: fq_dev_run3 */
#define FQ_DEVOP_FP_SELECT 9   /* the same on 16-byte rows */
#define FQ_DEVOP_FP_BASE 32    /* FQ_DEVOP_FP_BASE + FQ_FP_*: GF(p) ops on 16-byte rows, a (, b), out */
#define FQ_DEVOP_F25519_BASE 48 /* FQ_DEVOP_F25519_BASE + FQ_FP_MUL/_SQR/_INV/_ADD/_SUB: GF(2^255-19) ops on 32-byte rows */
#define FQ_DEVOP_DECODE 16     /* a = enc, out = xy, status */
#define FQ_DEVOP_ENCODE 17     /* a = xy, out = enc */
#define FQ_DEVOP_ON_CURVE 30      /* a = xy, out = ok (1 byte per row) */
#define FQ_DEVOP_DECODE_SPEC 29   /* as FQ_DEVOP_DECODE with the draft's t == 0 branch (fq_decode_spec) */
#define FQ_DEVOP_DH 18         /* a = k, b = enc_pt, out, status */
#define FQ_DEVOP_DH_AFFINE 19  /* a = k, b = xy, out = xy, status */
#define FQ_DEVOP_DH_BASE 20    /* a = k, out, status */
#define FQ_DEVOP_MUL_BASE 21   /* a = k, out */
#define FQ_DEVOP_X25519 22     /* a = k, b = u, out */
#define FQ_DEVOP_DH_ENDO 23
#define FQ_DEVOP_DH_ENDO_AFFINE 24
#define FQ_DEVOP_DH_ENDO_BASE 25
#define FQ_DEVOP_MUL_ENDO_BASE 26
#define FQ_DEVOP_DH_BASE_COMB 27    /* a = k, out, status */
#define FQ_DEVOP_MUL_BASE_COMB 28   /* a = k, out */
FQ_API int fq_dev_alloc(int dev, void** p, size_t bytes);
FQ_API int fq_dev_free(int dev, void* p);
FQ_API int fq_dev_upload(int dev, void* dst, const void* src, size_t bytes);
FQ_API int fq_dev_download(int dev, void* dst, const void* src, size_t bytes);
FQ_API int fq_dev_run(int op, int dev, const void* a, const void* b, void* out, void* status, size_t n, int iters, float* ms);
/* the same with a third input operand (FQ_DEVOP_FP_SELECT / FQ_DEVOP_FP2_SELECT: c = the condition bytes) */
FQ_API int fq_dev_run3(int op, int dev, const void* a, const void* b, const void* c, void* out, void* status, size_t n, int iters, float* ms);
/* CUDA-event milliseconds of the three kernels (prepare, ladder, finish) of the last launch of the last fq_dev_run of
 * this thread with a variable-base DH op (FQ_DEVOP_DH, _DH_AFFINE, _DH_ENDO, _DH_ENDO_AFFINE); zeros otherwise. */
FQ_API int fq_dev_last_phase_ms(float* ms3);
/* fq_dh_fixed (dh = 1) or fq_mul_fixed (dh = 0) on device buffers of GPU `dev`, `iters` launches as fq_dev_run (the first
 * call on a GPU builds the base's tables there before timing); status may be NULL for dh = 0 */
FQ_API int fq_base_dev_run(const fq_base* base, int dh, int dev, const void* k, void* out, void* status, size_t n, int iters, float* ms);
/* ---- stream-ordered entry points, for batches that already sit in GPU memory (a PyTorch job, inputs built by the caller's
 * own kernels).  The operation is enqueued on `stream` (a cudaStream_t; NULL = the legacy default stream) and the call
 * returns without waiting: the results are there once the stream reaches that point.
 *   - op is an FQ_DEVOP_* code with the operands of fq_dev_run3 above.  Outputs, statuses and the zero fill of failed rows
 *     are byte for byte those of the host entry point; rows past n are not written.  Table selection follows
 *     fq_set_select_mode.
 *   - Every operand must be device memory of one GPU (both ends of each range are checked), and a non-NULL stream must
 *     belong to that GPU (checked on calls outside capture: CUDA does not name the device of a capturing stream).  The call makes that GPU current and restores the calling thread's device before it returns;
 *     fq_set_device_base and ndev play no part.
 *   - Refused with FQ_ERR_ARG before anything is enqueued, outputs untouched: an unknown op; a NULL operand the op needs;
 *     an operand that is not device memory of that GPU; a stream of another GPU; a row operand that is not aligned as
 *     its kernel accesses it (32 bytes for rows of 32 and 64 bytes, 16 for GF(p) rows: an offset view of a tensor is the
 *     usual way to get this wrong); an output that overlaps an input other than as an exact alias of the same row width,
 *     or overlaps the other output (FQ_DEVOP_FP2_INV and the GF(2^255-19) inversion refuse even the exact alias: they park
 *     prefix products in out); for fq_base_stream_run a NULL base.  n == 0 returns FQ_OK and enqueues nothing.
 *   - Scratch (the DH ops, the fixed-base ops, X25519) comes from a memory pool the library keeps per GPU, allocated,
 *     zeroed and released on the caller's stream around the kernels: no workspace argument, and concurrent streams never
 *     share scratch.  The pool keeps up to ~4.9 GB per GPU mapped between calls (the scratch of one 2^22-row DH launch
 *     group) until fq_trim.
 *   - The first stream call on a GPU initialises the GPU (constant and comb tables, the pool), and the first with a base
 *     builds that base's tables there; both wait for the library's own stream once.  A first call on a stream that is
 *     being captured is therefore refused with FQ_ERR_ARG: make one call on that GPU outside capture first.  After that a
 *     call makes no synchronising call, no cudaMalloc / cudaFree and no event record, and takes no lock a host call
 *     holds, so it does not wait behind host calls on the same GPU and can be captured into a CUDA graph (the scratch
 *     becomes graph allocation nodes).
 *   - Statuses stay on the device: checking them on the host is the caller's synchronisation.
 *   - fq_base_destroy must not run while stream work that uses the base is pending, and a graph that captured such a call
 *     must not be replayed after the base is destroyed. */
FQ_API int fq_stream_run(int op, const void* a, const void* b, const void* c, void* out, void* status, size_t n, void* stream);
/* fq_dh_fixed (dh = 1) / fq_mul_fixed (dh = 0, status unused) of a registered base, the same way */
FQ_API int fq_base_stream_run(const fq_base* base, int dh, const void* k, void* out, void* status, size_t n, void* stream);

/* writes `bytes` of zeros over a scratch buffer larger than L2 (used between timed iterations) */
FQ_API int fq_dev_flush_l2(int dev);

/* ---- integer-multiply peak of GPU `dev`, measured live: 32x32->64 multiply-adds per second as IMAD.WIDE.U32
 * (the instruction the limb arithmetic is made of) and 32-bit IMAD per second.  The roofline denominator. */
FQ_API int fq_imad_peak(int dev, double* wide_per_s, double* imad32_per_s);

#ifdef __cplusplus
}
#endif
#endif
