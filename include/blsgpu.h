/* blsgpu.h -- C ABI of the B200-native BLS12-381 batch-verify / hash-to-G2 / aggregate / R1CS-check engine.
 *
 * Drop-in boundary for the hot path of lightec-xyz/bls-verify-gadget.  The reference is a Rust library with no FFI
 * of its own; each entry point below is what a Rust `extern "C"` block (INTEGRATION.md) binds to replace the
 * arkworks call named beside it.  All file:line citations are relative to the reference tree.
 *
 * Conventions
 *  - Plain pointers and sizes only.  Pointers are caller-owned; nothing is retained after return.
 *  - Pointer mode (blsgpu_set_pointer_mode): BLSGPU_HOST (default) = all data pointers are host memory, the call
 *    stages H2D/D2H itself and returns when results are in host memory; BLSGPU_DEVICE = all data pointers are
 *    device memory on the context's GPU (16-byte aligned), work is enqueued on the context's stream and the call
 *    returns without synchronising.
 *  - Return value: 0 = call ok, < 0 = call-level error (message via blsgpu_last_error).  Per-item outcomes go to
 *    status[] and never abort the batch.
 *  - Byte formats are exactly the reference's serialisations: public key = 48-byte and signature = 96-byte ZCash
 *    compressed big-endian with flag bits (src/bls.rs:219-260, 316-357), secret key = 32-byte little-endian
 *    canonical Fr (src/bls.rs:79-121), GT = 12 x 48-byte little-endian canonical in tower order
 *    c0.c0.c0 ... c1.c2.c1 (ark-serialize of Fp12).
 *  - Host mode copies with cudaMemcpyAsync straight from / to the caller's buffers: pageable memory works (the runtime stages it, the
 *    copy then is synchronous and slower); PINNED buffers (cudaHostAlloc / cudaHostRegister) give the PCIe rate and are what
 *    bench.py's e2e figure uses.
 *  - Every call runs on the context's device and restores the caller's current CUDA device before it returns.
 *  - One context per GPU per process; a context may be used by one host thread at a time.
 *  - There is no CPU fallback: every function fails with BLSGPU_ERR_CUDA if no sm_100 device is usable.
 */
#ifndef BLSGPU_H
#define BLSGPU_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct blsgpu_ctx blsgpu_ctx;

/* per-item status codes; BLSError of src/bls.rs:359-377 maps to 2 / 3 / 5 */
#define BLSGPU_ST_TRUE        0  /* Ok(true)                                            (src/bls.rs:457) */
#define BLSGPU_ST_FALSE       1  /* Ok(false): pairing product != 1                     (src/bls.rs:457) */
#define BLSGPU_ST_BAD_PUBKEY  2  /* Err(InvalidPublicKey): identity / undecodable / off-curve / wrong subgroup (src/bls.rs:434-442) */
#define BLSGPU_ST_BAD_SIG     3  /* Err(InvalidSignature): undecodable / off-curve / wrong subgroup          (src/bls.rs:443-447) */
#define BLSGPU_ST_EMPTY       4  /* aggregate of nothing = None                         (src/bls.rs:184-185, 289-290) */
#define BLSGPU_ST_BAD_SECKEY  5  /* Err(InvalidSecretKey): zero or non-canonical sk     (src/bls.rs:417-419) */
/* deserialisation detail codes returned by blsgpu_deserialize_g1/g2 */
#define BLSGPU_DE_OK 0
#define BLSGPU_DE_INFINITY 1        /* valid encoding of the identity */
#define BLSGPU_DE_BAD_FLAGS 2
#define BLSGPU_DE_OUT_OF_RANGE 3
#define BLSGPU_DE_NOT_ON_CURVE 4
#define BLSGPU_DE_NOT_IN_SUBGROUP 5

#define BLSGPU_ERR_ARG   (-1)
#define BLSGPU_ERR_CUDA  (-2)
#define BLSGPU_ERR_ALLOC (-3)

#define BLSGPU_HOST 0
#define BLSGPU_DEVICE 1

/* ---- context ---------------------------------------------------------------------------------------------- */
int  blsgpu_create(blsgpu_ctx** out, int device /* ordinal, or -1 for the current device */);
void blsgpu_destroy(blsgpu_ctx* ctx);
const char* blsgpu_last_error(blsgpu_ctx* ctx);
/* work is enqueued on the context's own non-blocking stream until a caller stream is set; cuda_stream is a cudaStream_t
 * (NULL = the legacy default stream); use_own != 0 switches back to the context's own stream */
int  blsgpu_set_stream(blsgpu_ctx* ctx, void* cuda_stream, int use_own);
int  blsgpu_set_pointer_mode(blsgpu_ctx* ctx, int mode);
int  blsgpu_synchronize(blsgpu_ctx* ctx);
/* kernels launched by this context since creation (bench.py's gpu_launches) */
uint64_t blsgpu_launch_count(blsgpu_ctx* ctx);
/* measurement hook: record CUDA events at the stage boundaries of blsgpu_verify_batch on the context's stream;
 * blsgpu_stage_times synchronises and returns the device time in ms of the last call's (last chunk's) stages:
 * [0] decode+check G1, [1] decode+check G2, [2] hash-to-G2, [3] Miller loop, [4] final exponentiation, [5] epilogue */
int blsgpu_set_profiling(blsgpu_ctx* ctx, int on);
/* blsgpu_verify_batch works in internal passes of at most `items` triples (default 2^20, ~9 GB of workspace with the split stage kernels,
 * ~1.2 GB without); a multiple of 64 */
int blsgpu_set_chunk(blsgpu_ctx* ctx, size_t items);
/* inside a pass the items are split into `lanes` (1..4, default 2) sub-ranges enqueued on separate internal streams that fork from and
 * join the context's stream, so that the tail wave of a stage kernel overlaps the other sub-range's work; 1 = strictly serial kernels
 * (use it with blsgpu_set_profiling: stage events of concurrent lanes would overlap) */
int blsgpu_set_lanes(blsgpu_ctx* ctx, int lanes);
/* 1 (default): inside blsgpu_verify_batch and the aggregate entry points hash-to-G2, the Miller loop and the final exponentiation run as
 * sequences of short specialised launches with the per-item state kept in the workspace between them -- hash_to_field | SSWU + isogeny per
 * field element | cofactor clearing; 8 x (line coefficients of both pairs | accumulator update); easy part, then 5 x (63 compressed
 * squarings | decompression + products).  0: one launch per stage (k_hash_to_g2, k_miller, k_final_exp).  Same results.  The short launches
 * are faster at every batch size measured (+12 % at 2^20 items: smaller working sets and less code per kernel) and much faster for batches
 * of a few waves (a CTA of the one-launch kernels runs 14-21 ms; the partly filled last wave of each costs a tenth of a 2^17-item pass).
 * Workspace: 8.7 KB per item of a pass instead of 1.2 KB (blsgpu_set_chunk bounds the pass). */
int blsgpu_set_split(blsgpu_ctx* ctx, int on);
/* six lanes per item (warp-cooperative Fp12, coop.cuh) in the accumulator update of the Miller loop and the hard part of the final
 * exponentiation, instead of one thread per item: 0 = never, 1 = always, 2 (default) = for passes of at most 4,096 items.  A small pass is
 * latency-bound -- every item is one thread's serial chain -- and the six-lane kernels shorten the chain at the price of more work; in mode 2
 * such a pass also runs its two decoders and its hash side by side on internal streams.  A single verify takes 12.4 ms instead of 28.6 ms, 1,024
 * take 12.7 ms instead of 30 ms; from one wave of resident threads (~38,000 items) on the thread-per-item kernels are faster
 * (profiles/latency_r02.json, latency_default_r02.json).  All forms produce identical statuses and GT bytes. */
int blsgpu_set_coop(blsgpu_ctx* ctx, int on);
int blsgpu_stage_times(blsgpu_ctx* ctx, float ms6[6]);

/* ---- BLS::verify over a batch  (replaces <BLS<P> as SignatureScheme>::verify, src/bls.rs:427-458, incl. the
 *      TryFrom decoding of tests/tests.rs:244-254) -----------------------------------------------------------
 * msg_off: n+1 byte offsets into msg, or NULL for fixed 32-byte messages.
 * status[n]; ok_bitmap (nullable): ceil(n/64) words, bit i set <=> status[i] == 0;
 * gt_acc_le576 (nullable): product over all items whose pairing was evaluated (status 0 or 1) of the GT value. */
int blsgpu_verify_batch(blsgpu_ctx* ctx, const uint8_t* pk48, const uint8_t* msg, const uint32_t* msg_off,
                        const uint8_t* sig96, size_t n, uint8_t* status, uint64_t* ok_bitmap, uint8_t* gt_acc_le576);

/* ---- random-linear-combination batch check (an ADDITIONAL fast path; the reference has no batch API: SURVEY 8(f)-3) ------
 * One pairing-product equation for the whole batch instead of one per item:
 *     prod_i e(r_i pk_i, H(m_i)) * e(-g1, sum_i r_i sig_i) == 1,   r_i = 64 non-zero bits of SHA-256(seed16 || le64(i)).
 * *all_ok = 1 iff every public key and signature decodes and validates (the checks of src/bls.rs:434-447) and the equation
 * holds; a batch that contains a triple BLS::verify would reject passes with probability <= 2^-64 over the choice of the seed,
 * which must be unpredictable to whoever produced the batch.  status (nullable, n bytes) receives the per-item decode
 * outcome only (0, 2 or 3): to locate a bad item after *all_ok == 0, use blsgpu_verify_batch_rlc_bisect (below).  Roughly 1.6x the
 * throughput of blsgpu_verify_batch: one pair per Miller loop and a single final exponentiation per batch. */
int blsgpu_verify_batch_rlc(blsgpu_ctx* ctx, const uint8_t* pk48, const uint8_t* msg, const uint32_t* msg_off,
                            const uint8_t* sig96, size_t n, const uint8_t seed16[16], uint8_t* status, uint8_t* all_ok);

/* The batch check with the EXACT per-item outcome (SURVEY 8(f)-3): one such equation per piece of 4,096 items, all pieces finished side by
 * side; every piece whose equation fails is re-run through the per-item path inside the call.  status[n] and ok_bitmap (nullable) equal
 * blsgpu_verify_batch's, except with probability <= 2^-64 per failing piece over the seed; *fallback_items (nullable, host memory) = number of
 * items that went through the per-item path. */
int blsgpu_verify_batch_rlc_bisect(blsgpu_ctx* ctx, const uint8_t* pk48, const uint8_t* msg, const uint32_t* msg_off,
                                   const uint8_t* sig96, size_t n, const uint8_t seed16[16], uint8_t* status, uint64_t* ok_bitmap, uint64_t* fallback_items);

/* ---- PublicKey::aggregate + verify  (src/bls.rs:183-195 then 427-458; tests/tests.rs:297-334) ---------------
 * ncomm committees of k keys each; bitmap (nullable): bit c*k+j selects key j of committee c (the gadget's
 * mapped_aggregate semantics, src/constraints.rs:169-191); agg_pk48_out (nullable): the aggregated keys. */
int blsgpu_fast_aggregate_verify_batch(blsgpu_ctx* ctx, const uint8_t* pks48, const uint64_t* bitmap, size_t k,
                                       const uint8_t* msg32, const uint8_t* sig96, size_t ncomm,
                                       uint8_t* status, uint8_t* agg_pk48_out);

/* ---- Eth2 AggregateVerify: one signature over k (public key, message) pairs with DISTINCT messages -- the category the reference's
 *      tests/readme.md:4-7 names and does not vendor (SURVEY 8(f)-4).  nsig signatures; signature s covers the pairs
 *      [pair_off[s], pair_off[s+1]) of pks48 / msg (msg_off: npairs + 1 offsets, NULL = fixed 32-byte messages).  True iff every key
 *      decodes, is not the identity and lies in the subgroup (the checks of src/bls.rs:434-442), the signature lies in the subgroup
 *      (src/bls.rs:443-447) and e(-g1, sig) * prod_j e(pk_j, H(m_j)) == 1.  status[s]: 0 / 1, 2 = a key failed, 3 = the signature failed,
 *      4 = no pairs (the draft's precondition n >= 1: callers treat it as false). */
int blsgpu_aggregate_verify_batch(blsgpu_ctx* ctx, const uint8_t* pks48, const uint8_t* msg, const uint32_t* msg_off, const uint32_t* pair_off,
                                  const uint8_t* sig96, size_t nsig, uint8_t* status);

/* ---- the same with a RESIDENT validator pool (BASELINE configs[2], variant "keys pre-decoded in HBM"): the pool's keys are
 *      decoded and subgroup-checked once (PublicKey::try_from, src/bls.rs:219-223) and kept in HBM as affine Montgomery limb-SoA;
 *      committees are lists of pool indices.  status (nullable) of pool_create: BLSGPU_DE_* per key; an index that is out of range or
 *      names an undecodable key makes its committee BLSGPU_ST_BAD_PUBKEY. */
int blsgpu_pool_create(blsgpu_ctx* ctx, const uint8_t* pks48, size_t n, int* handle, uint8_t* status);
int blsgpu_pool_free(blsgpu_ctx* ctx, int handle);
int blsgpu_pool_fast_aggregate_verify(blsgpu_ctx* ctx, int handle, const uint32_t* idx /* ncomm*k */, const uint64_t* bitmap, size_t k,
                                      const uint8_t* msg32, const uint8_t* sig96, size_t ncomm, uint8_t* status, uint8_t* agg_pk48_out);

/* ---- signature sets (the shape of Lighthouse's verify_signature_sets / blst's verify_multiple_aggregate_signatures): set s = the keys
 *      [key_off[s], key_off[s+1]) of pks48 (bitmap, nullable: bit i of the FLAT key list selects key i), the message
 *      msg[msg_off[s] .. msg_off[s+1]) (msg_off NULL = fixed 32-byte messages) and the signature sig96[s].  Committees of any size, messages of any length.
 * status[s] = exactly what blsgpu_fast_aggregate_verify_batch reports for that set:
 *   0 / 1 = pairing check true / false;
 *   2 = a selected key fails to decode / is outside the subgroup, no key is selected, or the aggregate is the identity;
 *   3 = the signature fails to decode / is outside the subgroup.
 * seed16 NULL: every set gets its own pairing check.
 * seed16 set:  one random-linear-combination equation per piece of 4,096 sets, r_s = 64 non-zero bits of SHA-256(seed16 || le64(s)) (the derivation of
 *              blsgpu_verify_batch_rlc); pieces whose equation fails are re-run per set inside the call, so status equals the seed16 == NULL outcome
 *              except with probability <= 2^-64 per failing piece.  The seed must be unpredictable to whoever produced the sets.
 * ok_bitmap (nullable): ceil(nsets/64) words, bit s set <=> status[s] == 0.  fallback_sets (nullable, HOST memory): sets re-run per set.
 * In device pointer mode key_off is read back to the host once (the internal passes are planned there); a decreasing key_off is BLSGPU_ERR_ARG. */
int blsgpu_verify_signature_sets(blsgpu_ctx* ctx, const uint8_t* pks48, const uint32_t* key_off, const uint64_t* bitmap,
                                 const uint8_t* msg, const uint32_t* msg_off, const uint8_t* sig96, size_t nsets,
                                 const uint8_t* seed16, uint8_t* status, uint64_t* ok_bitmap, uint64_t* fallback_sets);
/* the same with the keys given as indices into a resident pool (blsgpu_pool_create); an out-of-range index or an undecodable pool key
 * makes its set 2 (as blsgpu_pool_fast_aggregate_verify) */
int blsgpu_pool_verify_signature_sets(blsgpu_ctx* ctx, int handle, const uint32_t* idx, const uint32_t* key_off, const uint64_t* bitmap,
                                      const uint8_t* msg, const uint32_t* msg_off, const uint8_t* sig96, size_t nsets,
                                      const uint8_t* seed16, uint8_t* status, uint64_t* ok_bitmap, uint64_t* fallback_sets);

/* ---- hash_to_g2  (src/bls.rs:477-493; algorithm spec src/hasher.rs:58-173, 352-502, 294-348, 664-673) ------- */
int blsgpu_hash_to_g2_batch(blsgpu_ctx* ctx, const uint8_t* msg, const uint32_t* msg_off, size_t n, uint8_t* out96);

/* ---- PublicKey::aggregate / Signature::aggregate  (src/bls.rs:183-195, 288-300) ----------------------------
 * seg_off: nseg+1 point offsets.  status: 0 ok, 4 = empty segment (None), 2 / 3 = a member failed to decode. */
int blsgpu_g1_aggregate(blsgpu_ctx* ctx, const uint8_t* pts48, const uint32_t* seg_off, size_t nseg, uint8_t* out48, uint8_t* status);
int blsgpu_g2_aggregate(blsgpu_ctx* ctx, const uint8_t* pts96, const uint32_t* seg_off, size_t nseg, uint8_t* out96, uint8_t* status);

/* ---- TryFrom<&[u8]> for PublicKey / Signature  (src/bls.rs:219-223, 316-320) -> BLSGPU_DE_* per item -------- */
int blsgpu_deserialize_g1(blsgpu_ctx* ctx, const uint8_t* in48, size_t n, uint8_t* status);
int blsgpu_deserialize_g2(blsgpu_ctx* ctx, const uint8_t* in96, size_t n, uint8_t* status);

/* ---- ZCash UNCOMPRESSED encodings (96-byte G1 = x || y, 192-byte G2 = x.c1 || x.c0 || y.c1 || y.c0; ark-serialize's
 *      serialize_uncompressed / deserialize_uncompressed of the types of src/bls.rs:135-138, 262-265): conversion in both directions with
 *      full validation of the input (on curve + subgroup, Validate::Yes).  status (nullable): BLSGPU_DE_* of the input; an input that does
 *      not decode gives an all-zero output. */
int blsgpu_g1_uncompress(blsgpu_ctx* ctx, const uint8_t* in48, size_t n, uint8_t* out96, uint8_t* status);
int blsgpu_g1_compress(blsgpu_ctx* ctx, const uint8_t* in96, size_t n, uint8_t* out48, uint8_t* status);
int blsgpu_g2_uncompress(blsgpu_ctx* ctx, const uint8_t* in96, size_t n, uint8_t* out192, uint8_t* status);
int blsgpu_g2_compress(blsgpu_ctx* ctx, const uint8_t* in192, size_t n, uint8_t* out96, uint8_t* status);

/* ---- PublicKey::from(&PrivateKey) / keygen's derivation  (src/bls.rs:210-216, 395-409) ---------------------- */
int blsgpu_sk_to_pk_batch(blsgpu_ctx* ctx, const uint8_t* sk32_le, size_t n, uint8_t* pk48, uint8_t* status /* nullable; 5 = non-canonical */);
/* ---- BLS::sign  (src/bls.rs:411-425) ------------------------------------------------------------------------ */
int blsgpu_sign_batch(blsgpu_ctx* ctx, const uint8_t* sk32_le, const uint8_t* msg, const uint32_t* msg_off, size_t n,
                      uint8_t* sig96, uint8_t* status);

/* ---- Bls12::multi_pairing(...).0  (src/bls.rs:454-455; parity hook for GT bytes) ----------------------------
 * nprod products of npairs (1 or 2) pairings each: g1_48[nprod*npairs], g2_96[nprod*npairs] -> gt[nprod*576].
 * Pairs containing the identity are dropped like ark-ec does; status (nullable): 2/3 when a point fails to decode. */
int blsgpu_pairing_gt(blsgpu_ctx* ctx, const uint8_t* g1_48, const uint8_t* g2_96, size_t npairs, size_t nprod,
                      uint8_t* gt_le576, uint8_t* status);
/* fold GT partial products (multi-GPU epilogue): out = prod_i parts[i], parts = nparts x 576 bytes */
int blsgpu_gt_fold(blsgpu_ctx* ctx, const uint8_t* parts_le576, size_t nparts, uint8_t* out_le576);

/* ---- Fp Montgomery product on raw 48-byte little-endian limb images (kernel K0 parity hook) ----------------- */
int blsgpu_fp_mul_raw(blsgpu_ctx* ctx, const uint8_t* a48, const uint8_t* b48, size_t n, uint8_t* out48, int reps);
/* IMAD.WIDE.U32 issue-rate microbenchmark: returns measured 32x32->64 multiply-accumulates per second */
int blsgpu_imad_peak(blsgpu_ctx* ctx, int mode /* 0 = independent mad.wide.u32, 1 = mad.lo.cc/madc.hi.cc carry chains, 2 = chained Montgomery products */,
                     double* mac32_per_sec, double* ms);

/* ---- R1CS satisfaction check  (ark-relations ConstraintSystem::is_satisfied on the circuit of
 *      src/constraints.rs:90-128; every row is reported, no early exit) --------------------------------------
 * Three CSR matrices with canonical 48-byte little-endian coefficients in Fq; z = nwit vectors of ncols canonical
 * 48-byte little-endian values laid out witness-major ([w][col]); sat_bits: nwit x ceil(nrows/64) words. */
int blsgpu_r1cs_load(blsgpu_ctx* ctx, const uint64_t* const rowptr[3], const uint32_t* const col[3], const uint8_t* const coeff48[3],
                     size_t nrows, size_t ncols, int* handle);
int blsgpu_r1cs_check(blsgpu_ctx* ctx, int handle, const uint8_t* z48, size_t nwit, uint64_t* sat_bits, uint8_t* all_sat);
int blsgpu_r1cs_free(blsgpu_ctx* ctx, int handle);
/* The same through a file (format "BLSR1CS1": header, three CSR matrices, nwit assignments -- written by rust/examples/export_r1cs.rs from
 * arkworks' cs.to_matrices() after src/constraints.rs:335-367, or by bls_verify_gadget_b200/gadget.py; layout in csrc/r1cs.cuh).
 * shape4 (nullable) = {nrows, ncols, ninstance, nwit}.  blsgpu_r1cs_check_file checks assignments [first, first + count) of the file;
 * its sat_bits / all_sat are HOST pointers whatever the pointer mode. */
int blsgpu_r1cs_load_file(blsgpu_ctx* ctx, const char* path, int* handle, uint64_t shape4[4]);
int blsgpu_r1cs_check_file(blsgpu_ctx* ctx, int handle, const char* path, size_t first, size_t count, uint64_t* sat_bits, uint8_t* all_sat);
/* how blsgpu_r1cs_load classified the rows: counts[0] truth-table rows (<= 16 non-zeros on <= 5 distinct columns: evaluated bit-sliced over
 * 32 assignments when those columns are 0/1, generically otherwise), [1] generic short rows, [2] long rows, [3] the 32-term
 * metadata rounds the long-row kernel walks (sum over long rows and matrices of ceil(nnz / 32)) */
int blsgpu_r1cs_row_classes(blsgpu_ctx* ctx, int handle, uint64_t counts[4]);

/* ---- GPU witness generation for the verify circuit (SURVEY 8(f)-1; no counterpart in the reference, whose assignments come from
 *      running the gadget code of src/constraints.rs:335-370 under ark-relations) -------------------------------------------------
 * blsgpu_witness_load takes the witness program exported by the host-side builder (libblsgadget.so, blsgadget_program_export):
 * rules16 = ncols records {u8 kind, u8 0, u16 aux, u32 a, u32 b, u32 d}, lc_ptr[nlc + 1], lc_col / lc_coef48 (canonical LE) [nterms].
 * The program fixes the message length L of its circuit (blsgpu_witness_msg_len; the gadget takes &[UInt8] of any length,
 * src/constraints.rs:90-95, and the number of SHA-256 blocks depends on it): msg = nwit x L bytes.
 * blsgpu_witness_gen replays it for nwit (pk48, msg, sig96) triples: z48 = nwit * nvars * 48 bytes in the layout of
 * blsgpu_r1cs_check; status[i] (nullable) = 0, or 2 / 3 when the key / signature does not decode to a non-identity point. */
int blsgpu_witness_load(blsgpu_ctx* ctx, const uint8_t* rules16, const uint64_t* lc_ptr, const uint32_t* lc_col, const uint8_t* lc_coef48,
                        size_t ncols /* rules: circuit variables, then scratch columns */, size_t nvars /* circuit variables */, size_t nlc, size_t nterms,
                        const uint32_t* order /* variables sorted by dependency level */, const uint64_t* level_ptr /* nlevels + 1 */, size_t nlevels,
                        int* handle);   /* host pointers; the rules of one level run in parallel.  order, level_ptr and nlevels come from
                                         * blsgadget_program_levels and are required: BLSGPU_ERR_ARG without them */
int blsgpu_witness_gen(blsgpu_ctx* ctx, int handle, const uint8_t* pk48, const uint8_t* msg, const uint8_t* sig96, size_t nwit,
                       uint8_t* z48, uint8_t* status);
/* Generation and satisfaction check in one call: (pk, msg, sig) bytes in, per-constraint bits (words64 per assignment) and the
 * per-assignment flag out, as blsgpu_r1cs_check would report them for blsgpu_witness_gen's output -- but the assignments stay in
 * the device-side transposed layout (no row-major copy of 34 MB per assignment, no second transpose).  r1cs_handle must be the
 * system of the circuit the program was recorded with; all_sat and status are nullable. */
int blsgpu_witness_check(blsgpu_ctx* ctx, int wit_handle, int r1cs_handle, const uint8_t* pk48, const uint8_t* msg, const uint8_t* sig96, size_t nwit,
                         uint64_t* sat_bits, uint8_t* all_sat, uint8_t* status);
long blsgpu_witness_msg_len(blsgpu_ctx* ctx, int handle);   /* L of the loaded program, -1 for a bad handle */
/* how the loaded program was split: counts[0] "light" rules (0/1 and small-integer values: the SHA-256 / bit gadgets, evaluated bit-sliced by one CTA
 * per group of 32 assignments), [1] their dependency levels, [2] dependency levels of the remaining field rules, [3] integer scratch slots */
int blsgpu_witness_shape(blsgpu_ctx* ctx, int handle, uint64_t counts[4]);
/* The aggregate_verify circuit (BlsSignatureVerifyGadget::aggregate_verify / mapped_aggregate, src/constraints.rs:153-191): load the program
 * recorded by blsgadget_aggregate_verify_program with blsgpu_witness_load_aggregate (which takes its key count), then
 * pks48 = nwit x nkeys compressed keys, bitmap = nwit x nkeys bytes (0 / non-zero = the participation bits), msg = nwit x L bytes,
 * sig96 = nwit aggregate signatures.  status: 2 when any key of an item does not decode to a non-identity point, 3 for the signature. */
int blsgpu_witness_load_aggregate(blsgpu_ctx* ctx, const uint8_t* rules16, const uint64_t* lc_ptr, const uint32_t* lc_col, const uint8_t* lc_coef48,
                                  size_t ncols, size_t nvars, size_t nlc, size_t nterms, const uint32_t* order, const uint64_t* level_ptr, size_t nlevels,
                                  size_t nkeys, int* handle);
int blsgpu_witness_gen_aggregate(blsgpu_ctx* ctx, int handle, const uint8_t* pks48, const uint8_t* bitmap, const uint8_t* msg, const uint8_t* sig96, size_t nwit,
                                 uint8_t* z48, uint8_t* status);
int blsgpu_witness_check_aggregate(blsgpu_ctx* ctx, int wit_handle, int r1cs_handle, const uint8_t* pks48, const uint8_t* bitmap, const uint8_t* msg, const uint8_t* sig96, size_t nwit,
                                   uint64_t* sat_bits, uint8_t* all_sat, uint8_t* status);
int blsgpu_witness_free(blsgpu_ctx* ctx, int handle);

/* ---- every GPU of the box behind one handle (SURVEY 8(b), 8(e)) ---------------------------------------------------------------------
 * blsgpu_create_multi: devices = ndev ordinals (NULL / ndev <= 0: every visible device); one single-GPU context and stream per device and
 * one NCCL communicator over them (ncclCommInitAll; libnccl.so.2 is bound with dlopen at this point, never for single-GPU use).
 * blsgpu_multi_verify_batch = BLS::verify (src/bls.rs:427-458) over a batch sharded contiguously across the devices (shard sizes are
 * multiples of 64), HOST pointers, outputs as blsgpu_verify_batch.  No data-path collective; the one exchange is an all-gather of the
 * ok-bitmap shards and the 576-byte GT partials followed by a fold in rank order on every device, so each GPU ends with the whole-batch
 * bitmap and GT accumulator (blsgpu_multi_peek reads device i's copies back: the test hook).  One host thread at a time per handle. */
typedef struct blsgpu_multi blsgpu_multi;
int  blsgpu_create_multi(blsgpu_multi** out, const int* devices, int ndev);
void blsgpu_destroy_multi(blsgpu_multi* m);
const char* blsgpu_multi_last_error(blsgpu_multi* m);
int  blsgpu_multi_ndev(blsgpu_multi* m);
int  blsgpu_multi_nccl_version(blsgpu_multi* m);            /* ncclGetVersion of the library that was bound, e.g. 22703 */
blsgpu_ctx* blsgpu_multi_ctx(blsgpu_multi* m, int i);       /* device slot i's context (DEVICE pointer mode) for per-device calls of the rest of the ABI */
int  blsgpu_multi_verify_batch(blsgpu_multi* m, const uint8_t* pk48, const uint8_t* msg, const uint32_t* msg_off, const uint8_t* sig96, size_t n,
                               uint8_t* status, uint64_t* ok_bitmap, uint8_t* gt_acc_le576);
int  blsgpu_multi_peek(blsgpu_multi* m, int i, size_t n, uint64_t* ok_bitmap, uint8_t* gt_le576);

#ifdef __cplusplus
}
#endif
#endif
