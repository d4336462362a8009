//! `extern "C"` block: one declaration per entry point of include/blsgpu.h (the drop-in boundary).  Citations name the
//! reference interface each entry point replaces (paths relative to lightec-xyz/bls-verify-gadget).
#![allow(non_camel_case_types, dead_code)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)] pub struct blsgpu_ctx { _private: [u8; 0] }
#[repr(C)] pub struct blsgpu_multi { _private: [u8; 0] }

pub const ST_TRUE: u8 = 0;          // Ok(true)                          src/bls.rs:457
pub const ST_FALSE: u8 = 1;         // Ok(false)                         src/bls.rs:457
pub const ST_BAD_PUBKEY: u8 = 2;    // Err(InvalidPublicKey)             src/bls.rs:434-442
pub const ST_BAD_SIG: u8 = 3;       // Err(InvalidSignature)             src/bls.rs:443-447
pub const ST_EMPTY: u8 = 4;         // aggregate of nothing = None       src/bls.rs:184-185, 289-290
pub const ST_BAD_SECKEY: u8 = 5;    // Err(InvalidSecretKey)             src/bls.rs:417-419

extern "C" {
    pub fn blsgpu_create(out: *mut *mut blsgpu_ctx, device: c_int) -> c_int;
    pub fn blsgpu_destroy(ctx: *mut blsgpu_ctx);
    pub fn blsgpu_last_error(ctx: *mut blsgpu_ctx) -> *const c_char;
    pub fn blsgpu_set_stream(ctx: *mut blsgpu_ctx, cuda_stream: *mut c_void, use_own: c_int) -> c_int;
    pub fn blsgpu_set_pointer_mode(ctx: *mut blsgpu_ctx, mode: c_int) -> c_int;
    // memory / tuning switches (INTEGRATION.md section 7); results do not depend on them
    pub fn blsgpu_set_chunk(ctx: *mut blsgpu_ctx, items: usize) -> c_int;
    pub fn blsgpu_set_lanes(ctx: *mut blsgpu_ctx, lanes: c_int) -> c_int;
    pub fn blsgpu_set_split(ctx: *mut blsgpu_ctx, on: c_int) -> c_int;
    pub fn blsgpu_synchronize(ctx: *mut blsgpu_ctx) -> c_int;
    // <BLS<P> as SignatureScheme>::verify, src/bls.rs:427-458 (incl. the TryFrom decoding of tests/tests.rs:244-254)
    pub fn blsgpu_verify_batch(ctx: *mut blsgpu_ctx, pk48: *const u8, msg: *const u8, msg_off: *const u32, sig96: *const u8, n: usize,
                               status: *mut u8, ok_bitmap: *mut u64, gt_acc_le576: *mut u8) -> c_int;
    // additional fast path: one pairing-product equation per batch; on failure the bad items are located inside the library
    pub fn blsgpu_verify_batch_rlc(ctx: *mut blsgpu_ctx, pk48: *const u8, msg: *const u8, msg_off: *const u32, sig96: *const u8, n: usize,
                                   seed16: *const u8, status: *mut u8, all_ok: *mut u8) -> c_int;
    pub fn blsgpu_verify_batch_rlc_bisect(ctx: *mut blsgpu_ctx, pk48: *const u8, msg: *const u8, msg_off: *const u32, sig96: *const u8, n: usize,
                                          seed16: *const u8, status: *mut u8, ok_bitmap: *mut u64, nbad: *mut u64) -> c_int;
    // PublicKey::aggregate + verify, src/bls.rs:183-195 then 427-458 (tests/tests.rs:297-334)
    pub fn blsgpu_fast_aggregate_verify_batch(ctx: *mut blsgpu_ctx, pks48: *const u8, bitmap: *const u64, k: usize, msg32: *const u8,
                                              sig96: *const u8, ncomm: usize, status: *mut u8, agg_pk48_out: *mut u8) -> c_int;
    // Eth2 aggregate_verify (distinct messages; tests/readme.md:4-7 names the category): one signature over k (pk_j, msg_j) pairs
    pub fn blsgpu_aggregate_verify_batch(ctx: *mut blsgpu_ctx, pks48: *const u8, msg: *const u8, msg_off: *const u32, pair_off: *const u32,
                                         sig96: *const u8, nsig: usize, status: *mut u8) -> c_int;
    // signature sets (Lighthouse verify_signature_sets / blst verify_multiple_aggregate_signatures shape): keys [key_off[s], key_off[s+1]),
    // one message and one signature per set; seed16 non-null = per-piece random-linear-combination equations with the exact per-set outcome
    pub fn blsgpu_verify_signature_sets(ctx: *mut blsgpu_ctx, pks48: *const u8, key_off: *const u32, bitmap: *const u64, msg: *const u8, msg_off: *const u32,
                                        sig96: *const u8, nsets: usize, seed16: *const u8, status: *mut u8, ok_bitmap: *mut u64, fallback_sets: *mut u64) -> c_int;
    pub fn blsgpu_pool_verify_signature_sets(ctx: *mut blsgpu_ctx, handle: c_int, idx: *const u32, key_off: *const u32, bitmap: *const u64, msg: *const u8,
                                             msg_off: *const u32, sig96: *const u8, nsets: usize, seed16: *const u8, status: *mut u8, ok_bitmap: *mut u64,
                                             fallback_sets: *mut u64) -> c_int;
    pub fn blsgpu_hash_to_g2_batch(ctx: *mut blsgpu_ctx, msg: *const u8, msg_off: *const u32, n: usize, out96: *mut u8) -> c_int;          // src/bls.rs:477-493
    pub fn blsgpu_g1_aggregate(ctx: *mut blsgpu_ctx, pts48: *const u8, seg_off: *const u32, nseg: usize, out48: *mut u8, status: *mut u8) -> c_int;   // src/bls.rs:183-195
    pub fn blsgpu_g2_aggregate(ctx: *mut blsgpu_ctx, pts96: *const u8, seg_off: *const u32, nseg: usize, out96: *mut u8, status: *mut u8) -> c_int;   // src/bls.rs:288-300
    pub fn blsgpu_deserialize_g1(ctx: *mut blsgpu_ctx, in48: *const u8, n: usize, status: *mut u8) -> c_int;                                // src/bls.rs:219-223
    pub fn blsgpu_deserialize_g2(ctx: *mut blsgpu_ctx, in96: *const u8, n: usize, status: *mut u8) -> c_int;                                // src/bls.rs:316-320
    // uncompressed ZCash encodings (96 / 192 bytes): the other wire format of the upstream bls12-381-tests suite
    pub fn blsgpu_g1_uncompress(ctx: *mut blsgpu_ctx, in48: *const u8, n: usize, out96: *mut u8, status: *mut u8) -> c_int;
    pub fn blsgpu_g1_compress(ctx: *mut blsgpu_ctx, in96: *const u8, n: usize, out48: *mut u8, status: *mut u8) -> c_int;
    pub fn blsgpu_g2_uncompress(ctx: *mut blsgpu_ctx, in96: *const u8, n: usize, out192: *mut u8, status: *mut u8) -> c_int;
    pub fn blsgpu_g2_compress(ctx: *mut blsgpu_ctx, in192: *const u8, n: usize, out96: *mut u8, status: *mut u8) -> c_int;
    pub fn blsgpu_sk_to_pk_batch(ctx: *mut blsgpu_ctx, sk32_le: *const u8, n: usize, pk48: *mut u8, status: *mut u8) -> c_int;              // src/bls.rs:210-216
    pub fn blsgpu_sign_batch(ctx: *mut blsgpu_ctx, sk32_le: *const u8, msg: *const u8, msg_off: *const u32, n: usize, sig96: *mut u8, status: *mut u8) -> c_int;   // src/bls.rs:411-425
    pub fn blsgpu_pairing_gt(ctx: *mut blsgpu_ctx, g1_48: *const u8, g2_96: *const u8, npairs: usize, nprod: usize, gt_le576: *mut u8, status: *mut u8) -> c_int; // src/bls.rs:454-455
    pub fn blsgpu_gt_fold(ctx: *mut blsgpu_ctx, parts: *const u8, nparts: usize, out: *mut u8) -> c_int;
    // ark-relations ConstraintSystem::is_satisfied on the circuits of src/constraints.rs:90-191 (every row reported)
    pub fn blsgpu_r1cs_load(ctx: *mut blsgpu_ctx, rowptr: *const *const u64, col: *const *const u32, coeff48: *const *const u8,
                            nrows: usize, ncols: usize, handle: *mut c_int) -> c_int;
    pub fn blsgpu_r1cs_load_file(ctx: *mut blsgpu_ctx, path: *const c_char, handle: *mut c_int, shape4: *mut u64) -> c_int;
    pub fn blsgpu_r1cs_check(ctx: *mut blsgpu_ctx, handle: c_int, z48: *const u8, nwit: usize, sat_bits: *mut u64, all_sat: *mut u8) -> c_int;
    pub fn blsgpu_r1cs_check_file(ctx: *mut blsgpu_ctx, handle: c_int, path: *const c_char, first: usize, count: usize, sat_bits: *mut u64, all_sat: *mut u8) -> c_int;
    pub fn blsgpu_r1cs_free(ctx: *mut blsgpu_ctx, handle: c_int) -> c_int;
    // every GPU of the box behind one handle (NCCL exchange inside)
    pub fn blsgpu_create_multi(out: *mut *mut blsgpu_multi, devices: *const c_int, ndev: c_int) -> c_int;
    pub fn blsgpu_destroy_multi(m: *mut blsgpu_multi);
    pub fn blsgpu_multi_last_error(m: *mut blsgpu_multi) -> *const c_char;
    pub fn blsgpu_multi_ndev(m: *mut blsgpu_multi) -> c_int;
    pub fn blsgpu_multi_verify_batch(m: *mut blsgpu_multi, pk48: *const u8, msg: *const u8, msg_off: *const u32, sig96: *const u8, n: usize,
                                     status: *mut u8, ok_bitmap: *mut u64, gt_acc_le576: *mut u8) -> c_int;
}
