//! GPU-backed drop-in for the public surface of `lightec-xyz/bls-verify-gadget`'s `src/bls.rs`.
//!
//! Same names, argument meaning and error behaviour as the reference; every value type holds the crate's own
//! serialisation (48-byte / 96-byte ZCash compressed points, 32-byte little-endian scalar), which is exactly what the
//! C ABI of `include/blsgpu.h` consumes, so no arkworks type crosses the boundary:
//!
//! | reference (src/bls.rs)                                   | here                                            |
//! |----------------------------------------------------------|-------------------------------------------------|
//! | `Parameters` :25-36, `PrivateKey` :52-121                | same names, byte-backed                         |
//! | `PublicKey` :135-260 (`aggregate` :183-195, `From<&sk>`) | `blsgpu_g1_aggregate`, `blsgpu_sk_to_pk_batch`  |
//! | `Signature` :262-357 (`aggregate` :288-300)              | `blsgpu_g2_aggregate`                           |
//! | `TryFrom<&[u8] / &str / String>`, `Into<Vec<u8> / String>` | `blsgpu_deserialize_g1/g2` (validation)        |
//! | `BLS::{setup, keygen, sign, verify}` :379-475            | `blsgpu_sign_batch`, `blsgpu_verify_batch`      |
//! | `hash_to_g2` :477-493                                    | `blsgpu_hash_to_g2_batch`                       |
//! | `BLSError` :359-377                                      | status bytes 5 / 2 / 3                          |
//!
//! Batch callers (the case a GPU is for) use [`verify_batch`] / [`MultiGpu::verify_batch`]; the single-item methods are
//! n = 1 calls of the same entry points.  There is no CPU fallback: without a B200 every call fails.
pub mod ffi;
use ffi::*;
use std::ffi::CStr;
use std::fmt;
use std::sync::Mutex;

pub type Error = Box<dyn std::error::Error>;

#[derive(Debug)]
pub enum BLSError { InvalidSecretKey, InvalidPublicKey, InvalidSignature }          // src/bls.rs:359-364
impl fmt::Display for BLSError {
    fn fmt(&self, f: &mut fmt::Formatter<'_>) -> fmt::Result {
        f.write_str(match self { Self::InvalidSecretKey => "invalid secret key", Self::InvalidPublicKey => "invalid public key", Self::InvalidSignature => "invalid signature" })
    }
}
impl std::error::Error for BLSError {}

/// What `ark_serialize::SerializationError` is to the reference's `TryFrom` impls.
#[derive(Debug)]
pub enum SerializationError { InvalidData, UnexpectedFlags, NotEnoughSpace }
impl fmt::Display for SerializationError { fn fmt(&self, f: &mut fmt::Formatter<'_>) -> fmt::Result { write!(f, "{:?}", self) } }
impl std::error::Error for SerializationError {}

#[derive(Debug)]
pub struct GpuError(pub String);
impl fmt::Display for GpuError { fn fmt(&self, f: &mut fmt::Formatter<'_>) -> fmt::Result { f.write_str(&self.0) } }
impl std::error::Error for GpuError {}

// ---- the process-wide context (one GPU; a context serves one host thread at a time, hence the mutex)
struct Ctx(*mut blsgpu_ctx);
unsafe impl Send for Ctx {}
static CTX: Mutex<Option<Ctx>> = Mutex::new(None);
fn with_ctx<T>(f: impl FnOnce(*mut blsgpu_ctx) -> T) -> Result<T, Error> {
    let mut g = CTX.lock().unwrap();
    if g.is_none() {
        let mut p: *mut blsgpu_ctx = std::ptr::null_mut();
        let rc = unsafe { blsgpu_create(&mut p, -1) };
        if rc != 0 { return Err(Box::new(GpuError(format!("blsgpu_create failed (rc = {rc}): no usable sm_100 CUDA device; libblsgpu has no CPU fallback")))); }
        *g = Some(Ctx(p));
    }
    Ok(f(g.as_ref().unwrap().0))
}
fn check(ctx: *mut blsgpu_ctx, rc: i32) -> Result<(), Error> {
    if rc == 0 { return Ok(()); }
    let msg = unsafe { CStr::from_ptr(blsgpu_last_error(ctx)) }.to_string_lossy().into_owned();
    Err(Box::new(GpuError(format!("libblsgpu rc = {rc}: {msg}"))))
}

// ---- value types: Copy, returned by value, nothing retained between calls (src/bls.rs:25, 52, 135, 262)
#[derive(Copy, Clone, PartialEq, Eq, Debug)]
pub struct Parameters { pub g1_generator: [u8; 48] }
impl Default for Parameters {
    fn default() -> Self {          // G1Projective::generator(), compressed
        let mut g = [0u8; 48];
        hex::decode_to_slice("97f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb", &mut g).unwrap();
        Parameters { g1_generator: g }
    }
}

#[derive(Copy, Clone, PartialEq, Eq)]
pub struct PrivateKey { pub private_key: [u8; 32] }                   // canonical Fr, little-endian (src/bls.rs:79-121)
impl Default for PrivateKey { fn default() -> Self { PrivateKey { private_key: [0; 32] } } }
impl fmt::Debug for PrivateKey { fn fmt(&self, f: &mut fmt::Formatter) -> fmt::Result { write!(f, "{}", hex::encode(self.private_key)) } }
const R_ORDER_LE: [u8; 32] = [0x01, 0, 0, 0, 0xff, 0xff, 0xff, 0xff, 0xfe, 0x5b, 0xfe, 0xff, 0x02, 0xa4, 0xbd, 0x53, 0x05, 0xd8, 0xa1, 0x09, 0x08, 0xd8, 0x39, 0x33, 0x48, 0x7d, 0x9d, 0x29, 0x53, 0xa7, 0xed, 0x73];
impl TryFrom<&[u8]> for PrivateKey {
    type Error = SerializationError;
    fn try_from(bytes: &[u8]) -> Result<Self, SerializationError> {
        if bytes.len() < 32 { return Err(SerializationError::NotEnoughSpace); }
        let mut k = [0u8; 32]; k.copy_from_slice(&bytes[..32]);
        for i in (0..32).rev() { if k[i] != R_ORDER_LE[i] { return if k[i] < R_ORDER_LE[i] { Ok(PrivateKey { private_key: k }) } else { Err(SerializationError::InvalidData) }; } }
        Err(SerializationError::InvalidData)                                // == r is not canonical
    }
}
impl TryFrom<&str> for PrivateKey { type Error = SerializationError; fn try_from(s: &str) -> Result<Self, SerializationError> { PrivateKey::try_from(&hex::decode(s).unwrap()[..]) } }   // malformed hex panics, as in src/bls.rs:83, 92
impl TryFrom<String> for PrivateKey { type Error = SerializationError; fn try_from(s: String) -> Result<Self, SerializationError> { PrivateKey::try_from(s.as_str()) } }
impl From<PrivateKey> for Vec<u8> { fn from(k: PrivateKey) -> Vec<u8> { k.private_key.to_vec() } }
impl From<PrivateKey> for String { fn from(k: PrivateKey) -> String { hex::encode(k.private_key) } }

fn decode_code_to_result(code: u8) -> Result<(), SerializationError> {
    match code { 0 | 1 => Ok(()), 2 => Err(SerializationError::UnexpectedFlags), _ => Err(SerializationError::InvalidData) }       // BLSGPU_DE_* of include/blsgpu.h
}

#[derive(Copy, Clone, PartialEq, Eq)]
pub struct PublicKey { pub public_key: [u8; 48] }
impl Default for PublicKey { fn default() -> Self { let mut b = [0u8; 48]; b[0] = 0xc0; PublicKey { public_key: b } } }      // the identity (src/bls.rs:139-145)
impl fmt::Debug for PublicKey { fn fmt(&self, f: &mut fmt::Formatter) -> fmt::Result { write!(f, "{}", hex::encode(self.public_key)) } }
impl PublicKey {
    /// `PublicKey::aggregate` (src/bls.rs:183-195): the sum of the keys, `None` for an empty list.
    pub fn aggregate(public_keys: &Vec<PublicKey>) -> Option<PublicKey> {
        if public_keys.is_empty() { return None; }
        let flat: Vec<u8> = public_keys.iter().flat_map(|p| p.public_key).collect();
        let seg = [0u32, public_keys.len() as u32]; let (mut out, mut st) = ([0u8; 48], [0u8; 1]);
        with_ctx(|c| unsafe { blsgpu_g1_aggregate(c, flat.as_ptr(), seg.as_ptr(), 1, out.as_mut_ptr(), st.as_mut_ptr()) }).ok().filter(|rc| *rc == 0)?;
        if st[0] == ST_TRUE { Some(PublicKey { public_key: out }) } else { None }
    }
}
impl From<&PrivateKey> for PublicKey {                                  // generator * sk (src/bls.rs:210-216)
    fn from(sk: &PrivateKey) -> PublicKey {
        let (mut out, mut st) = ([0u8; 48], [0u8; 1]);
        with_ctx(|c| unsafe { blsgpu_sk_to_pk_batch(c, sk.private_key.as_ptr(), 1, out.as_mut_ptr(), st.as_mut_ptr()) }).expect("GPU context");
        PublicKey { public_key: out }
    }
}
impl TryFrom<&[u8]> for PublicKey {                                     // deserialize_compressed with validation (src/bls.rs:219-223)
    type Error = SerializationError;
    fn try_from(bytes: &[u8]) -> Result<Self, SerializationError> {
        if bytes.len() < 48 { return Err(SerializationError::NotEnoughSpace); }
        let mut st = [0u8; 1];
        with_ctx(|c| unsafe { blsgpu_deserialize_g1(c, bytes.as_ptr(), 1, st.as_mut_ptr()) }).map_err(|_| SerializationError::InvalidData)?;
        decode_code_to_result(st[0])?;
        let mut b = [0u8; 48]; b.copy_from_slice(&bytes[..48]); Ok(PublicKey { public_key: b })
    }
}
impl TryFrom<&str> for PublicKey { type Error = SerializationError; fn try_from(s: &str) -> Result<Self, SerializationError> { PublicKey::try_from(&hex::decode(s).unwrap()[..]) } }
impl TryFrom<String> for PublicKey { type Error = SerializationError; fn try_from(s: String) -> Result<Self, SerializationError> { PublicKey::try_from(s.as_str()) } }
impl From<PublicKey> for Vec<u8> { fn from(k: PublicKey) -> Vec<u8> { k.public_key.to_vec() } }
impl From<PublicKey> for String { fn from(k: PublicKey) -> String { hex::encode(k.public_key) } }

#[derive(Copy, Clone, PartialEq, Eq)]
pub struct Signature { pub sig: [u8; 96] }
impl Default for Signature { fn default() -> Self { let mut b = [0u8; 96]; b[0] = 0xc0; Signature { sig: b } } }
impl fmt::Debug for Signature { fn fmt(&self, f: &mut fmt::Formatter) -> fmt::Result { write!(f, "{}", hex::encode(self.sig)) } }
impl Signature {
    /// `Signature::aggregate` (src/bls.rs:288-300).
    pub fn aggregate(signatures: &Vec<Signature>) -> Option<Signature> {
        if signatures.is_empty() { return None; }
        let flat: Vec<u8> = signatures.iter().flat_map(|s| s.sig).collect();
        let seg = [0u32, signatures.len() as u32]; let (mut out, mut st) = ([0u8; 96], [0u8; 1]);
        with_ctx(|c| unsafe { blsgpu_g2_aggregate(c, flat.as_ptr(), seg.as_ptr(), 1, out.as_mut_ptr(), st.as_mut_ptr()) }).ok().filter(|rc| *rc == 0)?;
        if st[0] == ST_TRUE { Some(Signature { sig: out }) } else { None }
    }
}
impl TryFrom<&[u8]> for Signature {                                     // src/bls.rs:316-320
    type Error = SerializationError;
    fn try_from(bytes: &[u8]) -> Result<Self, SerializationError> {
        if bytes.len() < 96 { return Err(SerializationError::NotEnoughSpace); }
        let mut st = [0u8; 1];
        with_ctx(|c| unsafe { blsgpu_deserialize_g2(c, bytes.as_ptr(), 1, st.as_mut_ptr()) }).map_err(|_| SerializationError::InvalidData)?;
        decode_code_to_result(st[0])?;
        let mut b = [0u8; 96]; b.copy_from_slice(&bytes[..96]); Ok(Signature { sig: b })
    }
}
impl TryFrom<&str> for Signature { type Error = SerializationError; fn try_from(s: &str) -> Result<Self, SerializationError> { Signature::try_from(&hex::decode(s).unwrap()[..]) } }
impl TryFrom<String> for Signature { type Error = SerializationError; fn try_from(s: String) -> Result<Self, SerializationError> { Signature::try_from(s.as_str()) } }
impl From<Signature> for Vec<u8> { fn from(s: Signature) -> Vec<u8> { s.sig.to_vec() } }
impl From<Signature> for String { fn from(s: Signature) -> String { hex::encode(s.sig) } }

/// The `SignatureScheme` of the reference (src/bls.rs:379-475) with the same four entry points.
pub struct BLS;
impl BLS {
    pub fn setup<R: rand::Rng>(_rng: &mut R) -> Result<Parameters, Error> { Ok(Parameters::default()) }
    /// Uniform scalar by rejection on 255 bits, then `PublicKey::from(&sk)` (src/bls.rs:395-409).
    pub fn keygen<R: rand::Rng>(_parameters: &Parameters, rng: &mut R) -> Result<(PublicKey, PrivateKey), Error> {
        loop {
            let mut k = [0u8; 32]; rng.fill(&mut k[..]); k[31] &= 0x7f;
            if let Ok(sk) = PrivateKey::try_from(&k[..]) { return Ok((PublicKey::from(&sk), sk)); }
        }
    }
    pub fn sign<R: rand::Rng>(_parameters: &Parameters, sk: &PrivateKey, message: &[u8], _rng: &mut R) -> Result<Signature, Error> {
        let off = [0u32, message.len() as u32]; let (mut sig, mut st) = ([0u8; 96], [0u8; 1]);
        let dummy = [0u8; 1]; let m = if message.is_empty() { dummy.as_ptr() } else { message.as_ptr() };
        let (c, rc) = with_ctx(|c| (c, unsafe { blsgpu_sign_batch(c, sk.private_key.as_ptr(), m, off.as_ptr(), 1, sig.as_mut_ptr(), st.as_mut_ptr()) }))?;
        check(c, rc)?;
        if st[0] == ST_BAD_SECKEY { return Err(Box::new(BLSError::InvalidSecretKey)); }       // src/bls.rs:417-419
        Ok(Signature { sig })
    }
    pub fn verify(_parameters: &Parameters, pk: &PublicKey, message: &[u8], signature: &Signature) -> Result<bool, Error> {
        let off = [0u32, message.len() as u32]; let mut st = [0u8; 1];
        let dummy = [0u8; 1]; let m = if message.is_empty() { dummy.as_ptr() } else { message.as_ptr() };
        let (c, rc) = with_ctx(|c| (c, unsafe { blsgpu_verify_batch(c, pk.public_key.as_ptr(), m, off.as_ptr(), signature.sig.as_ptr(), 1, st.as_mut_ptr(), std::ptr::null_mut(), std::ptr::null_mut()) }))?;
        check(c, rc)?;
        match st[0] {
            ST_TRUE => Ok(true), ST_FALSE => Ok(false),
            ST_BAD_PUBKEY => Err(Box::new(BLSError::InvalidPublicKey)),                      // src/bls.rs:434-442
            _ => Err(Box::new(BLSError::InvalidSignature)),                                  // src/bls.rs:443-447
        }
    }
    pub fn randomize_public_key(_pp: &Parameters, _public_key: &PublicKey, _randomness: &[u8]) -> Result<PublicKey, Error> { unimplemented!() }     // as the reference (src/bls.rs:460-466)
    pub fn randomize_signature(_pp: &Parameters, _signature: &Signature, _randomness: &[u8]) -> Result<Signature, Error> { unimplemented!() }
}

/// `hash_to_g2` (src/bls.rs:477-493): BLS12381G2_XMD:SHA-256_SSWU_RO_ with the POP domain separation tag; compressed point.
pub fn hash_to_g2(message: &[u8]) -> Result<Signature, Error> {
    let off = [0u32, message.len() as u32]; let mut out = [0u8; 96];
    let dummy = [0u8; 1]; let m = if message.is_empty() { dummy.as_ptr() } else { message.as_ptr() };
    let (c, rc) = with_ctx(|c| (c, unsafe { blsgpu_hash_to_g2_batch(c, m, off.as_ptr(), 1, out.as_mut_ptr()) }))?;
    check(c, rc)?; Ok(Signature { sig: out })
}

/// The batch form: `status[i]` = 0 `Ok(true)`, 1 `Ok(false)`, 2 `Err(InvalidPublicKey)`, 3 `Err(InvalidSignature)`; collapsing `Err`
/// to `false` like tests/tests.rs:262 is `status[i] == 0`.  `messages` are concatenated, `msg_off` has n + 1 byte offsets.
pub fn verify_batch(pk48: &[u8], messages: &[u8], msg_off: &[u32], sig96: &[u8]) -> Result<Vec<u8>, Error> {
    let n = sig96.len() / 96; assert!(pk48.len() == 48 * n && msg_off.len() == n + 1 && *msg_off.last().unwrap() as usize <= messages.len());
    let mut st = vec![0u8; n];
    let (c, rc) = with_ctx(|c| (c, unsafe { blsgpu_verify_batch(c, pk48.as_ptr(), messages.as_ptr(), msg_off.as_ptr(), sig96.as_ptr(), n, st.as_mut_ptr(), std::ptr::null_mut(), std::ptr::null_mut()) }))?;
    check(c, rc)?; Ok(st)
}

/// Signature sets: set s = the keys `pk48[key_off[s]..key_off[s+1]]` (48 bytes each), the message `messages[msg_off[s]..msg_off[s+1]]` and
/// `sig96[s]`.  `status[s]` as [`verify_batch`] for the set's aggregate key (2 also for an empty set or an identity aggregate).  `seed16`:
/// `Some` = one random-linear-combination equation per 4,096 sets with the failing pieces re-run per set inside the library (same status except with
/// probability <= 2^-64 per failing piece; the seed must be unpredictable to whoever produced the sets).  -> (status, sets re-run per set)
pub fn verify_signature_sets(pk48: &[u8], key_off: &[u32], messages: &[u8], msg_off: &[u32], sig96: &[u8], seed16: Option<&[u8; 16]>) -> Result<(Vec<u8>, u64), Error> {
    let n = sig96.len() / 96;
    assert!(sig96.len() == 96 * n && key_off.len() == n + 1 && msg_off.len() == n + 1 && key_off.windows(2).all(|w| w[0] <= w[1]));
    assert!(48 * *key_off.last().unwrap() as usize <= pk48.len() && *msg_off.last().unwrap() as usize <= messages.len());
    let mut st = vec![0u8; n]; let mut rerun = 0u64;
    let dummy = [0u8; 1];
    let pk = if pk48.is_empty() { dummy.as_ptr() } else { pk48.as_ptr() }; let m = if messages.is_empty() { dummy.as_ptr() } else { messages.as_ptr() };
    let seed = seed16.map_or(std::ptr::null(), |s| s.as_ptr());
    let (c, rc) = with_ctx(|c| (c, unsafe { blsgpu_verify_signature_sets(c, pk, key_off.as_ptr(), std::ptr::null(), m, msg_off.as_ptr(), sig96.as_ptr(), n, seed,
                                                                         st.as_mut_ptr(), std::ptr::null_mut(), &mut rerun) }))?;
    check(c, rc)?; Ok((st, rerun))
}

/// Every GPU of the box (blsgpu_create_multi): contiguous shards, NCCL all-gather of the bitmap shards and GT partials inside the library.
pub struct MultiGpu(*mut blsgpu_multi);
impl MultiGpu {
    pub fn new(devices: &[i32]) -> Result<Self, Error> {
        let mut p: *mut blsgpu_multi = std::ptr::null_mut();
        let rc = unsafe { blsgpu_create_multi(&mut p, if devices.is_empty() { std::ptr::null() } else { devices.as_ptr() }, devices.len() as i32) };
        if rc != 0 { return Err(Box::new(GpuError(format!("blsgpu_create_multi failed (rc = {rc})")))); }
        Ok(MultiGpu(p))
    }
    pub fn ndev(&self) -> i32 { unsafe { blsgpu_multi_ndev(self.0) } }
    /// -> (status bytes, ok bitmap, 576-byte GT accumulator of the whole batch)
    pub fn verify_batch(&mut self, pk48: &[u8], messages: &[u8], msg_off: &[u32], sig96: &[u8]) -> Result<(Vec<u8>, Vec<u64>, [u8; 576]), Error> {
        let n = sig96.len() / 96; assert!(pk48.len() == 48 * n && msg_off.len() == n + 1);
        let (mut st, mut bm, mut gt) = (vec![0u8; n], vec![0u64; (n + 63) / 64], [0u8; 576]);
        let rc = unsafe { blsgpu_multi_verify_batch(self.0, pk48.as_ptr(), messages.as_ptr(), msg_off.as_ptr(), sig96.as_ptr(), n, st.as_mut_ptr(), bm.as_mut_ptr(), gt.as_mut_ptr()) };
        if rc != 0 { return Err(Box::new(GpuError(unsafe { CStr::from_ptr(blsgpu_multi_last_error(self.0)) }.to_string_lossy().into_owned()))); }
        Ok((st, bm, gt))
    }
}
impl Drop for MultiGpu { fn drop(&mut self) { unsafe { blsgpu_destroy_multi(self.0) } } }

#[cfg(test)]
mod tests {
    //! The reference's own inline tests (src/bls.rs:569-652), run on a B200 box with `cargo test`.
    use super::*;
    #[test] fn private_key_hex_round_trip() {                               // src/bls.rs:569-586
        let s = "88c522e40e4d57abd3386ff6cb2c5496d767606488f3c9f9494cd363741d4e67";
        let sk = PrivateKey::try_from(s).unwrap(); let back: String = sk.into(); assert_eq!(back, s);
    }
    #[test] fn aggregate_kat() {                                            // src/bls.rs:620-641
        let keys: Vec<PublicKey> = ["67", "68", "69", "6a"].iter().map(|l| PublicKey::from(&PrivateKey::try_from(format!("88c522e40e4d57abd3386ff6cb2c5496d767606488f3c9f9494cd363741d4e{l}")).unwrap())).collect();
        let agg: String = PublicKey::aggregate(&keys).unwrap().into();
        assert_eq!(agg, "88843ab5f8471de849950c06674238f68899e242cbc72f81bda95647caea52513139792c6511b18eaf2942d04fc54cae");
        assert!(PublicKey::aggregate(&vec![]).is_none());
    }
    #[test] fn hash_to_g2_kat() {                                           // src/bls.rs:643-652
        let h: String = hash_to_g2(&[0u8; 32]).unwrap().into();
        assert_eq!(h, "97502412bcfc3f1d88b71f1ad9b60fa37c332d19466fba1dc991d42bcd09bcd9f1c22a562646ffce0922793b6c69938b076e5cd6cfb3c361fc767e5f40ce05486e1668825ffeecab89d7daa455a179736a387ae93b9b15d283d45ffa14cd4af7");
    }
    #[test] fn sign_verify_round_trip() {
        let mut rng = rand::thread_rng(); let pp = BLS::setup(&mut rng).unwrap();
        let (pk, sk) = BLS::keygen(&pp, &mut rng).unwrap();
        let sig = BLS::sign(&pp, &sk, b"hello", &mut rng).unwrap();
        assert!(BLS::verify(&pp, &pk, b"hello", &sig).unwrap());
        assert!(!BLS::verify(&pp, &pk, b"hellp", &sig).unwrap());
        assert!(BLS::verify(&pp, &PublicKey::default(), b"hello", &sig).is_err());        // src/bls.rs:434-436
        assert!(BLS::sign(&pp, &PrivateKey::default(), b"hello", &mut rng).is_err());     // src/bls.rs:417-419
    }
}
