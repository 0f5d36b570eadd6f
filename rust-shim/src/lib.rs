//! Safe wrappers over `libb200zk.so` for a halo2_proofs fork (tag v2023_02_02), plus what the golden-vector dumper
//! needs: the ConstraintSystem -> blob serialiser and an rng wrapper that records every byte the prover draws.
//! Source only — see rust-shim/README.md.  Call sites in the reference: `/root/reference/src/circuits/utils.rs:28-63`.
pub mod dump;
pub mod sys;

use halo2_proofs::halo2curves::bn256::{Fr, G1Affine, G2Affine, G1};
use halo2_proofs::halo2curves::group::Curve;
use halo2_proofs::plonk::{Any, ConstraintSystem, Expression};
use rand_core::{CryptoRng, RngCore};
use std::ffi::CStr;
use std::os::raw::c_void;
use std::sync::OnceLock;

/// One context per process and device (`B200ZK_DEVICE`, default 0).  A ctx is used by one caller thread at a time:
/// halo2's prover calls best_multiexp / best_fft sequentially from one thread, rayon never wraps a commit.
pub struct Ctx(pub *mut sys::Ctx);
unsafe impl Send for Ctx {}
unsafe impl Sync for Ctx {}

pub fn ctx() -> *mut sys::Ctx {
    static CTX: OnceLock<Ctx> = OnceLock::new();
    CTX.get_or_init(|| {
        let dev: i32 = std::env::var("B200ZK_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
        let mut p = std::ptr::null_mut();
        let rc = unsafe { sys::b200zk_ctx_create(dev, &mut p) };
        assert_eq!(rc, sys::B200ZK_OK, "b200zk_ctx_create({dev}) failed: {rc} (no sm_100 device? there is no CPU fallback)");
        Ctx(p)
    })
    .0
}

/// A non-zero status becomes the panic the upstream function would have raised.
pub fn check(rc: i32) {
    if rc != sys::B200ZK_OK {
        let msg = unsafe { CStr::from_ptr(sys::b200zk_last_error(ctx())) }.to_string_lossy().into_owned();
        panic!("b200zk error {rc}: {msg}");
    }
}

/// arithmetic::best_multiexp for bn256 (coeffs: &[Fr], bases: &[G1Affine]) -> G1
pub fn best_multiexp(coeffs: &[Fr], bases: &[G1Affine]) -> G1 {
    assert_eq!(coeffs.len(), bases.len());
    let mut out = G1::default();
    check(unsafe { sys::b200zk_msm(ctx(), coeffs.as_ptr() as *const c_void, bases.as_ptr() as *const c_void, coeffs.len(), &mut out as *mut G1 as *mut c_void) });
    out
}

/// arithmetic::best_fft for G = Fr
pub fn best_fft(a: &mut [Fr], omega: Fr, log_n: u32) {
    assert_eq!(a.len(), 1usize << log_n);
    check(unsafe { sys::b200zk_fft(ctx(), a.as_mut_ptr() as *mut c_void, &omega as *const Fr as *const c_void, log_n) });
}

/// arithmetic::g_to_lagrange(g, k) for bn256: the Lagrange basis of 2^k G1Affine points
pub fn g_to_lagrange(g: &[G1Affine], k: u32) -> Vec<G1Affine> {
    assert_eq!(g.len(), 1usize << k);
    let mut out = vec![G1Affine::default(); g.len()];
    check(unsafe { sys::b200zk_g_to_lagrange(ctx(), g.as_ptr() as *const c_void, k, out.as_mut_ptr() as *mut c_void) });
    out
}

/// ParamsKZG with the SRS resident on the device.
pub struct Params(pub *mut sys::Params, pub u32);
impl Params {
    /// ParamsKZG::setup: `s = Fr::random(rng)` stays on the Rust side, the 2n bases are generated on the device.
    pub fn setup(k: u32, s: &Fr) -> Self {
        let mut p = std::ptr::null_mut();
        check(unsafe { sys::b200zk_params_setup(ctx(), k, s as *const Fr as *const c_void, &mut p) });
        Params(p, k)
    }
    pub fn load(k: u32, g: &[G1Affine], g_lagrange: &[G1Affine]) -> Self {
        assert_eq!(g.len(), 1usize << k);
        assert_eq!(g_lagrange.len(), 1usize << k);
        let mut p = std::ptr::null_mut();
        check(unsafe { sys::b200zk_params_load(ctx(), k, g.as_ptr() as *const c_void, g_lagrange.as_ptr() as *const c_void, &mut p) });
        Params(p, k)
    }
    /// ParamsKZG::downsize(k) as new params (g[..2^k] and its Lagrange basis); `self` and the proving keys built on
    /// it stay valid, where upstream truncates in place.
    pub fn downsize(&self, k: u32) -> Self {
        assert!(k <= self.1);
        let mut p = std::ptr::null_mut();
        check(unsafe { sys::b200zk_params_downsize(self.0, k, &mut p) });
        Params(p, k)
    }
    pub fn commit(&self, poly: &[Fr]) -> G1 {
        let mut out = G1::default();
        check(unsafe { sys::b200zk_commit(self.0, poly.as_ptr() as *const c_void, poly.len(), &mut out as *mut G1 as *mut c_void) });
        out
    }
    pub fn commit_lagrange(&self, poly: &[Fr]) -> G1 {
        let mut out = G1::default();
        check(unsafe { sys::b200zk_commit_lagrange(self.0, poly.as_ptr() as *const c_void, poly.len(), &mut out as *mut G1 as *mut c_void) });
        out
    }
    pub fn get_g(&self) -> (Vec<G1Affine>, Vec<G1Affine>) {
        let n = 1usize << self.1;
        let (mut g, mut gl) = (vec![G1Affine::default(); n], vec![G1Affine::default(); n]);
        check(unsafe { sys::b200zk_params_read(self.0, g.as_mut_ptr() as *mut c_void, gl.as_mut_ptr() as *mut c_void) });
        (g, gl)
    }
}
impl Drop for Params {
    fn drop(&mut self) {
        unsafe { sys::b200zk_params_destroy(self.0) }
    }
}

/// The proving key resident on the device (keygen_pk) and create_proof on it.
pub struct Pk(pub *mut sys::Pk);
impl Pk {
    /// `fixed`: pk.fixed_values (selectors compressed), `map_col` / `map_row`: permutation::keygen::Assembly::mapping (P x n)
    pub fn create(params: &Params, cs: &ConstraintSystem<Fr>, fixed: &[Vec<Fr>], map_col: &[u32], map_row: &[u32]) -> Self {
        let blob = cs_blob(cs, params.1);
        let cols: Vec<*const c_void> = fixed.iter().map(|c| c.as_ptr() as *const c_void).collect();
        let mut p = std::ptr::null_mut();
        check(unsafe { sys::b200zk_pk_create(params.0, blob.as_ptr(), blob.len(), cols.as_ptr(), map_col.as_ptr(), map_row.as_ptr(), &mut p) });
        Pk(p)
    }
    pub fn rng_draws(&self) -> usize {
        unsafe { sys::b200zk_pk_rng_draws(self.0) }
    }
    /// plonk::create_proof for one circuit: `advice` = the witness columns after batch_invert_assigned (unblinded),
    /// `rng_wide` = 64 bytes per Fr::random call in call order (rng.fill_bytes of 64 * rng_draws()), returns the bytes
    /// `transcript.finalize()` would.  Err(()) = Error::ConstraintSystemFailure / InstanceTooLarge upstream.
    pub fn create_proof(&self, advice: &[Vec<Fr>], instances: &[&[Fr]], rng_wide: &[u8], transcript_repr: &Fr) -> Result<Vec<u8>, ()> {
        assert!(rng_wide.len() >= 64 * self.rng_draws());
        let adv: Vec<*const c_void> = advice.iter().map(|c| c.as_ptr() as *const c_void).collect();
        let inst: Vec<*const c_void> = instances.iter().map(|c| c.as_ptr() as *const c_void).collect();
        let lens: Vec<u32> = instances.iter().map(|c| c.len() as u32).collect();
        let mut proof = vec![0u8; unsafe { sys::b200zk_pk_proof_size(self.0) }];
        let mut len = 0usize;
        let rc = unsafe {
            sys::b200zk_create_proof(self.0, adv.as_ptr(), inst.as_ptr(), lens.as_ptr(), rng_wide.as_ptr() as *const c_void,
                                     transcript_repr as *const Fr as *const c_void, proof.as_mut_ptr(), proof.len(), &mut len)
        };
        if rc == sys::B200ZK_ESYNTH {
            return Err(());
        }
        check(rc);
        proof.truncate(len);
        Ok(proof)
    }
    /// Extension (upstream has no such call): create_proof for several witnesses of this key at once, run side by side
    /// on lanes of its device (b200zk_create_proofs).  Entry i is exactly `create_proof(&advice[i], &instances[i],
    /// &rng_wide[i], transcript_repr)`: Err(()) where that witness hits ConstraintSystemFailure / InstanceTooLarge.
    pub fn create_proofs(&self, advice: &[Vec<Vec<Fr>>], instances: &[Vec<&[Fr]>], rng_wide: &[Vec<u8>], transcript_repr: &Fr) -> Vec<Result<Vec<u8>, ()>> {
        let count = advice.len();
        assert!(instances.len() == count && rng_wide.len() == count);
        assert!(rng_wide.iter().all(|w| w.len() >= 64 * self.rng_draws()));
        let adv: Vec<*const c_void> = advice.iter().flat_map(|a| a.iter().map(|c| c.as_ptr() as *const c_void)).collect();
        let inst: Vec<*const c_void> = instances.iter().flat_map(|i| i.iter().map(|c| c.as_ptr() as *const c_void)).collect();
        let lens: Vec<u32> = instances.iter().flat_map(|i| i.iter().map(|c| c.len() as u32)).collect();
        let rng: Vec<*const c_void> = rng_wide.iter().map(|w| w.as_ptr() as *const c_void).collect();
        let size = unsafe { sys::b200zk_pk_proof_size(self.0) };
        let mut proofs = vec![0u8; size * count];
        let mut status = vec![0i32; count];
        let rc = unsafe {
            sys::b200zk_create_proofs(self.0, count as u32, adv.as_ptr(), inst.as_ptr(), lens.as_ptr(), rng.as_ptr(),
                                      transcript_repr as *const Fr as *const c_void, proofs.as_mut_ptr(), proofs.len(), status.as_mut_ptr())
        };
        if rc != sys::B200ZK_ESYNTH {
            check(rc);
        }
        status.iter().enumerate().map(|(i, &s)| if s == 0 { Ok(proofs[i * size..(i + 1) * size].to_vec()) } else { Err(()) }).collect()
    }
}
impl Drop for Pk {
    fn drop(&mut self) {
        unsafe { sys::b200zk_pk_destroy(self.0) }
    }
}

/// Extension in the sense of `Pk::create_proofs`: plonk::verify_proof for many proofs of one verifying key with
/// AccumulatorStrategy (src/poly/kzg/strategy.rs), one pairing check for the batch (b200zk_verify_proofs).  `fixed` /
/// `sigma`: the vk's commitments; `g` = params.get_g()[0]; `g2` / `s_g2` = params.g2() / s_g2().  One Fr::random draw
/// per proof comes from OsRng, as `process` makes it; they must stay secret.  Entry i is verify_proof's verdict on
/// proof i, the pairing included.
pub fn verify_proofs(cs: &ConstraintSystem<Fr>, k: u32, fixed: &[G1Affine], sigma: &[G1Affine], g: &G1Affine, g2: &G2Affine,
                     s_g2: &G2Affine, instances: &[Vec<&[Fr]>], proofs: &[&[u8]], transcript_repr: &Fr) -> Vec<bool> {
    let count = proofs.len();
    assert_eq!(instances.len(), count);
    let blob = cs_blob(cs, k);
    let inst: Vec<*const c_void> = instances.iter().flat_map(|i| i.iter().map(|c| c.as_ptr() as *const c_void)).collect();
    let lens: Vec<u32> = instances.iter().flat_map(|i| i.iter().map(|c| c.len() as u32)).collect();
    let ptrs: Vec<*const u8> = proofs.iter().map(|p| p.as_ptr()).collect();
    let plens: Vec<usize> = proofs.iter().map(|p| p.len()).collect();
    let mut rng_wide = vec![0u8; 64 * count];
    rand_core::OsRng.fill_bytes(&mut rng_wide);
    let mut status = vec![0i32; count];
    let rc = unsafe {
        sys::b200zk_verify_proofs(ctx(), blob.as_ptr(), blob.len(), fixed.as_ptr() as *const c_void, sigma.as_ptr() as *const c_void,
                                  g as *const G1Affine as *const c_void, g2 as *const G2Affine as *const c_void,
                                  s_g2 as *const G2Affine as *const c_void, count as u32, inst.as_ptr(), lens.as_ptr(),
                                  transcript_repr as *const Fr as *const c_void, ptrs.as_ptr(), plens.as_ptr(),
                                  rng_wide.as_ptr() as *const c_void, status.as_mut_ptr(), std::ptr::null_mut())
    };
    if rc != sys::B200ZK_EVERIFY {
        check(rc);
    }
    status.iter().map(|&s| s == 0).collect()
}

/// Many `multi_miller_loop(..).final_exponentiation() == Gt::identity()` checks on the device in one call
/// (b200zk_pairing_checks): check j multiplies the m pairs `pairs[j * m .. (j + 1) * m]`.  One verdict per check.
pub fn pairing_checks(pairs: &[(G1Affine, G2Affine)], m: usize) -> Vec<bool> {
    assert!(m > 0 && !pairs.is_empty() && pairs.len() % m == 0);
    let g1: Vec<G1Affine> = pairs.iter().map(|p| p.0).collect();
    let g2: Vec<G2Affine> = pairs.iter().map(|p| p.1).collect();
    let mut status = vec![0i32; pairs.len() / m];
    let rc = unsafe {
        sys::b200zk_pairing_checks(ctx(), g1.as_ptr() as *const c_void, g2.as_ptr() as *const c_void, m as u32, status.len() as u32,
                                   status.as_mut_ptr())
    };
    if rc != sys::B200ZK_EVERIFY {
        check(rc);
    }
    status.iter().map(|&s| s == 0).collect()
}


// ---------------------------------------------------------------------------------------------------------------------
// ConstraintSystem -> the word format of halo2-experiments_b200/circuit.py::ConstraintSystem.to_blob (parsed by
// csrc/cs_desc.hpp::parse_cs).  Call it on the constraint system AFTER compress_selectors (vk.cs()).
const OP_CONST: u32 = 0;
const OP_FIXED: u32 = 1;
const OP_ADVICE: u32 = 2;
const OP_INSTANCE: u32 = 3;
const OP_NEG: u32 = 4;
const OP_ADD: u32 = 5;
const OP_MUL: u32 = 6;
const OP_SCALE: u32 = 7;

struct Emit {
    consts: Vec<Fr>,
    prog: Vec<u32>,
}
impl Emit {
    fn const_idx(&mut self, c: Fr) -> u32 {
        if let Some(i) = self.consts.iter().position(|x| *x == c) {
            return i as u32;
        }
        self.consts.push(c);
        (self.consts.len() - 1) as u32
    }
    /// postfix, children before the operator, left operand first (same order as circuit.py::emit)
    fn expr(&mut self, e: &Expression<Fr>) {
        match e {
            Expression::Constant(c) => {
                let i = self.const_idx(*c);
                self.prog.push(OP_CONST | (i << 8));
            }
            Expression::Selector(_) => panic!("selectors must be compressed into fixed columns before serialisation"),
            Expression::Fixed(q) => self.prog.push(OP_FIXED | ((q.index() as u32) << 8)),
            Expression::Advice(q) => self.prog.push(OP_ADVICE | ((q.index() as u32) << 8)),
            Expression::Instance(q) => self.prog.push(OP_INSTANCE | ((q.index() as u32) << 8)),
            Expression::Challenge(_) => panic!("multi-phase circuits are not supported by b200zk_create_proof"),
            Expression::Negated(a) => {
                self.expr(a);
                self.prog.push(OP_NEG);
            }
            Expression::Sum(a, b) => {
                self.expr(a);
                self.expr(b);
                self.prog.push(OP_ADD);
            }
            Expression::Product(a, b) => {
                self.expr(a);
                self.expr(b);
                self.prog.push(OP_MUL);
            }
            Expression::Scaled(a, c) => {
                self.expr(a);
                let i = self.const_idx(*c);
                self.prog.push(OP_SCALE | (i << 8));
            }
        }
    }
    fn range(&mut self, e: &Expression<Fr>) -> (u32, u32) {
        let off = self.prog.len() as u32;
        self.expr(e);
        (off, self.prog.len() as u32 - off)
    }
}

pub fn cs_blob(cs: &ConstraintSystem<Fr>, k: u32) -> Vec<u32> {
    let mut em = Emit { consts: vec![], prog: vec![] };
    let gates: Vec<(u32, u32)> = cs.gates().iter().flat_map(|g| g.polynomials().iter()).map(|p| em.range(p)).collect();
    let lookups: Vec<(Vec<(u32, u32)>, Vec<(u32, u32)>)> = cs
        .lookups()
        .iter()
        .map(|l| (l.input_expressions().iter().map(|e| em.range(e)).collect(), l.table_expressions().iter().map(|e| em.range(e)).collect()))
        .collect();
    let perm: Vec<(u32, u32)> = cs
        .permutation()
        .get_columns()
        .iter()
        .map(|c| (match c.column_type() { Any::Advice(_) => 0u32, Any::Fixed => 1, Any::Instance => 2 }, c.index() as u32))
        .collect();
    let mut w: Vec<u32> = vec![
        0x324B5A42, 1, k, cs.num_advice_columns() as u32, cs.num_fixed_columns() as u32, cs.num_instance_columns() as u32,
        cs.advice_queries().len() as u32, cs.fixed_queries().len() as u32, cs.instance_queries().len() as u32,
        gates.len() as u32, lookups.len() as u32, perm.len() as u32, em.consts.len() as u32, em.prog.len() as u32,
        cs.blinding_factors() as u32, cs.degree() as u32,
    ];
    for (c, r) in cs.advice_queries() { w.push(c.index() as u32); w.push(r.0 as u32); }
    for (c, r) in cs.fixed_queries() { w.push(c.index() as u32); w.push(r.0 as u32); }
    for (c, r) in cs.instance_queries() { w.push(c.index() as u32); w.push(r.0 as u32); }
    for (t, c) in &perm { w.push(*t); w.push(*c); }
    for (o, l) in &gates { w.push(*o); w.push(*l); }
    for (ins, tabs) in &lookups {
        w.push(ins.len() as u32);
        for (o, l) in ins.iter().chain(tabs.iter()) { w.push(*o); w.push(*l); }
    }
    for c in &em.consts {
        // canonical little-endian value, eight u32 words
        let repr = halo2_proofs::halo2curves::ff::PrimeField::to_repr(c);
        for chunk in repr.as_ref().chunks(4) { w.push(u32::from_le_bytes([chunk[0], chunk[1], chunk[2], chunk[3]])); }
    }
    w.extend_from_slice(&em.prog);
    w
}

// ---------------------------------------------------------------------------------------------------------------------
/// Wraps the prover's rng and keeps every byte it hands out: `Fr::random` consumes 64 bytes per call in halo2curves
/// (`from_bytes_wide` of `fill_bytes`, or 8 x `next_u64`: the same 64 bytes of a XorShiftRng), so the recorded stream is
/// exactly `rng_wide` of b200zk_create_proof.
pub struct RecordingRng<R: RngCore> {
    pub inner: R,
    pub bytes: Vec<u8>,
}
impl<R: RngCore> RecordingRng<R> {
    pub fn new(inner: R) -> Self {
        Self { inner, bytes: vec![] }
    }
}
impl<R: RngCore> RngCore for RecordingRng<R> {
    fn next_u32(&mut self) -> u32 {
        let v = self.inner.next_u32();
        self.bytes.extend_from_slice(&v.to_le_bytes());
        v
    }
    fn next_u64(&mut self) -> u64 {
        let v = self.inner.next_u64();
        self.bytes.extend_from_slice(&v.to_le_bytes());
        v
    }
    fn fill_bytes(&mut self, dest: &mut [u8]) {
        self.inner.fill_bytes(dest);
        self.bytes.extend_from_slice(dest);
    }
    fn try_fill_bytes(&mut self, dest: &mut [u8]) -> Result<(), rand_core::Error> {
        self.fill_bytes(dest);
        Ok(())
    }
}
impl<R: RngCore> CryptoRng for RecordingRng<R> {}

/// G1 -> affine for `transcript.write_point`, as `commit(..).to_affine()` upstream
pub fn to_affine(p: &G1) -> G1Affine {
    p.to_affine()
}
