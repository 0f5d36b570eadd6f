// halo2_proofs/src/arithmetic.rs (tag v2023_02_02) — bodies that replace the CPU implementations.
// The generic signatures stay; the bn256 instantiation (the only one the KZG prover of the reference reaches,
// /root/reference/src/circuits/utils.rs:40-48) goes to the device, anything else keeps the CPU path.
use b200zk_shim as gpu;
use std::any::TypeId;

pub fn best_multiexp<C: CurveAffine>(coeffs: &[C::Scalar], bases: &[C]) -> C::Curve {
    assert_eq!(coeffs.len(), bases.len());                                   // upstream's own assertion
    if TypeId::of::<C>() == TypeId::of::<halo2curves::bn256::G1Affine>() {
        // Fr / G1Affine / G1 are plain limb arrays: reinterpret the slices, no copy
        let coeffs = unsafe { &*(coeffs as *const [C::Scalar] as *const [halo2curves::bn256::Fr]) };
        let bases = unsafe { &*(bases as *const [C] as *const [halo2curves::bn256::G1Affine]) };
        let out = gpu::best_multiexp(coeffs, bases);
        return unsafe { std::mem::transmute_copy::<halo2curves::bn256::G1, C::Curve>(&out) };
    }
    best_multiexp_cpu(coeffs, bases)                                         // the original body, renamed
}

pub fn best_fft<G: Group>(a: &mut [G], omega: G::Scalar, log_n: u32) {
    assert_eq!(a.len(), 1 << log_n);
    if TypeId::of::<G>() == TypeId::of::<halo2curves::bn256::Fr>() {
        let a = unsafe { &mut *(a as *mut [G] as *mut [halo2curves::bn256::Fr]) };
        let omega = unsafe { std::mem::transmute_copy::<G::Scalar, halo2curves::bn256::Fr>(&omega) };
        return gpu::best_fft(a, omega, log_n);
    }
    best_fft_cpu(a, omega, log_n)
}

// g_to_lagrange (ParamsKZG::downsize): the G1 NTT and the n^-1 scaling on the device, normalised there as well
pub fn g_to_lagrange<C: CurveAffine>(g_projective: Vec<C::Curve>, k: u32) -> Vec<C> {
    if TypeId::of::<C>() == TypeId::of::<halo2curves::bn256::G1Affine>() {
        let mut g = vec![C::identity(); g_projective.len()];
        C::Curve::batch_normalize(&g_projective, &mut g);
        let g = unsafe { &*(g.as_slice() as *const [C] as *const [halo2curves::bn256::G1Affine]) };
        return gpu::g_to_lagrange(g, k).into_iter().map(|p| unsafe { std::mem::transmute_copy::<halo2curves::bn256::G1Affine, C>(&p) }).collect();
    }
    g_to_lagrange_cpu(g_projective, k)
}
