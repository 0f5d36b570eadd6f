// halo2_proofs/src/poly/kzg/commitment.rs (tag v2023_02_02) — ParamsKZG<Bn256> keeps `g`, `g_lagrange` lazily (read back
// with b200zk_params_read only if a caller asks for get_g()), plus a device handle `dev: b200zk_shim::Params` and
// `retired: Vec<b200zk_shim::Params>` (device params replaced by downsize, kept for the proving keys built on them).
impl ParamsKZG<Bn256> {
    pub fn setup<R: RngCore>(k: u32, rng: R) -> Self {
        assert!(k <= Fr::S);
        let s = Fr::random(rng);                                   // the only randomness of setup (64 bytes of the rng)
        let dev = b200zk_shim::Params::setup(k, &s);               // g[i] = [s^i]G, g_lagrange[i] = [l_i(s)]G on the device
        let g2 = <Bn256 as Engine>::G2Affine::generator();
        let s_g2 = (g2 * s).into();                                // two G2 operations stay on the CPU
        Self { k, n: 1 << k, dev, retired: Vec::new(), g2, s_g2, g: OnceCell::new(), g_lagrange: OnceCell::new() }
    }
    /// Keeps g[..2^k] and rebuilds g_lagrange with g_to_lagrange, both on the device.  The device params are replaced
    /// by new ones; the old ones stay alive in `retired`, because device proving keys built before the call use them.
    pub fn downsize(&mut self, k: u32) {
        assert!(k <= self.k);
        let small = self.dev.downsize(k);
        self.retired.push(std::mem::replace(&mut self.dev, small));
        self.k = k;
        self.n = 1 << k;
        self.g = OnceCell::new();
        self.g_lagrange = OnceCell::new();
    }
}
impl<'params> Params<'params, G1Affine> for ParamsKZG<Bn256> {
    fn commit_lagrange(&self, poly: &Polynomial<Fr, LagrangeCoeff>, _: Blind<Fr>) -> G1 {
        self.dev.commit_lagrange(&poly.values)                     // best_multiexp(poly, g_lagrange[..len]) on resident bases
    }
}
impl<'params> ParamsProver<'params, G1Affine> for ParamsKZG<Bn256> {
    fn commit(&self, poly: &Polynomial<Fr, Coeff>, _: Blind<Fr>) -> G1 {
        self.dev.commit(&poly.values)
    }
}
// ParamsKZG::write / read: b200zk_params_serialize / b200zk_params_deserialize produce and consume the same byte layout
// (k u32 LE | g | g_lagrange compressed | g2 | s_g2) with the 2n points (de)compressed on the device.
