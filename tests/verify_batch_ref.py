"""Reference restatement of what a batch verifier accumulates (test infrastructure, next to oracle/prover.py's
verify_full, which it reuses up to the SHPLONK opening):

    shplonk_dual(...)     VerifierSHPLONK's DualMSM of one proof: (left, right) = (h2, u*h2 + L / z_0) as integer affine
                          points (None = identity), where L = sum_i v^i z_i sum_j y^j (C_ij - [r_ij(u)] G) - Z_T(u) h1
    accumulate(duals, rs) AccumulatorStrategy::process in order (src/poly/kzg/strategy.rs): acc = r_i * acc + D_i
    wide_to_fr(w)         Fr::from_bytes_wide of one 64-byte draw

A proof is accepted when e(left, [s]_2) = e(right, [1]_2), i.e. s * left == right with the SRS secret s."""
from oracle import prover as OP
from oracle import pyref as P

R = OP.R


def shplonk_dual(pk, instances, proof, transcript_repr, fixed_commitments=None, params_g=None):
    """The (left, right) pair of one proof.  The fixed / permutation commitments are taken from pk when it is a
    verifying_key(), else committed from its polynomials over params_g (as verify_full does)."""
    cs, dom = pk.cs, pk.dom
    Q, st = OP.verify_proof(None, pk, instances, proof, transcript_repr)
    x, rd = st["x"], st["rd"]
    have_vk = hasattr(pk, "fixed_commitments")
    fixed_c = {}
    for (col, rot), e in zip(cs.fixed_queries, st["fixed_evals"]):
        if col not in fixed_c:
            fixed_c[col] = pk.fixed_commitments[col] if have_vk else OP.commit(params_g, pk.fixed_polys[col])
        Q.append((("fix", col), fixed_c[col], OP.rotate_omega(dom, x, rot), e))
    for j, e in enumerate(st["sigma_evals"]):
        Q.append((("sig", j), pk.sigma_commitments[j] if have_vk else OP.commit(params_g, pk.perm_polys[j]), x, e))
    Q.append((("h",), st["h_commit"], x, st["expected_h"]))
    Q.append((("rand",), st["random_c"], x, st["random_eval"]))
    y, v = rd.squeeze(), rd.squeeze()
    h1 = rd.read_point()
    u = rd.squeeze()
    h2 = rd.read_point()
    comm_sets, super_points = [], set()
    for cid, c, pt, e in Q:
        super_points.add(pt)
        for entry in comm_sets:
            if entry[0] == cid:
                entry[2][pt] = e
                break
        else:
            comm_sets.append([cid, c, {pt: e}])
    rot_sets = []
    for cid, c, pe in comm_sets:
        fs = frozenset(pe)
        for entry in rot_sets:
            if entry[0] == fs:
                entry[1].append((c, pe))
                break
        else:
            rot_sets.append((fs, [(c, pe)]))
    super_points = sorted(super_points)

    def vanish(roots):
        acc = 1
        for r in roots:
            acc = acc * (u - r) % R
        return acc

    Lpt, v_pow, z0 = None, 1, None
    for fs, items in rot_sets:
        points = sorted(fs)
        z_i = vanish([p for p in super_points if p not in points])
        z0 = z_i if z0 is None else z0
        y_pow = 1
        for c, pe in items:
            low = OP.lagrange_interpolate(points, [pe[p] for p in points])
            r_eval = sum(cf * pow(u, i, R) for i, cf in enumerate(low)) % R
            t = P.g1_add(c, P.g1_mul(P.G1_GEN, (-r_eval) % R))
            Lpt = P.g1_add(Lpt, P.g1_mul(t, y_pow * z_i % R * v_pow % R) if t is not None else None)
            y_pow = y_pow * y % R
        v_pow = v_pow * v % R
    Lpt = P.g1_add(Lpt, P.g1_mul(h1, (-vanish(super_points)) % R) if h1 is not None else None)
    Lpt = P.g1_mul(Lpt, pow(z0, -1, R)) if Lpt is not None else None
    right = P.g1_add(P.g1_mul(h2, u) if h2 is not None else None, Lpt)
    return h2, right


def _scale(pt, k):
    return P.g1_mul(pt, k) if pt is not None else None


def accumulate(duals, rs):
    """process(proof_i) for i in order: acc <- r_i * acc + D_i.  A dual of (None, None) stands for a proof that adds
    nothing (it still scales what came before by its r_i)."""
    left = right = None
    for (l, r), k in zip(duals, rs):
        left = P.g1_add(_scale(left, k), l)
        right = P.g1_add(_scale(right, k), r)
    return left, right


def wide_to_fr(w):
    """Fr::from_bytes_wide of one draw given as 8 little-endian u64 words (or 64 bytes)."""
    b = bytes(w) if isinstance(w, (bytes, bytearray)) else w.astype("<u8").tobytes()
    return int.from_bytes(b, "little") % R
