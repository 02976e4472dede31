"""Big-integer model of batched ZIP215 verification (ed25519_verify_zip215_batched): the weights and the batch equation one
GPU lane checks over its rows, and generators of lane layouts that exercise each case.

A row is included when ZIP215's encoding rules pass (S < L, A and R decode); its weight is
    z = SHA-512(seed || t || S)[0..16) as a little-endian integer, bit 0 set,   t = SHA-512(R || A || M) mod L,
and a lane's equation over its included rows is
    8 ( (sum z S mod L) B + sum (z t mod L) (-A) + sum z (-R) ) == O.
Within a verify pass, lane l of warp w holds rows 32 K w + l + 32 r, r < K (K = EDDSA_B200_VERIFY_BATCH_ROWS)."""
import hashlib

import edmodel as em
import verify_policy_model as vm

L = em.L
K = 8


def included(sig, pub):
    """ZIP215's encoding rules: S < L and both points decode (any encoding)."""
    A, _ = vm.decode(pub)
    R, _ = vm.decode(sig[:32])
    return A is not None and R is not None and int.from_bytes(bytes(sig[32:]), "little") < L


def weight(seed, sig, pub, msg):
    t = em.h_mod_l(bytes(sig[:32]), bytes(pub), bytes(msg))
    h = hashlib.sha512(bytes(seed) + t.to_bytes(32, "little") + bytes(sig[32:])).digest()
    return int.from_bytes(h[:16], "little") | 1


def lane_holds(rows, seed=None, unit_weights=False):
    """The batch equation over rows [(sig, pub, msg), ...]; excluded rows take no part."""
    acc, s_sum = vm.O, 0
    for sig, pub, msg in rows:
        if not included(sig, pub):
            continue
        A, _ = vm.decode(pub)
        R, _ = vm.decode(sig[:32])
        z = 1 if unit_weights else weight(seed, sig, pub, msg)
        t = em.h_mod_l(bytes(sig[:32]), bytes(pub), bytes(msg))
        s = int.from_bytes(bytes(sig[32:]), "little")
        s_sum = (s_sum + z * s) % L
        acc = vm.padd(acc, vm.pmul(z * t % L, vm.ext(em.neg(A))))
        acc = vm.padd(acc, vm.pmul(z, vm.ext(em.neg(R))))
    acc = vm.padd(acc, vm.pmul(s_sum, vm.ext(em.B)))
    return vm.is_identity(vm.pmul(8, acc))


def all_valid(rows):
    """What the equation must decide: every included row is ZIP215-valid."""
    return all(vm.decisions(s, p, m)[vm.ZIP215] for s, p, m in rows if included(s, p))


def cancelling_pair(sig1, pub1, msg1, sig2, pub2, msg2, delta=1):
    """Two invalid rows whose errors cancel under unit weights: S_1 + delta and S_2 - delta (both stay below L)."""
    s1 = int.from_bytes(bytes(sig1[32:]), "little") + delta
    s2 = int.from_bytes(bytes(sig2[32:]), "little") - delta
    assert 0 <= s1 < L and 0 <= s2 < L
    return (bytes(sig1[:32]) + s1.to_bytes(32, "little"), pub1, msg1), (bytes(sig2[:32]) + s2.to_bytes(32, "little"), pub2, msg2)


def layouts(rows, decisions):
    """Lanes of at most K rows from rows [(sig, pub, msg, cls)] with their (n, 3) decisions: honest lanes, lanes of
    ZIP215-only rows (valid under ZIP215, rejected under REFERENCE: torsion-shifted or non-canonical R need the cofactor),
    lanes with one invalid row, lanes with excluded rows among valid ones, a short lane, and a cancelling pair."""
    valid = [r[:3] for r, d in zip(rows, decisions) if d[vm.ZIP215]]
    zip_only = [r[:3] for r, d in zip(rows, decisions) if d[vm.ZIP215] and not d[vm.REFERENCE]]
    invalid = [r[:3] for r, d in zip(rows, decisions) if not d[vm.ZIP215] and included(r[0], r[1])]
    excluded = [r[:3] for r in rows if not included(r[0], r[1])]
    lanes = [valid[:K], valid[K:2 * K], zip_only[:K], zip_only[K:2 * K]]
    for i in range(3):
        lanes.append(valid[2 * K + i * (K - 1): 2 * K + (i + 1) * (K - 1)] + [invalid[i]])
        lanes.append(zip_only[i:i + K - 2] + excluded[2 * i:2 * i + 2])
    lanes.append(valid[:3])                                  # short last group
    lanes.append(list(cancelling_pair(*valid[0], *valid[1])) + valid[2:K])
    return [lane for lane in lanes if lane]
