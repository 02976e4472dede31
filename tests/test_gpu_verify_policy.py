"""The three acceptance rules of ed25519_verify_policy_batch / _dev on the B200 (REFERENCE, STRICT, ZIP215), against the
big-integer model of tests/verify_policy_model.py: every fixture row and every generated row under each rule, through the host
API, the device API and the ragged form, in a batch of several passes mixed among honest rows, under a bit-flip fuzz, on the
full-length scalar path and, where two GPUs exist, sharded."""
import os
import subprocess
import sys

import numpy as np
import pytest

import verify_policy_model as vm

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def model():
    rows, want, cls = vm.all_rows()
    sig, pub, blob, off = vm.as_arrays(rows)
    return rows, want, cls, sig, pub, blob, off


def _bad(got, want):
    return np.nonzero(np.asarray(got) != np.asarray(want))[0][:10]


@pytest.mark.parametrize("policy", vm.POLICIES, ids=[vm.NAMES[p] for p in vm.POLICIES])
def test_every_row_host_api(ed, model, policy):
    """Fixture and generated rows through the host API, ragged messages: the model's decision on every row."""
    rows, want, cls, sig, pub, blob, off = model
    got = ed.ed25519_verify_policy_batch(sig, pub, blob, off, 0, policy)
    assert not len(_bad(got, want[:, policy])), [(int(i), int(cls[i])) for i in _bad(got, want[:, policy])]
    if policy == vm.REFERENCE:
        assert (got == ed.ed25519_verify_batch(sig, pub, blob, off, 0)).all()


@pytest.mark.parametrize("policy", vm.POLICIES, ids=[vm.NAMES[p] for p in vm.POLICIES])
def test_every_row_device_api(ed, model, policy):
    """The same rows through the device API on a non-default stream; the flags land at an odd address between guard bytes."""
    import torch
    rows, want, cls, sig, pub, blob, off = model
    n = len(sig)
    dev = torch.device("cuda", 0)
    d_sig, d_pub = torch.from_numpy(sig).to(dev), torch.from_numpy(pub).to(dev)
    d_blob = torch.from_numpy(np.concatenate([blob, np.zeros(16, np.uint8)])).to(dev)
    d_off = torch.from_numpy(off.astype(np.int64)).to(dev)
    ok = torch.full((n + 2 * 17,), 0xA5, dtype=torch.uint8, device=dev)
    s = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(s):
        ed.ed25519_verify_policy_batch_dev(ok[17:17 + n], d_sig, d_pub, d_blob, d_off, 0, policy)
    s.synchronize()
    out = ok.cpu().numpy()
    assert (out[:17] == 0xA5).all() and (out[17 + n:] == 0xA5).all(), "guard bytes overwritten"
    got = out[17:17 + n]
    assert not len(_bad(got, want[:, policy])), [(int(i), int(cls[i])) for i in _bad(got, want[:, policy])]


def test_unknown_policy_is_refused(ed, model):
    rows, want, cls, sig, pub, blob, off = model
    for bad in (-1, 3):
        with pytest.raises(ed.EddsaB200Error):
            ed.ed25519_verify_policy_batch(sig[:4], pub[:4], blob, off[:5], 0, bad)
        with pytest.raises(ed.EddsaB200Error):
            ed.ed25519_verify_policy_batch(sig[:0], pub[:0], blob, off[:1], 0, bad)


def _honest(ed, n, seed, mlen=64):
    rng = np.random.default_rng(seed)
    sec = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    msgs = rng.integers(0, 256, (n, mlen), dtype=np.uint8)
    pub = ed.ed25519_genpub_batch(sec)
    sig = ed.ed25519_sign_batch(sec, pub, msgs, fixed_len=mlen)
    return sig, pub, msgs


@pytest.mark.slow
def test_several_passes_mixed_with_honest_rows(ed, model):
    """2 x the verify pass + 77 signatures (148 SMs x 4 blocks x 128 threads x 16 waves per pass): 2^18 honest signatures from
    ed25519_sign_batch, repeated, with every model row scattered among them; ragged messages; host and device API, every rule."""
    import torch
    rows, want, cls, sig_m, pub_m, blob_m, off_m = model
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 2 * sms * 4 * 128 * 16 + 77
    hs, hp, hm = _honest(ed, 1 << 18, 4242)
    for pol in vm.POLICIES:                                          # honest signatures: accepted by every rule
        assert ed.ed25519_verify_policy_batch(hs, hp, hm, None, 64, pol).all(), vm.NAMES[pol]
    rng = np.random.default_rng(99)
    pos = np.sort(rng.choice(n, size=len(rows), replace=False))
    src = np.arange(n) % (1 << 18)
    sig, pub = hs[src], hp[src]
    sig[pos], pub[pos] = sig_m, pub_m
    parts, prev = [], 0
    for k, i in enumerate(pos):
        parts += [hm[src[prev:i]].tobytes(), rows[k][2]]
        prev = i + 1
    parts.append(hm[src[prev:]].tobytes())
    lens = np.full(n, 64, np.int64)
    lens[pos] = [len(r[2]) for r in rows]
    off = np.zeros(n + 1, np.uint64)
    off[1:] = np.cumsum(lens)
    blob = np.frombuffer(b"".join(parts) + bytes(16), np.uint8)
    assert blob.size == int(off[-1]) + 16
    d_sig, d_pub = torch.from_numpy(sig).cuda(), torch.from_numpy(pub).cuda()
    d_blob, d_off = torch.from_numpy(blob).cuda(), torch.from_numpy(off.astype(np.int64)).cuda()
    for pol in vm.POLICIES:
        expect = np.ones(n, np.uint8)
        expect[pos] = want[:, pol]
        got = ed.ed25519_verify_policy_batch(sig, pub, blob, off, 0, pol)
        assert not len(_bad(got, expect)), (vm.NAMES[pol], _bad(got, expect))
        ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        ed.ed25519_verify_policy_batch_dev(ok, d_sig, d_pub, d_blob, d_off, 0, pol)
        torch.cuda.synchronize()
        assert not len(_bad(ok.cpu().numpy(), expect)), (vm.NAMES[pol], "device API")


def test_bit_flip_fuzz(ed, model):
    """Single bit flips in R, S, A or the message of honest, generated and fixture rows: every rule decides like the model."""
    rows, want, cls, *_ = model
    rng = np.random.default_rng(31337)
    hs, hp, hm = _honest(ed, 600, 7, 40)
    base = [(hs[i].tobytes(), hp[i].tobytes(), hm[i].tobytes(), 0) for i in range(len(hs))]
    base += [rows[i] for i in rng.choice(len(rows), size=900, replace=False)]
    fuzzed = []
    for s, p, m, c in base:
        s, p, m = bytearray(s), bytearray(p), bytearray(m)
        where = rng.integers(0, 4 if m else 3)
        if where == 0: s[rng.integers(0, 32)] ^= 1 << rng.integers(0, 8)
        elif where == 1: s[32 + rng.integers(0, 32)] ^= 1 << rng.integers(0, 8)
        elif where == 2: p[rng.integers(0, 32)] ^= 1 << rng.integers(0, 8)
        else: m[rng.integers(0, len(m))] ^= 1 << rng.integers(0, 8)
        fuzzed.append((bytes(s), bytes(p), bytes(m), c))
    rows2 = base + fuzzed
    exp = vm.decide_rows(rows2)
    sig, pub, blob, off = vm.as_arrays(rows2)
    for pol in vm.POLICIES:
        got = ed.ed25519_verify_policy_batch(sig, pub, blob, off, 0, pol)
        assert not len(_bad(got, exp[:, pol])), (vm.NAMES[pol], _bad(got, exp[:, pol]))


def test_full_length_scalars(model):
    """EDDSA_B200_DEBUG_FULL_SCALARS=1 (read at start-up, so in a fresh interpreter): every signature takes the (rho, tau) = (1, t)
    path, and every rule decides every row as before."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys, os, numpy as np; sys.path[:0] = [os.getcwd(), os.path.join(os.getcwd(), 'tests')]\n"
            "import libeddsa_b200 as ed, verify_policy_model as vm\n"
            "rows, want, cls = vm.all_rows(); sig, pub, blob, off = vm.as_arrays(rows)\n"
            "for pol in vm.POLICIES:\n"
            "    got = ed.ed25519_verify_policy_batch(sig, pub, blob, off, 0, pol)\n"
            "    assert (got == want[:, pol]).all(), (pol, np.nonzero(got != want[:, pol])[0][:10])\n"
            "print('full-scalar rules ok')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env=dict(os.environ, EDDSA_B200_DEBUG_FULL_SCALARS="1"),
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "full-scalar rules ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_sharded_over_two_gpus(ed, model):
    """A host-API call large enough to be split over two devices decides like the model under every rule."""
    if ed.device_count() < 2:
        pytest.skip("one GPU")
    rows, want, cls, sig, pub, blob, off = model
    reps = 5                                          # > 16 384 signatures: the batch is sharded
    sig5, pub5, blob5, off5 = vm.as_arrays(rows * reps)
    for pol in vm.POLICIES:
        got = ed.ed25519_verify_policy_batch(sig5, pub5, blob5, off5, 0, pol)
        assert not len(_bad(got, np.tile(want[:, pol], reps))), vm.NAMES[pol]
