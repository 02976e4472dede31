"""Batched ZIP215 verification (ed25519_verify_zip215_batched / _dev) on the B200.  Its output must equal per-signature ZIP215
(ed25519_verify_policy_batch(..., VERIFY_ZIP215)) on every row: the fixture and generated rows of tests/verify_policy_model.py,
through the host API (ragged) and the device API, in a batch of several passes, under a bit-flip fuzz, on the full-length
scalar path and, where two GPUs exist, sharded.  Under EDDSA_B200_DEBUG_NO_FALLBACK=1 the raw batch equation is visible:
a group with an invalid included row (among them a pair of rows whose errors cancel under unit weights) zeroes its rows."""
import os
import subprocess
import sys

import numpy as np
import pytest

import verify_policy_model as vm

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
L = 2 ** 252 + 27742317777372353535851937790883648493
SEED = bytes(range(100, 132))


@pytest.fixture(scope="module")
def model():
    rows, want, cls = vm.all_rows()
    sig, pub, blob, off = vm.as_arrays(rows)
    return want[:, vm.ZIP215], sig, pub, blob, off


def _bad(got, want):
    return np.nonzero(np.asarray(got) != np.asarray(want))[0][:10]


@pytest.mark.parametrize("seed", [SEED, None], ids=["seed", "getrandom"])
def test_every_row_host_api(ed, model, seed):
    want, sig, pub, blob, off = model
    got = ed.ed25519_verify_zip215_batched(sig, pub, blob, off, 0, seed)
    assert not len(_bad(got, want)), _bad(got, want)


def test_every_row_device_api(ed, model):
    """Non-default stream; the flags land at an odd address between guard bytes."""
    import torch
    want, sig, pub, blob, off = model
    n = len(sig)
    dev = torch.device("cuda", 0)
    d_sig, d_pub = torch.from_numpy(sig).to(dev), torch.from_numpy(pub).to(dev)
    d_blob = torch.from_numpy(np.concatenate([blob, np.zeros(16, np.uint8)])).to(dev)
    d_off = torch.from_numpy(off.astype(np.int64)).to(dev)
    ok = torch.full((n + 2 * 17,), 0xA5, dtype=torch.uint8, device=dev)
    s = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(s):
        ed.ed25519_verify_zip215_batched_dev(ok[17:17 + n], d_sig, d_pub, d_blob, d_off, 0, SEED)
    s.synchronize()
    out = ok.cpu().numpy()
    assert (out[:17] == 0xA5).all() and (out[17 + n:] == 0xA5).all(), "guard bytes overwritten"
    assert not len(_bad(out[17:17 + n], want)), _bad(out[17:17 + n], want)


def test_bad_seed_length_is_refused(ed, model):
    want, sig, pub, blob, off = model
    with pytest.raises(ValueError):
        ed.ed25519_verify_zip215_batched(sig[:4], pub[:4], blob, off[:5], 0, b"short")


def _honest(ed, n, seed, mlen=64):
    rng = np.random.default_rng(seed)
    sec = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    msgs = rng.integers(0, 256, (n, mlen), dtype=np.uint8)
    pub = ed.ed25519_genpub_batch(sec)
    sig = ed.ed25519_sign_batch(sec, pub, msgs, fixed_len=mlen)
    return sig, pub, msgs


def _set_s(sig, i, s):
    sig[i, 32:] = np.frombuffer(int(s).to_bytes(32, "little"), np.uint8)


def _s(sig, i):
    return int.from_bytes(sig[i, 32:].tobytes(), "little")


@pytest.mark.slow
@pytest.mark.parametrize("seed", [SEED, None], ids=["seed", "getrandom"])
def test_several_passes_mixed_with_adversarial_rows(ed, model, seed):
    """2 x the verify pass + 77 signatures from ed25519_sign_batch, with every model row scattered among them (fixed length
    messages: the model rows' messages are padded into a second, ragged call over the same rows)."""
    want, msig, mpub, mblob, moff = model
    npass = 148 * 4 * 128 * 16
    n = 2 * npass + 77
    base = 1 << 16
    sig, pub, msgs = _honest(ed, base, 11)
    rep = (n + base - 1) // base
    sig, pub, msgs = (np.tile(x, (rep, 1))[:n].copy() for x in (sig, pub, msgs))
    rng = np.random.default_rng(5)
    pos = rng.choice(n, len(msig), replace=False)
    sig[pos], pub[pos] = msig, mpub
    lens = np.full(n, 64, np.int64)
    lens[pos] = np.diff(moff)
    off = np.zeros(n + 1, np.int64)
    off[1:] = np.cumsum(lens)
    blob = np.zeros(int(off[-1]), np.uint8)
    starts = off[:-1]
    honest = np.ones(n, bool)
    honest[pos] = False
    idx = np.nonzero(honest)[0]
    blob[(starts[idx][:, None] + np.arange(64)).ravel()] = msgs[idx].ravel()
    for k, p in enumerate(pos):
        blob[off[p]:off[p + 1]] = mblob[moff[k]:moff[k + 1]]
    ref = ed.ed25519_verify_policy_batch(sig, pub, blob, off, 0, ed.VERIFY_ZIP215)
    assert (ref[pos] == want).all() and ref[idx].all()
    got = ed.ed25519_verify_zip215_batched(sig, pub, blob, off, 0, seed)
    assert not len(_bad(got, ref)), _bad(got, ref)


def test_bitflip_fuzz(ed):
    """One random bit of the signature, key or message flipped in 3 of 4 rows: equal to ZIP215 on every row."""
    n = 20000
    sig, pub, msgs = _honest(ed, n, 21)
    rng = np.random.default_rng(22)
    for i in np.nonzero(rng.random(n) < 0.75)[0]:
        which = rng.integers(0, 3)
        arr = (sig, pub, msgs)[which]
        b = rng.integers(0, arr.shape[1] * 8)
        arr[i, b // 8] ^= 1 << (b % 8)
    ref = ed.ed25519_verify_policy_batch(sig, pub, msgs, None, 64, ed.VERIFY_ZIP215)
    for seed in (SEED, None):
        got = ed.ed25519_verify_zip215_batched(sig, pub, msgs, None, 64, seed)
        assert not len(_bad(got, ref)), _bad(got, ref)


_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, {root!r})
import libeddsa_b200 as ed
d = np.load({npz!r})
ok = ed.ed25519_verify_zip215_batched(d["sig"], d["pub"], d["msgs"], None, 64, {seed!r})
ref = ed.ed25519_verify_policy_batch(d["sig"], d["pub"], d["msgs"], None, 64, ed.VERIFY_ZIP215)
np.savez({out!r}, ok=ok, ref=ref)
"""


def _child(tmp_path, env, sig, pub, msgs, seed=SEED):
    npz, out = str(tmp_path / "in.npz"), str(tmp_path / "out.npz")
    np.savez(npz, sig=sig, pub=pub, msgs=msgs)
    e = dict(os.environ, **env)
    subprocess.run([sys.executable, "-c", _CHILD.format(root=ROOT, npz=npz, out=out, seed=seed)], env=e, check=True, timeout=600)
    r = np.load(out)
    return r["ok"], r["ref"]


def _crafted(ed, K):
    """Groups of K rows (warp w, lane l: rows 32 K w + l + 32 r) with: honest rows only; one corrupted message; an excluded
    row (S + L, S >= L) among honest ones; a cancelling pair (S_1 + 1, S_2 - 1 in one group: the errors B and -B cancel
    with unit weights); and a short last group.  Returns sig, pub, msgs and the expected raw lane decision per row."""
    n = 32 * K * 3 + 45
    sig, pub, msgs = _honest(ed, n, 31)
    group = (np.arange(n) // (32 * K)) * 32 + np.arange(n) % 32
    lane_fails = np.zeros(group.max() + 1, bool)
    zip_ok = np.ones(n, bool)
    # group of row 1: corrupted message (included, invalid)
    msgs[1, 0] ^= 1; zip_ok[1] = False; lane_fails[group[1]] = True
    # group of row 2: S >= L (excluded: its group still holds)
    _set_s(sig, 2, _s(sig, 2) + L); zip_ok[2] = False
    # cancelling pair in the group of row 3 (rows 3 and 3 + 32)
    _set_s(sig, 3, _s(sig, 3) + 1); _set_s(sig, 3 + 32, _s(sig, 3 + 32) - 1)
    zip_ok[[3, 35]] = False; lane_fails[group[3]] = True
    # a corrupted row in the short last group
    last = n - 3
    msgs[last, 5] ^= 0x40; zip_ok[last] = False; lane_fails[group[last]] = True
    raw = zip_ok & ~lane_fails[group]
    return sig, pub, msgs, raw, zip_ok


def test_no_fallback_shows_the_raw_equation(ed, tmp_path):
    """EDDSA_B200_DEBUG_NO_FALLBACK=1: a group whose equation fails zeroes its rows, the others keep the ZIP215 decision;
    the cancelling pair fails under the real weights."""
    sig, pub, msgs, raw, zip_ok = _crafted(ed, ed.VERIFY_BATCH_ROWS)
    ok, ref = _child(tmp_path, {"EDDSA_B200_DEBUG_NO_FALLBACK": "1"}, sig, pub, msgs)
    assert (ref.astype(bool) == zip_ok).all()
    assert not len(_bad(ok.astype(bool), raw)), _bad(ok.astype(bool), raw)
    ok2 = ed.ed25519_verify_zip215_batched(sig, pub, msgs, None, 64, SEED)      # with the fallback: exact ZIP215
    assert (ok2.astype(bool) == zip_ok).all()


def test_full_scalars_fallback(ed, tmp_path, model):
    """EDDSA_B200_DEBUG_FULL_SCALARS=1: the re-checked rows take the full-length scalar path; still equal to ZIP215."""
    sig, pub, msgs, raw, zip_ok = _crafted(ed, ed.VERIFY_BATCH_ROWS)
    ok, ref = _child(tmp_path, {"EDDSA_B200_DEBUG_FULL_SCALARS": "1"}, sig, pub, msgs)
    assert (ref.astype(bool) == zip_ok).all() and (ok == ref).all()


def test_sharded_over_two_gpus(ed, model):
    """A host-API call large enough to be split over two devices equals ZIP215."""
    if ed.device_count() < 2:
        pytest.skip("one GPU")
    want, sig, pub, blob, off = model
    n = 40000
    hs, hp, hm = _honest(ed, n, 41)
    hm[::97, 0] ^= 1
    ref = ed.ed25519_verify_policy_batch(hs, hp, hm, None, 64, ed.VERIFY_ZIP215)
    got = ed.ed25519_verify_zip215_batched(hs, hp, hm, None, 64, SEED)
    assert (got == ref).all() and int(ref.sum()) == n - len(range(0, n, 97))
