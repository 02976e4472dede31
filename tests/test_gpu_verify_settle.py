"""Every pending-carry settle of the verify window loops on the B200 (tests/golden/verify_settle.bin; see
tests/test_verify_settle.py for what the corpus holds).

Per-signature rows: every row is accepted under REFERENCE, STRICT and ZIP215 and by ed25519_verify_batch, through the host
API and the device API (non-default stream, flags at an odd offset).  Each row is replicated to fill two warps, and every
row needs exactly 33 windows, so every warp of k_verify runs the 33 windows the probe ran and each row takes its sites.

Batched lanes: each corpus lane is placed where lane l of warp w of k_verify_batched reads its rows (32 K w + l + 32 r), and
the device API runs one device with the committed seed, so each lane computes the equation the probe ran.  Under
EDDSA_B200_DEBUG_NO_FALLBACK=1 (a fresh interpreter) every equation must hold; with the fallback the output must equal
per-signature ZIP215."""
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_verify_settle as corpus_file  # noqa: E402

pytestmark = pytest.mark.gpu
MLEN = 32
REPEAT = 64              # copies of each row: two warps


def _arrays(rows):
    return tuple(np.array([np.frombuffer(r[k], np.uint8) for r in rows]) for k in range(3))


@pytest.fixture(scope="module")
def corpus():
    return corpus_file.load()


@pytest.fixture(scope="module")
def replicated(corpus):
    rows = corpus[0]
    return tuple(np.repeat(a, REPEAT, axis=0) for a in _arrays(rows))


def _bad(got):
    return np.nonzero(np.asarray(got) != 1)[0][:10]


def test_rows_host_api(ed, replicated):
    sig, pub, msg = replicated
    for name, got in [("ed25519_verify_batch", ed.ed25519_verify_batch(sig, pub, msg, None, MLEN))] + [
            (f"policy {p}", ed.ed25519_verify_policy_batch(sig, pub, msg, None, MLEN, p))
            for p in (ed.VERIFY_REFERENCE, ed.VERIFY_STRICT, ed.VERIFY_ZIP215)]:
        assert not len(_bad(got)), (name, _bad(got) // REPEAT)


def test_rows_device_api(ed, replicated):
    import torch
    sig, pub, msg = replicated
    n = len(sig)
    dev = torch.device("cuda", 0)
    d_sig, d_pub, d_msg = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (sig, pub, msg))
    s = torch.cuda.Stream(device=dev)
    calls = [("ed25519_verify_batch_dev", lambda ok: ed.ed25519_verify_batch_dev(ok, d_sig, d_pub, d_msg, None, MLEN))] + [
        (f"policy {p}", lambda ok, p=p: ed.ed25519_verify_policy_batch_dev(ok, d_sig, d_pub, d_msg, None, MLEN, p))
        for p in (ed.VERIFY_REFERENCE, ed.VERIFY_STRICT, ed.VERIFY_ZIP215)]
    for name, call in calls:
        ok = torch.full((n + 2 * 17,), 0xA5, dtype=torch.uint8, device=dev)
        with torch.cuda.stream(s):
            call(ok[17:17 + n])
        s.synchronize()
        out = ok.cpu().numpy()
        assert (out[:17] == 0xA5).all() and (out[17 + n:] == 0xA5).all(), (name, "guard bytes overwritten")
        assert not len(_bad(out[17:17 + n])), (name, _bad(out[17:17 + n]) // REPEAT)


def lane_layout(corpus, K):
    """Rows (sig, pub, msg) of whole warps in which lane l of warp w holds corpus lane (32 w + l) mod #lanes, at rows
    32 K w + l + 32 r; the returned map gives the corpus lane of each GPU lane."""
    _, pool, lanes, _ = corpus
    warps = (len(lanes) + 31) // 32
    psig, ppub, pmsg = _arrays(pool)
    idx = np.zeros(32 * K * warps, np.int64)
    which = []
    for w in range(warps):
        for lane in range(32):
            q = (32 * w + lane) % len(lanes)
            which.append(q)
            for r, k in enumerate(lanes[q][3]):
                idx[32 * K * w + lane + 32 * r] = k
    return psig[idx], ppub[idx], pmsg[idx], which


_CHILD = r"""
import sys, numpy as np, torch
sys.path.insert(0, {root!r})
import libeddsa_b200 as ed
d = np.load({npz!r})
dev = torch.device("cuda", 0)
sig, pub, msg = (torch.from_numpy(d[k]).to(dev) for k in ("sig", "pub", "msg"))
ok = torch.zeros(len(d["sig"]), dtype=torch.uint8, device=dev)
ed.ed25519_verify_zip215_batched_dev(ok, sig, pub, msg, None, {mlen}, bytes(d["seed"]))
torch.cuda.synchronize()
np.save({out!r}, ok.cpu().numpy())
"""


def _child(tmp_path, env, sig, pub, msg, seed):
    npz, out = str(tmp_path / "in.npz"), str(tmp_path / "out.npy")
    np.savez(npz, sig=sig, pub=pub, msg=msg, seed=np.frombuffer(seed, np.uint8))
    e = {k: v for k, v in os.environ.items() if not k.startswith("EDDSA_B200_DEBUG_")}
    e.update(env)
    subprocess.run([sys.executable, "-c", _CHILD.format(root=ROOT, npz=npz, out=out, mlen=MLEN)], env=e, check=True, timeout=600)
    return np.load(out)


def test_batched_lanes_raw_equations(ed, corpus, tmp_path):
    sig, pub, msg, which = lane_layout(corpus, ed.VERIFY_BATCH_ROWS)
    seed = corpus[3]
    raw = _child(tmp_path, {"EDDSA_B200_DEBUG_NO_FALLBACK": "1"}, sig, pub, msg, seed)
    bad = _bad(raw)
    assert not len(bad), ("corpus lanes whose equation failed", sorted({which[(i // (32 * ed.VERIFY_BATCH_ROWS)) * 32 + i % 32] for i in bad}))
    got = _child(tmp_path, {}, sig, pub, msg, seed)
    ref = ed.ed25519_verify_policy_batch(sig, pub, msg, None, MLEN, ed.VERIFY_ZIP215)
    assert ref.all() and (got == ref).all()
