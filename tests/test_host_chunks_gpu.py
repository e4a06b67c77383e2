"""GPU: the host-buffer Ed448 entry points cut a device's shard into chunks that run on the device's three streams at
once, every stream with its own scratch slots (csrc/hostbatch.h: run_chunks; csrc/internal.h: scratch_get).  Batches
large enough to be chunked (>= 2^19 items) must give the bytes of the single-stream device-pointer pipelines -- which
the other tests pin to the oracle -- and the oracle's on a seeded sample; a bad point in a late chunk must still be
reported.

Matches KeyPair::new (ecc/keypair.rs:41-51), sign / verify (ecc/signable.rs:40-86), the ECDH core of key_encrypt
(ecc/encryptable.rs:36-38)."""
import numpy as np
import pytest
import torch

from capycrypt_b200 import _binding as B
from oracle import ref_ed448 as E

pytestmark = pytest.mark.gpu

N = (1 << 19) + (1 << 18) + 777  # three chunks, ragged last block


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def batch(engine):
    rnd = np.random.default_rng(77)
    pw = rnd.integers(0, 256, size=N * 16, dtype=np.uint8)
    po = np.arange(N + 1, dtype=np.uint64) * 16
    lens = rnd.integers(0, 200, size=N)
    mo = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    msg = rnd.integers(0, 256, size=int(mo[-1]), dtype=np.uint8)
    sc = rnd.integers(0, 256, size=N * 56, dtype=np.uint8)
    return dict(pw=pw, po=po, msg=msg, mo=mo, sc=sc, sample=np.sort(rnd.choice(N, size=96, replace=False)))


def test_chunked_host_pipelines_match_the_device_pipelines(engine, oracle, batch):
    pw, po, msg, mo, sc, pick = (batch[k] for k in ("pw", "po", "msg", "mo", "sc", "sample"))
    t_pw, t_po, t_msg, t_mo, t_sc = _dev(pw), _dev(po.astype(np.int64)), _dev(msg), _dev(mo.astype(np.int64)), _dev(sc)
    # fixed base
    pts = engine.ed448_fixed_base(sc)
    t_pts = torch.zeros(N * 112, dtype=torch.uint8, device="cuda")
    engine.ed448_fixed_base_dev(t_sc, N, t_pts)
    torch.cuda.synchronize()
    assert np.array_equal(pts.reshape(-1), t_pts.cpu().numpy())
    assert np.array_equal(pts[pick], oracle.fixed_base_batch(sc.reshape(N, 56)[pick].reshape(-1), threads=0))
    # keygen
    pub = engine.ed448_keygen(pw, po, 512)
    t_pub = torch.zeros(N * 112, dtype=torch.uint8, device="cuda")
    engine.ed448_keygen_dev(t_pw, t_po, 512, t_pub)
    torch.cuda.synchronize()
    assert np.array_equal(pub.reshape(-1), t_pub.cpu().numpy())
    # sign
    h, z = engine.ed448_sign(pw, po, msg, mo, 512)
    t_h, t_z = torch.zeros(N * 56, dtype=torch.uint8, device="cuda"), torch.zeros(N * 56, dtype=torch.uint8, device="cuda")
    engine.ed448_sign_dev(t_pw, t_po, t_msg, t_mo, 512, t_h, t_z)
    torch.cuda.synchronize()
    assert np.array_equal(h.reshape(-1), t_h.cpu().numpy()) and np.array_equal(z.reshape(-1), t_z.cpu().numpy())
    s_pw = pw.reshape(N, 16)[pick].reshape(-1)
    s_po = np.arange(len(pick) + 1, dtype=np.uint64) * 16
    s_msgs = [msg[int(mo[i]):int(mo[i + 1])] for i in pick]
    s_mo = np.concatenate([[0], np.cumsum([len(m) for m in s_msgs])]).astype(np.uint64)
    s_msg = np.concatenate(s_msgs) if s_mo[-1] else np.zeros(0, np.uint8)
    hw, zw = oracle.sign_batch(s_pw, s_po, s_msg, s_mo, 512, threads=0)
    assert np.array_equal(h[pick], hw) and np.array_equal(z[pick], zw)
    # verify: all good; then tampered items in the first, the middle and the last chunk
    rc, ok = engine.ed448_verify(pub, msg, mo, h, z, 512)
    assert rc == 0 and ok.all()
    h2 = h.copy()
    bad_items = [5, (1 << 18) + 9, N - 1]
    for i in bad_items:
        h2[i, 3] ^= 0x40
    rc, ok = engine.ed448_verify(pub, msg, mo, h2, z, 512)
    assert rc == 0 and int(ok.sum()) == N - len(bad_items) and not ok[bad_items].any()
    # an off-curve key in the LAST chunk: reported through the status, the item fails, the others do not
    pub2 = pub.copy()
    pub2[N - 3] = np.frombuffer(E.point_to_bytes((5, 7)), dtype=np.uint8)
    rc, ok = engine.ed448_verify(pub2, msg, mo, h, z, 512)
    assert rc == B.ERR_BAD_POINT and int(ok.sum()) == N - 1 and ok[N - 3] == 0


def test_chunked_var_base_and_ecdh(engine, oracle, batch):
    sc, pick = batch["sc"], batch["sample"]
    n = (1 << 19) + 333  # two chunks
    pts = engine.ed448_fixed_base(sc[: n * 56])
    k = np.roll(sc[: n * 56], 11)
    rc, out = engine.ed448_var_base(k, pts)
    assert rc == 0
    t_out = torch.zeros(n * 112, dtype=torch.uint8, device="cuda")
    engine.ed448_var_base_dev(_dev(k), _dev(pts.reshape(-1)), n, t_out)
    torch.cuda.synchronize()
    assert np.array_equal(out.reshape(-1), t_out.cpu().numpy())
    p = pick[pick < n][:32]
    rc_o, want = oracle.var_base_batch(k.reshape(n, 56)[p].reshape(-1), pts[p].reshape(-1), threads=0)
    assert rc_o == 0 and np.array_equal(out[p], want)
    rc, wx, Z = engine.ed448_ecdh(k, pts)
    assert rc == 0
    rc_o, wx_o = oracle.ecdh_batch(k.reshape(n, 56)[p].reshape(-1), pts[p].reshape(-1), threads=0)
    assert rc_o == 0 and np.array_equal(wx[p], wx_o)
    # Z = [4 k mod r]G: the same nonce scalars through the fixed-base entry point after the reference's scalar map
    # is covered by test_ecdh_agreement; here: a bad point in the second chunk surfaces, its row is zeroed
    pts2 = pts.copy()
    pts2[n - 2] = np.frombuffer(E.point_to_bytes((5, 7)), dtype=np.uint8)
    rc, out2 = engine.ed448_var_base(k, pts2)
    assert rc == B.ERR_BAD_POINT and not out2[n - 2].any()
    keep = np.ones(n, bool)
    keep[n - 2] = False
    assert np.array_equal(out2[keep], out[keep])
