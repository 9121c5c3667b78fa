"""Pins the oracle (oracle/ref_py) to the reference's own fixtures and KATs (tests/golden/,
extracted from a checkout of the reference by tests/golden/make_golden.py) and to OpenSSL / libsodium."""
import gzip
import hashlib
import json
import os

import pytest

from oracle.ref_py import curves
from oracle.ref_py.bn import RefError
from oracle.ref_py.ec import EC, KeyPair
from oracle.ref_py.eddsa import EDDSA

G = os.path.join(os.path.dirname(__file__), "golden")
KATS = json.load(open(os.path.join(G, "ecdsa_kats.json")))


def test_secp256k1_precomputed_tables_match_reference_file():
    """The oracle regenerates lib/elliptic/precomputed/secp256k1.js; digests must match."""
    ref = json.load(open(os.path.join(G, "secp256k1_precomputed.json")))
    pre = curves.get("secp256k1").g.precomputed
    dig = lambda ps: hashlib.sha256(b"".join(p.x.to_bytes(32, "big") + p.y.to_bytes(32, "big") for p in ps)).hexdigest()
    assert pre.doubles[0] == 4 and pre.naf[0] == 7
    assert dig(pre.doubles[1][1:]) == ref["doubles_sha256"]
    assert dig(pre.naf[1][1:]) == ref["naf_sha256"]
    assert ["%064x" % v for v in (pre.naf[1][-1].x, pre.naf[1][-1].y)] == ref["naf_last"]


def test_secp256k1_endomorphism_constants_and_split():
    """test/curve-test.js:154-167."""
    c = curves.get("secp256k1").curve
    assert "%x" % c.endo["beta"] == KATS["secp256k1_beta"]
    assert "%x" % c.endo["lambda"] == KATS["secp256k1_lambda"]
    k = 0x1234567890123456789012345678901234
    k1, k2 = c._endo_split(k)
    assert (k1 + k2 * c.endo["lambda"]) % c.n == k
    # lambda*G == (beta*x, y)
    lg = c.g.mul(c.endo["lambda"])
    assert (lg.x, lg.y) == (c.endo["beta"] * c.g.x % c.p, c.g.y)


def test_maxwell_trick_vectors():
    """test/ecdsa-test.js:352-451 (p256/p384 verify true/false incl. the r+n<p branch)."""
    for v in KATS["maxwell"]:
        ec = EC(v["curve"])
        assert ec.verify(v["msg"], v["sig"], v["pub"], "hex") is v["result"], v


def test_rfc6979_vectors_sign_and_verify():
    """test/ecdsa-test.js:135-350: exact r, s from sign(); pub validates; verify true."""
    from oracle.ref_py.curves import HASHES
    for blk in KATS["rfc6979"]:
        for case in blk["cases"]:
            ec = EC(blk["curve"], HASHES[case["hash"]])
            dgst = HASHES[case["hash"]](case["message"].encode()).digest()
            sig = ec.sign(dgst, int(blk["key"], 16))
            assert "%x" % sig.r == case["r"].lstrip("0") and "%x" % sig.s == case["s"].lstrip("0"), (blk["curve"], case)
            pub = {"x": blk["x"], "y": blk["y"]}
            assert ec.curve.validate(ec.key_from_public(pub).get_public())
            assert ec.verify(dgst, sig, pub) is True


def test_wycheproof_p192_truncation_forms():
    """test/ecdsa-test.js:492-534: hex string, byte array and BN + msgBitLength pin _truncateToN."""
    w = KATS["wycheproof_p192"]
    ec = EC("p192")
    assert ec.verify(w["msg"], w["sig"], w["pub"], "hex") is True
    assert ec.verify(bytes.fromhex(w["msg"]), w["sig"], w["pub"], "hex") is True
    assert ec.verify(int(w["msg"], 16), w["sig"], w["pub"], "hex", msg_bit_length=256) is True


def test_sec1_codec_kats():
    """test/curve-test.js:298-346."""
    c = curves.get("secp256k1").curve
    for v in KATS["sec1"]:
        for enc in ("compact", "encoded", "hybrid"):
            p = c.decode_point(v[enc], "hex")
            assert ("%064x" % p.x, "%064x" % p.y) == (v["x"], v["y"])
        p = c.point(int(v["x"], 16), int(v["y"], 16))
        assert p.encode(True).hex() == v["compact"] and p.encode().hex() == v["encoded"]
    with pytest.raises(RefError):
        c.decode_point("05" + KATS["sec1"][0]["x"], "hex")


def test_curve25519_ladder_kat_and_twist_rejection():
    """test/curve-test.js:348-356 and test/ecdh-test.js:31-43."""
    c = curves.get("curve25519")
    assert "%x" % c.g.mul(6).get_x() == KATS["curve25519_g_mul_6"]
    ec = EC("curve25519")
    k = KeyPair(ec, priv=0x1234567)
    with pytest.raises(RefError):
        k.derive(c.curve.point(14, 16))
    a, b = KeyPair(ec, priv=0x1111111111111111), KeyPair(ec, priv=0x2222222222222222222)
    assert a.derive(b.get_public()) == b.derive(a.get_public())


def test_ed25519_point_from_y_kat():
    """test/curve-test.js:90-112."""
    v = KATS["ed25519_point_from_y"]
    c = curves.get("ed25519").curve
    p = c.point_from_y(int.from_bytes(bytes(v["y_le_bytes"]), "little"), v["odd"])
    assert "%x" % p.get_x() == v["x"]


def _sign_input_chunk(vecs):
    import nacl.signing
    ed = EDDSA()
    for v in vecs:
        msg = bytes.fromhex(v["msg"])
        priv, _ = ed.priv_from_secret(v["secret"])
        assert ed.encode_point(ed.g.mul(priv)).hex() == v["pk"]
        assert ed.sign(msg, v["secret"]).hex() == v["sig"]
        assert ed.verify(msg, v["sig"], v["pk"]) is True
        forged = bytearray(msg) if msg else bytearray(b"x")
        forged[-1] = (forged[-1] + 1) & 0xFF
        assert ed.verify(bytes(forged), v["sig"], v["pk"]) is False
        nacl.signing.VerifyKey(bytes.fromhex(v["pk"])).verify(msg, bytes.fromhex(v["sig"]))
    return len(vecs)


def test_ed25519_sign_input_vectors():
    """test/ed25519-test.js:44-85 on all 1024 lines of test/fixtures/sign.input: public key, exact signature,
    verify true, forged message false; cross-check with libsodium.  (Worker processes: ~0.1 s per vector.)"""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import benchdata
    data = json.load(gzip.open(os.path.join(G, "ed25519_sign_input.json.gz"), "rt"))
    vecs = data["vectors"]
    assert len(vecs) == 1024
    done = benchdata._pmap(_sign_input_chunk, [vecs[i:i + 16] for i in range(0, len(vecs), 16)], min_items=2)
    assert sum(done) == 1024


def test_ed25519_derivation_fixtures():
    """test/ed25519-test.js:16-42 on all 256 entries of derivation-fixtures.js."""
    data = json.load(open(os.path.join(G, "ed25519_derivation.json")))
    ed = EDDSA()
    for v in data["vectors"][::4]:
        priv, _ = ed.priv_from_secret(v["secret_hex"])
        assert priv.to_bytes(32, "little").hex().upper() == v["a_hex"]
        A = ed.g.mul(priv)
        assert ed.encode_point(A).hex().upper() == v["A_hex"]
        # the fixture's A_P.x is encodeInt(x): little-endian bytes (test/ed25519-test.js:33-35)
        assert ed.decode_point(ed.encode_point(A)).get_x().to_bytes(32, "little").hex().upper() == v["x"]


def test_ed25519_invalid_encodings_throw_like_the_reference():
    """Non-residue -> bn.js sqrt assertion ('Assertion failed'); x = 0 with sign bit -> 'invalid point'."""
    ed = EDDSA()
    p = ed.curve.p
    bad = None
    for y in range(2, 200):
        u, v = (y * y - 1) % p, (ed.curve.d * y * y + 1) % p
        if pow(u * pow(v, -1, p) % p, (p - 1) // 2, p) == p - 1:
            bad = y
            break
    with pytest.raises(RefError, match="Assertion failed"):
        ed.decode_point(bad.to_bytes(32, "little"))
    one = bytearray((1).to_bytes(32, "little")); one[31] |= 0x80
    with pytest.raises(RefError, match="invalid point"):
        ed.decode_point(bytes(one))


def test_openssl_cross_check_short_curves():
    from cryptography.hazmat.primitives import hashes
    from cryptography.hazmat.primitives.asymmetric import ec as cec, utils as cutils
    import os as _os
    for name, cc, hh in (("secp256k1", cec.SECP256K1(), hashes.SHA256()), ("p256", cec.SECP256R1(), hashes.SHA256()),
                         ("p384", cec.SECP384R1(), hashes.SHA384())):
        e = EC(name)
        for _ in range(12):
            sk = cec.generate_private_key(cc)
            digest = _os.urandom(hh.digest_size)
            der = sk.sign(digest, cec.ECDSA(cutils.Prehashed(hh)))
            pn = sk.public_key().public_numbers()
            assert e.verify(digest, der, {"x": pn.x, "y": pn.y}) is True
            bad = bytearray(digest); bad[3] ^= 1
            assert e.verify(bytes(bad), der, {"x": pn.x, "y": pn.y}) is False
            s = e.sign(digest, sk.private_numbers().private_value)
            sk.public_key().verify(s.to_der(), digest, cec.ECDSA(cutils.Prehashed(hh)))


def test_op_counts_match_baseline_table():
    """BASELINE.md section 2: field multiplications per secp256k1 verify ~ 2216 (1225 M + 992 S)."""
    from oracle.ref_py import bn
    ec = EC("secp256k1")
    d = 0xC0FFEE
    Q = ec.g.mul(d)
    ec.verify(b"\x01" * 32, ec.sign(b"\x01" * 32, d), {"x": Q.x, "y": Q.y})   # warm G's beta table
    tot = 0
    for i in range(20):
        m = hashlib.sha256(b"%d" % i).digest()
        sig = ec.sign(m, d)
        bn.reset_count()
        assert ec.verify(m, sig, {"x": Q.x, "y": Q.y})
        c = bn.snapshot_count()
        assert c["I"] == 0
        tot += c["M"] + c["S"]
    assert 2100 < tot / 20 < 2350, tot / 20


def test_ed25519_reference_vectors_verify_from_hex():
    """Every 8th line of test/fixtures/sign.input (stored in tests/golden/ed25519_sign_input.json.gz), with message,
    signature and public key passed as the hex strings the fixture holds."""
    ed = EDDSA()
    data = json.load(gzip.open(os.path.join(G, "ed25519_sign_input.json.gz"), "rt"))
    assert data["total_lines"] == len(data["vectors"]) == 1024
    for v in data["vectors"][::8]:
        assert ed.verify(v["msg"], v["sig"], v["pk"]) is True


@pytest.mark.parametrize("name", ["p192", "p224", "p256", "p384", "p521", "secp256k1"])
def test_oracle_accepts_openssl_signatures_on_every_short_preset(name):
    """Independent pin for the presets without verify vectors in the reference: signatures made by OpenSSL
    (`cryptography`) over random digests verify under the oracle, and stop verifying when the digest changes."""
    import random
    from cryptography.hazmat.primitives.asymmetric import ec as cec, utils as cutils
    from cryptography.hazmat.primitives import hashes
    from oracle.ref_py.ec import EC
    curve = {"p192": cec.SECP192R1(), "p224": cec.SECP224R1(), "p256": cec.SECP256R1(), "p384": cec.SECP384R1(),
             "p521": cec.SECP521R1(), "secp256k1": cec.SECP256K1()}[name]
    ec = EC(name)
    rnd = random.Random(7)
    try:
        key = cec.generate_private_key(curve)
    except Exception as ex:                       # an OpenSSL build without the small curves
        pytest.skip(str(ex))
    pub = key.public_key().public_numbers()
    for _ in range(4):
        dg = rnd.randbytes(32)
        r, s = cutils.decode_dss_signature(key.sign(dg, cec.ECDSA(cutils.Prehashed(hashes.SHA256()))))
        # OpenSSL truncates the digest to the bit length of n exactly as _truncateToN does for a byte array
        assert ec.verify(dg, {"r": r, "s": s}, {"x": pub.x, "y": pub.y}) is True
        bad = bytearray(dg); bad[0] ^= 0x40
        assert ec.verify(bytes(bad), {"r": r, "s": s}, {"x": pub.x, "y": pub.y}) is False
