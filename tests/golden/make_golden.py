#!/usr/bin/env python3
"""Extract the reference's own fixtures for the module-lattice hot path into
small committed files under tests/golden/.

Needs a checkout of cloudflare/circl; the tests read only the files written here:
       python tests/golden/make_golden.py <path to the circl checkout>

Nothing here executes reference code (it is Go; there is no Go toolchain).  It
only re-packages the reference's test DATA:
  * NIST ACVP vectors   kem/mlkem/testdata/*, sign/mldsa/testdata/*   (internal/test/acvp.go:15-87)
  * sampler vectors embedded as Go literals in *_test.go files
  * PQCgenKAT SHA-256 digests (kem/kyber/kat_test.go:25-33, sign/dilithium/kat_test.go:25-35)
  * Keccak ShortMsgKATs (internal/sha3/testdata/keccakKats.json.deflate), subsampled
  * Wycheproof ML-DSA vectors (sign/schemes/testdata/wycheproof)
"""
import gzip
import json
import lzma
import os
import re
import sys
import zlib

REF = None  # the circl checkout, set from the command line
OUT = os.path.dirname(os.path.abspath(__file__))


def jgz(path):
    return json.load(gzip.open(os.path.join(REF, path)))


def acvp(sub_dir):
    prompt = jgz(f"{sub_dir}/prompt.json.gz")
    exp = jgz(f"{sub_dir}/expectedResults.json.gz")
    results = {}
    for g in exp["testGroups"]:
        for t in g["tests"]:
            results[t["tcId"]] = t
    return prompt, results


def dump(name, obj):
    raw = json.dumps(obj, separators=(",", ":"), sort_keys=True).encode()
    path = os.path.join(OUT, name)
    if name.endswith(".xz"):  # for the fixtures gzip would leave above 1 MB
        with open(path, "wb") as f:
            f.write(lzma.compress(raw, preset=9 | lzma.PRESET_EXTREME))
    else:
        with gzip.GzipFile(path, "wb", mtime=0) as f:
            f.write(raw)
    print(f"{name}: {os.path.getsize(path)} bytes")


def mlkem():
    out = {"source": "kem/mlkem/testdata (NIST ACVP FIPS 203)", "encap": {}, "decap": {}, "keygen": {}}
    prompt, res = acvp("kem/mlkem/testdata/ML-KEM-encapDecap-FIPS203")
    for g in prompt["testGroups"]:
        ps = g["parameterSet"]
        if g["function"] == "encapsulation":
            out["encap"][ps] = [
                {"tcId": t["tcId"], "ek": t["ek"], "m": t["m"], "c": res[t["tcId"]]["c"], "k": res[t["tcId"]]["k"]}
                for t in g["tests"]
            ]
        else:
            out["decap"][ps] = {
                "dk": g["dk"],
                "tests": [{"tcId": t["tcId"], "c": t["c"], "k": res[t["tcId"]]["k"]} for t in g["tests"]],
            }
    prompt, res = acvp("kem/mlkem/testdata/ML-KEM-keyGen-FIPS203")
    for g in prompt["testGroups"]:
        out["keygen"][g["parameterSet"]] = [
            {"tcId": t["tcId"], "d": t["d"], "z": t["z"], "ek": res[t["tcId"]]["ek"], "dk": res[t["tcId"]]["dk"]}
            for t in g["tests"]
        ]
    dump("mlkem_acvp.json.gz", out)


def mldsa65():
    ps = "ML-DSA-65"
    out = {"source": "sign/mldsa/testdata (NIST ACVP FIPS 204), ML-DSA-65 groups only", "siggen": [], "sigver": {}, "keygen": []}
    prompt, res = acvp("sign/mldsa/testdata/ML-DSA-sigGen-FIPS204")
    for g in prompt["testGroups"]:
        if g["parameterSet"] != ps:
            continue
        for t in g["tests"]:
            out["siggen"].append({
                "tcId": t["tcId"], "deterministic": g["deterministic"], "sk": t["sk"], "message": t["message"],
                "rnd": t.get("rnd", "00" * 32), "signature": res[t["tcId"]]["signature"],
            })
    prompt, res = acvp("sign/mldsa/testdata/ML-DSA-sigVer-FIPS204")
    for g in prompt["testGroups"]:
        if g["parameterSet"] != ps:
            continue
        out["sigver"] = {
            "pk": g["pk"],
            "tests": [{"tcId": t["tcId"], "message": t["message"], "signature": t["signature"],
                       "testPassed": res[t["tcId"]]["testPassed"]} for t in g["tests"]],
        }
    prompt, res = acvp("sign/mldsa/testdata/ML-DSA-keyGen-FIPS204")
    for g in prompt["testGroups"]:
        if g["parameterSet"] != ps:
            continue
        out["keygen"] = [{"tcId": t["tcId"], "seed": t["seed"], "pk": res[t["tcId"]]["pk"], "sk": res[t["tcId"]]["sk"]}
                         for t in g["tests"]]
    dump("mldsa65_acvp.json.gz", out)


def mldsa_other():
    """ML-DSA-44 and ML-DSA-87: every vector of their groups in the same ACVP files."""
    out = {"source": "sign/mldsa/testdata (NIST ACVP FIPS 204), ML-DSA-44 / ML-DSA-87, all vectors of their groups"}
    for ps in ("ML-DSA-44", "ML-DSA-87"):
        o = {"siggen": [], "sigver": {}, "keygen": []}
        prompt, res = acvp("sign/mldsa/testdata/ML-DSA-sigGen-FIPS204")
        for g in prompt["testGroups"]:
            if g["parameterSet"] != ps:
                continue
            for t in g["tests"]:
                o["siggen"].append({"tcId": t["tcId"], "deterministic": g["deterministic"], "sk": t["sk"],
                                    "message": t["message"], "rnd": t.get("rnd", "00" * 32),
                                    "signature": res[t["tcId"]]["signature"]})
        prompt, res = acvp("sign/mldsa/testdata/ML-DSA-sigVer-FIPS204")
        for g in prompt["testGroups"]:
            if g["parameterSet"] != ps:
                continue
            tests = g["tests"]
            o["sigver"] = {"pk": g["pk"], "tests": [{"tcId": t["tcId"], "message": t["message"], "signature": t["signature"],
                                                     "testPassed": res[t["tcId"]]["testPassed"]} for t in tests]}
        prompt, res = acvp("sign/mldsa/testdata/ML-DSA-keyGen-FIPS204")
        for g in prompt["testGroups"]:
            if g["parameterSet"] != ps:
                continue
            o["keygen"] = [{"tcId": t["tcId"], "seed": t["seed"], "pk": res[t["tcId"]]["pk"], "sk": res[t["tcId"]]["sk"]}
                           for t in g["tests"]]
        out[ps] = o
    dump("mldsa_other_acvp.json.gz", out)


def go_array(path, func, var=None, which=0):
    """Pull the `which`-th `{...}` integer literal that follows `func <func>(` in a Go test file."""
    src = open(os.path.join(REF, path)).read()
    start = src.index(f"func {func}(")
    body = src[start:]
    nxt = body.find("\nfunc ", 1)
    if nxt > 0:
        body = body[:nxt]
    lits = re.findall(r"(?:Poly|\]uint32|\]int16|\]byte)\{([^{}]*)\}", body, flags=re.S)
    vals = [int(x, 0) for x in re.findall(r"-?(?:0x[0-9a-fA-F]+|\d+)", lits[which])]
    return vals


def samplers():
    out = {"note": "seed = bytes 0..31 in every vector"}
    f = "pke/kyber/internal/common/sample_test.go"
    out["kyber_noise3_nonce37"] = go_array(f, "TestPolyDeriveNoise3Ref")            # :23
    out["kyber_noise2_nonce37"] = go_array(f, "TestPolyDeriveNoise2Ref")            # :57
    out["kyber_uniform_x1_y0"] = go_array(f, "TestPolyDeriveUniformRef")            # :93
    out["dil_uniform_nonce30000"] = go_array("sign/mldsa/mldsa65/internal/sample_test.go", "TestVectorDeriveUniform")
    f = "sign/dilithium/mode3/internal/params_test.go"
    out["dil_leqeta4_nonce30000"] = go_array(f, "TestVectorDeriveUniformLeqEta")
    out["dil_legamma1_19_nonce30000"] = go_array(f, "TestVectorDeriveUniformLeGamma1")
    for k, v in out.items():
        if isinstance(v, list):
            assert len(v) == 256, (k, len(v))
    # zero-state permutation, simd/keccakf1600/f1600x_test.go:9-19
    src = open(os.path.join(REF, "simd/keccakf1600/f1600x_test.go")).read()
    m = re.search(r"permutationOfZeroes = \[.*?\]uint64\{(.*?)\}", src, flags=re.S)
    out["keccak_f1600_of_zero"] = [int(x, 16) for x in re.findall(r"0x[0-9A-Fa-f]+", m.group(1))]
    assert len(out["keccak_f1600_of_zero"]) == 25
    # lazy-Barrett schedule of the inverse NTT, pke/kyber/internal/common/ntt.go:38-50
    src = open(os.path.join(REF, "pke/kyber/internal/common/ntt.go")).read()
    m = re.search(r"InvNTTReductions = \[\.\.\.\]int\{(.*?)\n\}", src, flags=re.S)
    body = re.sub(r"//[^\n]*", "", m.group(1))
    out["kyber_invntt_reductions"] = [int(x) for x in re.findall(r"-?\d+", body)]
    out["kat_sha256"] = {  # kem/kyber/kat_test.go:25-33, sign/dilithium/kat_test.go:25-35
        "ML-KEM-512": re.search(r'"ML-KEM-512", "([0-9a-f]{64})"', open(os.path.join(REF, "kem/kyber/kat_test.go")).read()).group(1),
        "ML-KEM-768": re.search(r'"ML-KEM-768", "([0-9a-f]{64})"', open(os.path.join(REF, "kem/kyber/kat_test.go")).read()).group(1),
        "ML-KEM-1024": re.search(r'"ML-KEM-1024", "([0-9a-f]{64})"', open(os.path.join(REF, "kem/kyber/kat_test.go")).read()).group(1),
        "ML-DSA-65": re.search(r'"ML-DSA-65", "([0-9a-f]{64})"', open(os.path.join(REF, "sign/dilithium/kat_test.go")).read()).group(1),
        "Kyber512": re.search(r'"Kyber512", "([0-9a-f]{64})"', open(os.path.join(REF, "kem/kyber/kat_test.go")).read()).group(1),
        "Kyber768": re.search(r'"Kyber768", "([0-9a-f]{64})"', open(os.path.join(REF, "kem/kyber/kat_test.go")).read()).group(1),
        "Kyber1024": re.search(r'"Kyber1024", "([0-9a-f]{64})"', open(os.path.join(REF, "kem/kyber/kat_test.go")).read()).group(1),
        "ML-DSA-44": re.search(r'"ML-DSA-44", "([0-9a-f]{64})"', open(os.path.join(REF, "sign/dilithium/kat_test.go")).read()).group(1),
        "ML-DSA-87": re.search(r'"ML-DSA-87", "([0-9a-f]{64})"', open(os.path.join(REF, "sign/dilithium/kat_test.go")).read()).group(1),
        "Dilithium2": re.search(r'"Dilithium2", "([0-9a-f]{64})"', open(os.path.join(REF, "sign/dilithium/kat_test.go")).read()).group(1),
        "Dilithium3": re.search(r'"Dilithium3", "([0-9a-f]{64})"', open(os.path.join(REF, "sign/dilithium/kat_test.go")).read()).group(1),
        "Dilithium5": re.search(r'"Dilithium5", "([0-9a-f]{64})"', open(os.path.join(REF, "sign/dilithium/kat_test.go")).read()).group(1),
    }
    dump("sampler_vectors.json.gz", out)


def x25519_vectors():
    """dh/x25519/testdata (RFC 7748 section 5.2 and 6.1, Wycheproof) + the X-Wing draft vectors hash."""
    import gzip
    td = os.path.join(REF, "dh/x25519/testdata")
    out = {"source": "dh/x25519/testdata/{rfc7748_kat_test,rfc7748_times_test,wycheproof_kat}.json.gz; kem/xwing/xwing_test.go:78-80"}
    out["rfc7748_kat"] = json.load(gzip.open(os.path.join(td, "rfc7748_kat_test.json.gz")))
    out["rfc7748_times"] = [v for v in json.load(gzip.open(os.path.join(td, "rfc7748_times_test.json.gz"))) if v["times"] <= 1000]
    out["wycheproof"] = [{k: v[k] for k in ("tcId", "public", "private", "shared", "result")}
                         for v in json.load(gzip.open(os.path.join(td, "wycheproof_kat.json.gz")))]
    src = open(os.path.join(REF, "kem/xwing/xwing_test.go")).read()
    out["xwing_vectors_shake128"] = re.search(r'want := "([0-9a-f]{64})"', src).group(1)
    dump("x25519_vectors.json.gz", out)


def wycheproof():
    """sign/schemes/testdata/wycheproof/mldsa_{44,65,87}_*: the vectors sign/schemes/wycheproof_test.go replays
    (malformed keys and signatures, context strings, hint encodings, signatures that need many rejection rounds)."""
    td = "sign/schemes/testdata/wycheproof"
    out = {"source": td + " (all nine files, every group and test case; replayed as sign/schemes/wycheproof_test.go:40-150 does)"}
    for f in sorted(os.listdir(os.path.join(REF, td))):
        if not f.endswith(".json.gz"):
            continue
        ts = jgz(f"{td}/{f}")
        groups = []
        for g in ts["testGroups"]:
            o = {"type": g["type"], "tests": [{k: t.get(k) for k in ("tcId", "msg", "ctx", "sig", "result", "comment", "flags")}
                                              for t in g["tests"]]}
            for k in ("privateKey", "privateSeed", "publicKey"):
                if k in g:
                    o[k] = g[k]
            groups.append(o)
        out[f.replace(".json.gz", "")] = {"algorithm": ts["algorithm"], "groups": groups}
    dump("mldsa_wycheproof.json.xz", out)


def keccak_kats():
    raw = open(os.path.join(REF, "internal/sha3/testdata/keccakKats.json.deflate"), "rb").read()
    kats = json.loads(zlib.decompress(raw, -15))["kats"]
    out = {"source": "internal/sha3/testdata/keccakKats.json.deflate (byte-aligned messages, every 24th + all <= 64 bits)"}
    for alg in ("SHA3-256", "SHA3-512", "SHAKE128", "SHAKE256"):
        sel = []
        for i, k in enumerate(kats[alg]):
            if k["length"] % 8:
                continue
            if k["length"] <= 64 or i % 24 == 0 or k["length"] in (1080, 1088, 1096, 1336, 1344, 1352, 568, 576, 584):
                sel.append({"length": k["length"], "message": k["message"][: k["length"] // 4], "digest": k["digest"]})
        out[alg] = sel
    dump("keccak_kats.json.gz", out)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    REF = sys.argv[1]
    mlkem()
    mldsa65()
    mldsa_other()
    samplers()
    keccak_kats()
    x25519_vectors()
    wycheproof()
