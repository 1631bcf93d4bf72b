"""GPU tests of the layer between the caller's buffers and the kernels.

Host-pointer batches travel through HBM in chunks (`run_staged` in csrc/api.cu, the own pipelines of ML-DSA sign and
verify in csrc/mldsa.cu); device-pointer calls fork internal lanes off the caller's stream and join back.  The tests
here run that layer where it actually does something:

  1. batches of 4C + 1 and 6C + 13 operations (C = the entry point's chunk), so that staging slots are reused, the
     short ramp chunks run and a 13-row chunk sits between full ones, with the rows at every chunk edge checked;
  2. pinned host buffers (asynchronous copies) besides pageable ones, strided host rows, in-place and aliased buffers;
  3. ML-DSA sign / verify / keygen on device pointers;
  4. device-pointer calls queued behind a busy caller stream, whose outputs must be final when the stream passes the
     call and must not be touched afterwards.

The chunk sizes below mirror the sources; tests/test_batch_paths_table.py checks that they still do.
"""
from __future__ import annotations

import ctypes as C
import functools
import hashlib
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# ---------------------------------------------------------------- staging schedule of the host-pointer paths
SLOTS = {"staged": 4, "sign": 3, "verify": 1}  # Dev::kSlots; ML-DSA sign's own three slots; verify's one
# (entry point, source under circl_b200/csrc, function that sets the chunk, chunk, pipeline)
CHUNK_TABLE = [
    ("cb200_mlkem_encaps", "mlkem.cu", "mlkem_encaps_entry", 1 << 16, "staged"),
    ("cb200_mlkem_decaps", "mlkem.cu", "cb200_mlkem_decaps", 1 << 15, "staged"),
    ("cb200_mlkem_keygen", "mlkem.cu", "keygen_entry", 1 << 15, "staged"),
    ("cb200_kyber_kem_keygen", "mlkem.cu", "keygen_entry", 1 << 15, "staged"),
    ("cb200_kyber_kem_encaps", "mlkem.cu", "kyber_kem_run", 1 << 15, "staged"),
    ("cb200_kyber_kem_decaps", "mlkem.cu", "kyber_kem_run", 1 << 15, "staged"),
    ("cb200_kyber_derive_uniform", "mlkem.cu", "cb200_kyber_derive_uniform", 1 << 16, "staged"),
    ("cb200_xwing_keygen", "hybrid.cu", "cb200_xwing_keygen", 1 << 15, "staged"),
    ("cb200_xwing_encaps", "hybrid.cu", "cb200_xwing_encaps", 1 << 15, "staged"),
    ("cb200_xwing_decaps", "hybrid.cu", "cb200_xwing_decaps", 1 << 15, "staged"),
    ("cb200_hybrid_encaps", "hybrid.cu", "cb200_hybrid_encaps", 1 << 15, "staged"),
    ("cb200_hybrid_decaps", "hybrid.cu", "cb200_hybrid_decaps", 1 << 15, "staged"),
    ("cb200_x25519", "hybrid.cu", "cb200_x25519", 1 << 17, "staged"),
    ("cb200_kyber_ntt", "api.cu", "cb200_kyber_ntt", 1 << 17, "staged"),
    ("cb200_kyber_dot", "api.cu", "cb200_kyber_dot", 1 << 17, "staged"),  # divided by k
    ("cb200_kyber_poly_op", "api.cu", "cb200_kyber_poly_op", 1 << 17, "staged"),
    ("cb200_dil_ntt", "dil_kernels.cu", "cb200_dil_ntt", 1 << 16, "staged"),
    ("cb200_sha3", "keccak_api.cu", "cb200_sha3", 1 << 16, "staged"),
    ("cb200_dil_derive_uniform", "mldsa.cu", "sampler_entry", 1 << 15, "staged"),
    ("cb200_mldsa_sign", "mldsa.cu", "cb200_mldsa_sign", 1 << 16, "sign"),
    ("cb200_mldsa_verify", "mldsa.cu", "cb200_mldsa_verify", 1 << 15, "verify"),
    ("cb200_mldsa_keygen", "mldsa.cu", "cb200_mldsa_keygen", 1 << 14, "staged"),
]
PER_K = {"cb200_kyber_dot"}  # chunk = table value / k


def chunk_of(entry: str, k: int = 1) -> int:
    for name, _, _, c, _ in CHUNK_TABLE:
        if name == entry:
            return c // k if entry in PER_K else c
    raise KeyError(entry)


def schedule(n: int, chunk: int, pipeline: str = "staged"):
    """(first, count, slot) of every chunk a one-GPU host call of n operations runs, in order."""
    counts = []
    if pipeline == "staged":
        if chunk == 0 or chunk > n:
            chunk = n
        tail, left = [], n
        if n >= 6 * chunk and chunk >= 4096:  # short ramp chunks at both ends
            for r in (chunk // 4, chunk // 4, chunk // 2):
                counts.append(r)
                tail.append(r)
                left -= 2 * r
        while left > 0:
            counts.append(min(left, chunk))
            left -= counts[-1]
        counts += tail[::-1]
    else:
        counts = [min(chunk, n - f) for f in range(0, n, chunk)]
    out, first = [], 0
    for ci, cnt in enumerate(counts):
        out.append((first, cnt, ci % SLOTS[pipeline]))
        first += cnt
    return out


def boundary_rows(n: int, chunk: int, pipeline: str = "staged"):
    """The first and last rows of every chunk and their neighbours."""
    rows = set()
    for first, cnt, _ in schedule(n, chunk, pipeline):
        rows.update(r for r in (first - 1, first, first + 1, first + cnt - 2, first + cnt - 1, first + cnt) if 0 <= r < n)
    return sorted(rows)


def sample_rows(n: int, chunk: int, pipeline: str = "staged", stride: int = 499):
    return sorted(set(boundary_rows(n, chunk, pipeline)) | set(range(0, n, stride)) | {n - 1})


SIZES = {"4C+1": lambda c: 4 * c + 1, "6C+13": lambda c: 6 * c + 13}

ERR_ARG, ERR_PUBKEY, ERR_PRIVKEY = -1, -3, -5
Q_KYBER, Q_DIL = 3329, 8380417
NT = os.cpu_count() or 4


# ---------------------------------------------------------------- buffers
@pytest.fixture(scope="module")
def cb():
    import circl_b200
    circl_b200.init(0)
    yield circl_b200
    circl_b200.shutdown()


@pytest.fixture(scope="module")
def L(cb):
    from circl_b200 import _ffi
    return _ffi.lib()


def hbuf(shape, dtype=np.uint8, mem="pinned"):
    """Host array in pinned (page-locked, asynchronous copies) or pageable memory."""
    shape = (shape,) if isinstance(shape, int) else tuple(shape)
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    if mem == "pinned":
        import torch
        raw = torch.empty(max(nbytes, 1), dtype=torch.uint8, pin_memory=True).numpy()[:nbytes]
    else:
        raw = np.empty(nbytes, dtype=np.uint8)
    return raw.view(dtype).reshape(shape)


def put(a, mem="pinned"):
    a = np.ascontiguousarray(a)
    out = hbuf(a.shape, a.dtype, mem)
    out[...] = a
    return out


def ptr(a) -> int:
    return a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr()


def dev(a):
    """Flat uint8 CUDA tensor holding the bytes of a."""
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).cuda()


def dzeros(nbytes: int):
    import torch
    return torch.zeros(nbytes, dtype=torch.uint8, device="cuda")


def host(t, shape, dtype=np.uint8):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy().view(dtype).reshape(shape)


def rand_bytes(tag: bytes, n: int, width: int) -> np.ndarray:
    return np.frombuffer(hashlib.shake_256(tag).digest(n * width), dtype=np.uint8).reshape(n, width).copy()


def omap(fn, items):
    """Per-operation oracle calls; ctypes drops the GIL, so threads run them in parallel."""
    with ThreadPoolExecutor(max_workers=NT) as ex:
        return list(ex.map(fn, items))


def diff_rows(a, b):
    """Indices of the rows where a and b differ (both (n, ...))."""
    n = a.shape[0]
    a, b = a.reshape(n, -1), b.reshape(n, -1)
    bad = [np.flatnonzero((a[i:i + 65536] != b[i:i + 65536]).any(axis=1)) + i for i in range(0, n, 65536)]
    return np.concatenate(bad) if bad else np.zeros(0, dtype=np.int64)


def assert_rows_equal(got, want, what, rows=None):
    if rows is not None:
        got, want = got[rows], want[rows]
    d = diff_rows(got, want)
    if rows is not None:
        d = np.asarray(rows)[d]
    assert d.size == 0, f"{what}: {d.size} rows differ, first {d[:8].tolist()}"


def cstr(b: bytes):
    return C.create_string_buffer(b, max(len(b), 1))


def u64_ptr(x):
    return C.cast(C.pointer(x), C.c_void_p)


@functools.lru_cache(maxsize=None)
def mlkem_pool(k: int, count: int = 64):
    import oracle
    keys = [oracle.mlkem_keygen(k, hashlib.shake_256(b"pool%d" % j).digest(64)) for j in range(count)]
    ek = np.stack([np.frombuffer(e, dtype=np.uint8) for e, _ in keys])
    dk = np.stack([np.frombuffer(d, dtype=np.uint8) for _, d in keys])
    return ek, dk


@functools.lru_cache(maxsize=None)
def mldsa_pool(mode: int, count: int = 16):
    import oracle
    keys = [oracle.mldsa_keygen(mode, hashlib.shake_256(b"dsa%d-%d" % (mode, j)).digest(32)) for j in range(count)]
    pk = np.stack([np.frombuffer(p, dtype=np.uint8) for p, _ in keys])
    sk = np.stack([np.frombuffer(s, dtype=np.uint8) for _, s in keys])
    return pk, sk


def messages(n: int, tag: bytes, maxlen: int = 80):
    lens = np.frombuffer(hashlib.shake_256(tag + b"len").digest(n), dtype=np.uint8) % maxlen
    blob = np.frombuffer(hashlib.shake_256(tag).digest(int(lens.sum()) + 1), dtype=np.uint8)
    off = np.zeros(n + 1, dtype=np.uint64)
    off[1:] = np.cumsum(lens)
    return [blob[off[i]:off[i + 1]].tobytes() for i in range(n)]


def pack_messages(msgs, mem="pinned"):
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(m) for m in msgs])
    blob = np.frombuffer(b"".join(msgs) + b"\0", dtype=np.uint8)
    return put(blob, mem), put(off, mem)


def noncanonical(ek_row):
    ek_row[0], ek_row[1] = 0xFF, ek_row[1] | 0x0F  # first coefficient 4095 >= q: kem.ErrPubKey


# ---------------------------------------------------------------- 2. host batches across chunks, against the oracle
def _mlkem768_encaps_case(L, n, mem):
    import oracle
    k, eksz, ctsz = 3, 1184, 1088
    pool, _ = mlkem_pool(k)
    eks = put(pool[np.arange(n) % len(pool)], mem)
    sch = schedule(n, chunk_of("cb200_mlkem_encaps"))
    bad = {sch[4][0], n - 1}  # a reused slot and the last row
    bad |= {sch[7][0] + 6} if len(sch) == 11 else {sch[2][0] + sch[2][1] - 1}  # the 13-row chunk / a chunk end
    bad = sorted(bad)
    for r in bad:
        noncanonical(eks[r])
    seeds = put(rand_bytes(b"enc768-%d" % n, n, 32), mem)
    ct, ss, st = hbuf((n, ctsz), mem=mem), hbuf((n, 32), mem=mem), hbuf(n, mem=mem)
    ct[...], ss[...], st[...] = 0xAA, 0xAA, 0xAA
    assert L.cb200_mlkem_encaps(k, ptr(eks), eksz, ptr(seeds), ptr(ct), ptr(ss), ptr(st), n) == ERR_PUBKEY
    assert np.flatnonzero(st).tolist() == bad and (st[bad] == 1).all()
    assert not ct[bad].any() and not ss[bad].any()
    wct, wss, fails = oracle.mlkem_encaps_batch(k, eks, seeds, nthreads=NT)
    assert fails == len(bad)
    good = np.setdiff1d(np.arange(n), bad)
    assert_rows_equal(ct, wct, "ct", good)
    assert_rows_equal(ss, wss, "ss", good)


@pytest.mark.parametrize("size,mem", [("4C+1", "pinned"), ("6C+13", "pinned"), ("6C+13", "pageable")])
def test_mlkem768_encaps_per_op_keys_with_bad_keys_at_chunk_edges(L, size, mem):
    _mlkem768_encaps_case(L, SIZES[size](chunk_of("cb200_mlkem_encaps")), mem)


@pytest.mark.parametrize("size", list(SIZES))
def test_mlkem1024_encaps_shared_key(L, size):
    import oracle
    k, ctsz = 4, 1568
    n = SIZES[size](chunk_of("cb200_mlkem_encaps"))
    ek = put(mlkem_pool(k)[0][5])
    seeds = put(rand_bytes(b"enc1024" + size.encode(), n, 32))
    ct, ss, st = hbuf((n, ctsz)), hbuf((n, 32)), hbuf(n)
    st[...] = 0xAA
    assert L.cb200_mlkem_encaps(k, ptr(ek), 0, ptr(seeds), ptr(ct), ptr(ss), ptr(st), n) == 0
    assert not st.any()
    wct, wss, fails = oracle.mlkem_encaps_batch(k, ek, seeds, nthreads=NT)
    assert fails == 0
    assert_rows_equal(ct, wct, "ct")
    assert_rows_equal(ss, wss, "ss")


@pytest.mark.parametrize("size", list(SIZES))
@pytest.mark.parametrize("shared", [False, True], ids=["per-op-dk", "shared-dk"])
def test_mlkem768_decaps_rejection_and_privkey_at_chunk_edges(L, size, shared):
    import oracle
    k, dksz = 3, 2400
    C_ = chunk_of("cb200_mlkem_decaps")
    n = SIZES[size](C_)
    pek, pdk = mlkem_pool(k)
    idx = np.zeros(n, dtype=np.int64) if shared else np.arange(n) % len(pek)
    m = rand_bytes(b"dec" + size.encode(), n, 32)
    cts, want, fails = oracle.mlkem_encaps_batch(k, pek[0] if shared else pek[idx], m, nthreads=NT)
    assert fails == 0
    edges = boundary_rows(n, C_)
    corrupt = edges[::2]
    cts[corrupt, 5] ^= 0x40  # implicit rejection there
    sch = schedule(n, C_)
    hbad = None if shared else sch[min(5, len(sch) - 1)][0] + (0 if len(sch) == 11 else -1)
    while hbad is not None and hbad in corrupt:
        hbad += 1
    want[corrupt] = np.stack(omap(lambda r: np.frombuffer(oracle.mlkem_decaps(k, pdk[idx[r]].tobytes(), cts[r].tobytes()),
                                                           dtype=np.uint8), corrupt))
    dks = put(pdk[0]) if shared else put(pdk[idx])
    if hbad is not None:
        dks[hbad, 768 * k + 32 + 1] ^= 1  # H(ek) stored in dk
    ctp = put(cts)
    ss, st = hbuf((n, 32)), hbuf(n)
    ss[...], st[...] = 0xAA, 0xAA
    rc = L.cb200_mlkem_decaps(k, ptr(dks), 0 if shared else dksz, ptr(ctp), ptr(ss), ptr(st), n)
    if shared:
        assert rc == 0 and not st.any()
        assert_rows_equal(ss, want, "ss")
    else:
        assert rc == ERR_PRIVKEY
        assert np.flatnonzero(st).tolist() == [hbad] and st[hbad] == 2 and not ss[hbad].any()
        assert_rows_equal(ss, want, "ss", np.setdiff1d(np.arange(n), [hbad]))
    sample = [r for r in range(0, n, 997) if r != hbad]
    got = omap(lambda r: oracle.mlkem_decaps(k, dks.reshape(-1, dksz)[0 if shared else r].tobytes(), ctp[r].tobytes()), sample)
    assert [ss[r].tobytes() for r in sample] == got


@pytest.mark.parametrize("size", list(SIZES))
def test_mlkem768_keygen(L, size):
    import oracle
    k = 3
    n = SIZES[size](chunk_of("cb200_mlkem_keygen"))
    seeds = put(rand_bytes(b"kg" + size.encode(), n, 64))
    ek, dk = hbuf((n, 1184)), hbuf((n, 2400))
    assert L.cb200_mlkem_keygen(k, ptr(seeds), ptr(ek), ptr(dk), n) == 0
    d_s, d_ek, d_dk = dev(seeds), dzeros(n * 1184), dzeros(n * 2400)
    assert L.cb200_mlkem_keygen(k, ptr(d_s), ptr(d_ek), ptr(d_dk), n) == 0
    assert_rows_equal(ek, host(d_ek, (n, 1184)), "ek vs device call")
    assert_rows_equal(dk, host(d_dk, (n, 2400)), "dk vs device call")
    rows = sample_rows(n, chunk_of("cb200_mlkem_keygen"))
    want = omap(lambda r: oracle.mlkem_keygen(k, seeds[r].tobytes()), rows)
    assert [(ek[r].tobytes(), dk[r].tobytes()) for r in rows] == want


def test_kyber768_round3_kem_across_chunks(L):
    import oracle
    k, eksz, dksz, ctsz = 3, 1184, 2400, 1088
    C_ = chunk_of("cb200_kyber_kem_encaps")
    n = SIZES["6C+13"](C_)
    rows = sample_rows(n, C_)
    seeds = put(rand_bytes(b"r3kg", n, 64))
    ek, dk = hbuf((n, eksz)), hbuf((n, dksz))
    assert L.cb200_kyber_kem_keygen(k, ptr(seeds), ptr(ek), ptr(dk), n) == 0
    assert [(ek[r].tobytes(), dk[r].tobytes()) for r in rows] == omap(
        lambda r: oracle.kyber_kem_keygen(k, seeds[r].tobytes()), rows)
    es = put(rand_bytes(b"r3enc", n, 32))
    ct, ss = hbuf((n, ctsz)), hbuf((n, 32))
    assert L.cb200_kyber_kem_encaps(k, ptr(ek), eksz, ptr(es), ptr(ct), ptr(ss), n) == 0
    d_ek, d_es, d_ct, d_ss = dev(ek), dev(es), dzeros(n * ctsz), dzeros(n * 32)
    assert L.cb200_kyber_kem_encaps(k, ptr(d_ek), eksz, ptr(d_es), ptr(d_ct), ptr(d_ss), n) == 0
    assert_rows_equal(ct, host(d_ct, (n, ctsz)), "ct vs device call")
    assert_rows_equal(ss, host(d_ss, (n, 32)), "ss vs device call")
    assert [(ct[r].tobytes(), ss[r].tobytes()) for r in rows] == omap(
        lambda r: oracle.kyber_kem_encaps(k, ek[r].tobytes(), es[r].tobytes()), rows)
    corrupt = boundary_rows(n, C_)[1::2]
    ct[corrupt, 17] ^= 0x08
    want = ss.copy()
    want[corrupt] = np.stack([np.frombuffer(x, dtype=np.uint8) for x in omap(
        lambda r: oracle.kyber_kem_decaps(k, dk[r].tobytes(), ct[r].tobytes()), corrupt)])
    out = hbuf((n, 32))
    assert L.cb200_kyber_kem_decaps(k, ptr(dk), dksz, ptr(ct), ptr(out), n) == 0
    assert_rows_equal(out, want, "decapsulated ss")


@pytest.mark.parametrize("size", list(SIZES))
def test_xwing_keygen_encaps_decaps(L, size):
    import oracle
    C_ = chunk_of("cb200_xwing_encaps")
    n = SIZES[size](C_)
    rows = sample_rows(n, C_)
    seeds = put(rand_bytes(b"xw" + size.encode(), n, 32))
    pk = hbuf((n, 1216))
    assert L.cb200_xwing_keygen(ptr(seeds), ptr(pk), n) == 0
    d_seeds, d_pk = dev(seeds), dzeros(n * 1216)
    assert L.cb200_xwing_keygen(ptr(d_seeds), ptr(d_pk), n) == 0
    assert_rows_equal(pk, host(d_pk, (n, 1216)), "pk vs device call")
    assert [pk[r].tobytes() for r in rows] == omap(lambda r: oracle.xwing_keygen(seeds[r].tobytes()), rows)
    es = put(rand_bytes(b"xwe" + size.encode(), n, 64))
    ct, ss, st = hbuf((n, 1120)), hbuf((n, 32)), hbuf(n)
    st[...] = 0xAA
    assert L.cb200_xwing_encaps(ptr(pk), 1216, ptr(es), ptr(ct), ptr(ss), ptr(st), n) == 0
    assert not st.any()
    d_es, d_ct, d_ss, d_st = dev(es), dzeros(n * 1120), dzeros(n * 32), dzeros(n)
    assert L.cb200_xwing_encaps(ptr(d_pk), 1216, ptr(d_es), ptr(d_ct), ptr(d_ss), ptr(d_st), n) == 0
    assert_rows_equal(ct, host(d_ct, (n, 1120)), "ct vs device call")
    assert_rows_equal(ss, host(d_ss, (n, 32)), "ss vs device call")
    assert [(ct[r].tobytes(), ss[r].tobytes()) for r in rows] == omap(
        lambda r: oracle.xwing_encaps(pk[r].tobytes(), es[r].tobytes()), rows)
    corrupt = boundary_rows(n, C_)[::2]
    ct[corrupt, 3] ^= 0x20  # in the ML-KEM part: implicit rejection
    want = ss.copy()
    want[corrupt] = np.stack([np.frombuffer(x, dtype=np.uint8) for x in omap(
        lambda r: oracle.xwing_decaps(seeds[r].tobytes(), ct[r].tobytes()), corrupt)])
    out = hbuf((n, 32))
    assert L.cb200_xwing_decaps(ptr(seeds), 32, ptr(ct), ptr(out), n) == 0
    assert_rows_equal(out, want, "decapsulated ss")


SMALL_ORDER = [bytes(32), bytes([1]) + bytes(31),
               bytes.fromhex("e0eb7a7c3b41b8ae1656e3faf19fc46ada098deb9c32b1fd866205165f49b800")]


@pytest.mark.parametrize("size", list(SIZES))
def test_x25519_shared_with_small_order_points_at_chunk_edges(L, size):
    import oracle
    C_ = chunk_of("cb200_x25519")
    n = SIZES[size](C_)
    sch = schedule(n, C_)
    sc = put(rand_bytes(b"x25519s" + size.encode(), n, 32))
    pts = put(rand_bytes(b"x25519p" + size.encode(), n, 32))
    bad = sorted({sch[4][0], sch[1][0] + sch[1][1] - 1, n - 1} | ({sch[7][0] + 12} if len(sch) == 11 else set()))
    for j, r in enumerate(bad):
        pts[r] = np.frombuffer(SMALL_ORDER[j % len(SMALL_ORDER)], dtype=np.uint8)
    out, st = hbuf((n, 32)), hbuf(n)
    out[...], st[...] = 0xAA, 0xAA
    assert L.cb200_x25519(ptr(sc), ptr(pts), ptr(out), ptr(st), n) == ERR_PUBKEY
    assert np.flatnonzero(st).tolist() == bad and not out[bad].any()
    d_sc, d_pts, d_out, d_st = dev(sc), dev(pts), dzeros(n * 32), dzeros(n)
    assert L.cb200_x25519(ptr(d_sc), ptr(d_pts), ptr(d_out), ptr(d_st), n) == 0
    assert_rows_equal(out, host(d_out, (n, 32)), "vs device call")
    assert np.array_equal(st, host(d_st, (n,)))
    rows = sample_rows(n, C_)
    want = omap(lambda r: oracle.x25519(sc[r].tobytes(), pts[r].tobytes()), rows)
    assert [(out[r].tobytes(), st[r] == 0) for r in rows] == want


def _mldsa65_sign_case(L, n):
    """Per-op keys, hedged rnd, a context, empty messages at chunk starts and one >= 64 KiB message in the last chunk:
    host call vs device-pointer call on every row, and vs the oracle at the chunk edges and a stride."""
    import oracle
    mode, sksz, sigsz = 65, 4032, 3309
    C_ = chunk_of("cb200_mldsa_sign")
    _, psk = mldsa_pool(mode)
    idx = np.arange(n) % len(psk)
    msgs = messages(n, b"sign%d" % n)
    for first, _, _ in schedule(n, C_, "sign"):
        msgs[first] = b""
    msgs[n - 2] = hashlib.shake_256(b"long").digest(65536 + 77)
    blob, off = pack_messages(msgs)
    sks, rnd = put(psk[idx]), put(rand_bytes(b"rnd%d" % n, n, 32))
    ctx = b"chunked batch"
    sig, st = hbuf((n, sigsz)), hbuf(n)
    st[...] = 0xAA
    att = C.c_uint64(0)
    assert L.cb200_mldsa_sign(mode, ptr(sks), sksz, ptr(blob), ptr(off), cstr(ctx), len(ctx), ptr(rnd), ptr(sig), ptr(st),
                              n, 0, u64_ptr(att)) == 0, L.cb200_last_error()
    assert not st.any()
    d_sk, d_blob, d_off, d_rnd = dev(sks), dev(blob), dev(off), dev(rnd)
    d_sig, d_st, datt = dzeros(n * sigsz), dzeros(n), C.c_uint64(0)
    assert L.cb200_mldsa_sign(mode, ptr(d_sk), sksz, ptr(d_blob), ptr(d_off), cstr(ctx), len(ctx), ptr(d_rnd), ptr(d_sig),
                              ptr(d_st), n, 0, u64_ptr(datt)) == 0, L.cb200_last_error()
    assert_rows_equal(sig, host(d_sig, (n, sigsz)), "signatures vs device call")
    assert att.value == datt.value
    rows = sample_rows(n, C_, "sign")
    want = omap(lambda r: oracle.mldsa_sign(mode, psk[idx[r]].tobytes(), msgs[r], ctx, rnd[r].tobytes())[0], rows)
    assert [sig[r].tobytes() for r in rows] == want


def test_mldsa65_sign_per_op_keys_across_chunks(L):
    _mldsa65_sign_case(L, 3 * (1 << 16) + 5)


def test_mldsa65_sign_shared_key_across_chunks(L):
    import oracle
    mode, sigsz = 65, 3309
    n = (1 << 16) + 1
    _, psk = mldsa_pool(mode)
    msgs = messages(n, b"shared")
    blob, off = pack_messages(msgs)
    sk, rnd = put(psk[3]), put(rand_bytes(b"rnd-shared", n, 32))
    sig, att = hbuf((n, sigsz)), C.c_uint64(0)
    assert L.cb200_mldsa_sign(mode, ptr(sk), 0, ptr(blob), ptr(off), None, 0, ptr(rnd), ptr(sig), None, n, 0,
                              u64_ptr(att)) == 0
    want, want_att = oracle.mldsa_sign_batch(mode, psk[3], msgs, rnd=rnd, nthreads=NT)
    assert_rows_equal(sig, want, "signatures")
    assert att.value == want_att


def test_mldsa65_verify_with_tampered_signatures_at_chunk_edges(L):
    import oracle
    mode, pksz, sksz, sigsz = 65, 1952, 4032, 3309
    C_ = chunk_of("cb200_mldsa_verify")
    n = 2 * C_ + 3
    ppk, psk = mldsa_pool(mode)
    idx = np.arange(n) % len(ppk)
    msgs = messages(n, b"verify")
    blob, off = pack_messages(msgs)
    ctx = b"verify ctx"
    sig = hbuf((n, sigsz))
    assert L.cb200_mldsa_sign(mode, ptr(put(psk[idx])), sksz, ptr(blob), ptr(off), cstr(ctx), len(ctx), None, ptr(sig),
                              None, n, 0, None) == 0
    tampered = boundary_rows(n, C_, "verify")
    sig[tampered, 100] ^= 0x01
    ok = hbuf(n)
    ok[...] = 0xAA
    assert L.cb200_mldsa_verify(mode, ptr(put(ppk[idx])), pksz, ptr(blob), ptr(off), cstr(ctx), len(ctx), ptr(sig), ptr(ok),
                                n, 0) == 0
    assert np.flatnonzero(ok != 1).tolist() == tampered and not ok[tampered].any()
    rows = tampered[:6] + list(range(1, n, 4099))
    assert [bool(ok[r]) for r in rows] == omap(
        lambda r: oracle.mldsa_verify(mode, ppk[idx[r]].tobytes(), msgs[r], sig[r].tobytes(), ctx), rows)


@pytest.mark.parametrize("size", list(SIZES))
def test_mldsa65_keygen(L, size):
    import oracle
    mode, pksz, sksz = 65, 1952, 4032
    C_ = chunk_of("cb200_mldsa_keygen")
    n = SIZES[size](C_)
    seeds = put(rand_bytes(b"dkg" + size.encode(), n, 32))
    pk, sk = hbuf((n, pksz)), hbuf((n, sksz))
    assert L.cb200_mldsa_keygen(mode, ptr(seeds), ptr(pk), ptr(sk), n) == 0
    d_s, d_pk, d_sk = dev(seeds), dzeros(n * pksz), dzeros(n * sksz)
    assert L.cb200_mldsa_keygen(mode, ptr(d_s), ptr(d_pk), ptr(d_sk), n) == 0
    assert_rows_equal(pk, host(d_pk, (n, pksz)), "pk vs device call")
    assert_rows_equal(sk, host(d_sk, (n, sksz)), "sk vs device call")
    rows = sample_rows(n, C_)
    assert [(pk[r].tobytes(), sk[r].tobytes()) for r in rows] == omap(
        lambda r: oracle.mldsa_keygen(mode, seeds[r].tobytes()), rows)


# ---- raw ring ops
@pytest.mark.parametrize("mem", ["pinned", "pageable"])
def test_kyber_ntt_in_place_over_the_ramp(L, mem):
    import oracle
    C_ = chunk_of("cb200_kyber_ntt")
    n = SIZES["6C+13"](C_)
    rng = np.random.default_rng(11)
    p = rng.integers(-Q_KYBER, Q_KYBER + 1, size=(n, 256), dtype=np.int16)
    want = p.copy()
    oracle.kyber_ntt_inplace_mt(want, False, NT)
    got = put(p, mem)
    del p
    assert L.cb200_kyber_ntt(ptr(got), n, 0) == 0
    assert_rows_equal(got, want, "NTT")


def test_kyber_dot_k3_over_the_ramp(L):
    import oracle
    k = 3
    C_ = chunk_of("cb200_kyber_dot", k)
    n = SIZES["6C+13"](C_)
    rng = np.random.default_rng(12)
    a = put(rng.integers(-Q_KYBER, Q_KYBER + 1, size=(n, k, 256), dtype=np.int16))
    b = put(rng.integers(-Q_KYBER, Q_KYBER + 1, size=(n, k, 256), dtype=np.int16))
    out = hbuf((n, 256), np.int16)
    assert L.cb200_kyber_dot(ptr(out), ptr(a), ptr(b), k, n) == 0
    assert_rows_equal(out, oracle.kyber_dot(a, b, k), "PolyDotHat")


def test_dilithium_ntt_in_place_over_the_ramp(L):
    import oracle
    C_ = chunk_of("cb200_dil_ntt")
    n = SIZES["6C+13"](C_)
    p = np.random.default_rng(13).integers(0, Q_DIL, size=(n, 256), dtype=np.uint32)
    got = put(p)
    assert L.cb200_dil_ntt(ptr(got), n, 0) == 0
    assert_rows_equal(got, oracle.dil_ntt(p), "NTT")


def test_kyber_poly_op_with_out_aliasing_the_input(L):
    import oracle
    C_ = chunk_of("cb200_kyber_poly_op")
    n = SIZES["4C+1"](C_)
    a = np.random.default_rng(14).integers(-32768, 32768, size=(n, 256), dtype=np.int16)
    want = hbuf((n, 256), np.int16)
    src = put(a)
    assert L.cb200_kyber_poly_op(2, ptr(want), ptr(src), None, n) == 0  # BarrettReduce, separate output
    assert L.cb200_kyber_poly_op(2, ptr(src), ptr(src), None, n) == 0   # out == a
    assert_rows_equal(src, want, "aliased vs separate output")
    rows = sample_rows(n, C_)
    assert_rows_equal(src[rows], oracle.kyber_barrett(a[rows]), "BarrettReduce vs oracle")


# ---- strided host rows: op i uses base + i * stride
def _strided(rows: np.ndarray, stride: int):
    """rows (n, w) placed at a stride of `stride` bytes, the gaps filled with 0xFF."""
    n, w = rows.shape
    out = hbuf(n * stride + w)
    out[...] = 0xFF
    view = np.lib.stride_tricks.as_strided(out, shape=(n, w), strides=(stride, 1))
    view[...] = rows
    return out


@pytest.mark.parametrize("pad", [16, 1])
def test_mlkem_encaps_and_decaps_strided_keys(L, pad):
    k, eksz, dksz, ctsz = 3, 1184, 2400, 1088
    n = chunk_of("cb200_mlkem_encaps") + 5
    pek, pdk = mlkem_pool(k)
    idx = np.arange(n) % len(pek)
    seeds = put(rand_bytes(b"strided", n, 32))
    dense = [hbuf((n, ctsz)), hbuf((n, 32))]
    assert L.cb200_mlkem_encaps(k, ptr(put(pek[idx])), eksz, ptr(seeds), ptr(dense[0]), ptr(dense[1]), None, n) == 0
    ct, ss, st = hbuf((n, ctsz)), hbuf((n, 32)), hbuf(n)
    assert L.cb200_mlkem_encaps(k, ptr(_strided(pek[idx], eksz + pad)), eksz + pad, ptr(seeds), ptr(ct), ptr(ss), ptr(st),
                                n) == 0, L.cb200_last_error()
    assert_rows_equal(ct, dense[0], "ct")
    assert_rows_equal(ss, dense[1], "ss")
    m = chunk_of("cb200_mlkem_decaps") + 5
    out = hbuf((m, 32))
    assert L.cb200_mlkem_decaps(k, ptr(_strided(pdk[idx[:m]], dksz + pad)), dksz + pad, ptr(put(ct[:m])), ptr(out), None,
                                m) == 0, L.cb200_last_error()
    assert_rows_equal(out, ss[:m], "decapsulated ss")


@pytest.mark.parametrize("pad", [16, 1])
def test_mldsa_strided_sk_and_pk(L, pad):
    mode, pksz, sksz, sigsz = 65, 1952, 4032, 3309
    n = chunk_of("cb200_mldsa_sign") + 3
    ppk, psk = mldsa_pool(mode)
    idx = np.arange(n) % len(psk)
    msgs = messages(n, b"strided-dsa")
    blob, off = pack_messages(msgs)
    dense, sig = hbuf((n, sigsz)), hbuf((n, sigsz))
    assert L.cb200_mldsa_sign(mode, ptr(put(psk[idx])), sksz, ptr(blob), ptr(off), None, 0, None, ptr(dense), None, n, 0,
                              None) == 0
    assert L.cb200_mldsa_sign(mode, ptr(_strided(psk[idx], sksz + pad)), sksz + pad, ptr(blob), ptr(off), None, 0, None,
                              ptr(sig), None, n, 0, None) == 0, L.cb200_last_error()
    assert_rows_equal(sig, dense, "signatures")
    m = chunk_of("cb200_mldsa_verify") + 3
    sig[m - 1, 9] ^= 1
    ok = hbuf(m)
    assert L.cb200_mldsa_verify(mode, ptr(_strided(ppk[idx[:m]], pksz + pad)), pksz + pad, ptr(blob), ptr(off), None, 0,
                                ptr(sig), ptr(ok), m, 0) == 0, L.cb200_last_error()
    assert ok[:m - 1].all() and ok[m - 1] == 0


@pytest.mark.parametrize("pad", [16, 1])
def test_sampler_seed_stride_and_sha3_in_stride(L, pad):
    n = chunk_of("cb200_kyber_derive_uniform") + 5
    seeds = rand_bytes(b"seeds", n, 32)
    xy = put(rand_bytes(b"xy", n, 2) % 3)
    dense, got = hbuf((n, 256), np.int16), hbuf((n, 256), np.int16)
    assert L.cb200_kyber_derive_uniform(ptr(dense), ptr(put(seeds)), 32, ptr(xy), n) == 0
    assert L.cb200_kyber_derive_uniform(ptr(got), ptr(_strided(seeds, 32 + pad)), 32 + pad, ptr(xy), n) == 0
    assert_rows_equal(got, dense, "DeriveUniform")
    n = chunk_of("cb200_sha3") + 5
    inlen = 50
    msgs = rand_bytes(b"sha3in", n, inlen)
    dense, got = hbuf((n, 32)), hbuf((n, 32))
    assert L.cb200_sha3(128, ptr(put(msgs)), inlen, inlen, ptr(dense), 32, n) == 0
    assert L.cb200_sha3(128, ptr(_strided(msgs, inlen + pad)), inlen + pad, inlen, ptr(got), 32, n) == 0
    assert_rows_equal(got, dense, "SHAKE128")
    for r in (0, n // 2, n - 1):
        assert got[r].tobytes() == hashlib.shake_128(msgs[r].tobytes()).digest(32)


@pytest.mark.parametrize("pad", [16, 1])
def test_xwing_strided_host_keys(L, pad):
    """Host rows may sit at any stride >= the row size; device strides must be multiples of 16 bytes."""
    n = chunk_of("cb200_xwing_encaps") + 5
    seeds = rand_bytes(b"xws", n, 32)
    pk = hbuf((n, 1216))
    assert L.cb200_xwing_keygen(ptr(put(seeds)), ptr(pk), n) == 0
    es = put(rand_bytes(b"xwes", n, 64))
    dense = [hbuf((n, 1120)), hbuf((n, 32))]
    assert L.cb200_xwing_encaps(ptr(pk), 1216, ptr(es), ptr(dense[0]), ptr(dense[1]), None, n) == 0
    ct, ss = hbuf((n, 1120)), hbuf((n, 32))
    assert L.cb200_xwing_encaps(ptr(_strided(pk, 1216 + pad)), 1216 + pad, ptr(es), ptr(ct), ptr(ss), None,
                                n) == 0, L.cb200_last_error()
    assert_rows_equal(ct, dense[0], "ct")
    assert_rows_equal(ss, dense[1], "ss")
    out = hbuf((n, 32))
    assert L.cb200_xwing_decaps(ptr(_strided(seeds, 32 + pad)), 32 + pad, ptr(ct), ptr(out), n) == 0, L.cb200_last_error()
    assert_rows_equal(out, ss, "decapsulated ss")
    if pad % 16:
        d_pk, d_es, d_ct, d_ss = dev(_strided(pk[:4], 1216 + pad)), dev(es[:4]), dzeros(4 * 1120), dzeros(4 * 32)
        assert L.cb200_xwing_encaps(ptr(d_pk), 1216 + pad, ptr(d_es), ptr(d_ct), ptr(d_ss), None, 4) == ERR_ARG
        d_sk = dev(_strided(seeds[:4], 32 + pad))
        assert L.cb200_xwing_decaps(ptr(d_sk), 32 + pad, ptr(d_ct), ptr(d_ss), 4) == ERR_ARG


def test_host_batches_sharded_over_several_gpus(cb, L):
    """Shard boundaries (n * s / shards) fall inside staging chunks."""
    if cb.device_count() < 2:
        pytest.skip("needs at least two GPUs in this process")
    try:
        cb.init_devices(0)
        _mlkem768_encaps_case(L, SIZES["6C+13"](chunk_of("cb200_mlkem_encaps")), "pinned")
        _mldsa65_sign_case(L, 3 * (1 << 16) + 5)
    finally:
        cb.init(0)


# ---------------------------------------------------------------- 3. ML-DSA through device pointers
DSA_MODES = {"ML-DSA-44": 44, "ML-DSA-65": 65, "ML-DSA-87": 87, "Dilithium3": 3}


@pytest.mark.parametrize("ps", list(DSA_MODES))
@pytest.mark.parametrize("shared", [False, True], ids=["per-op-sk", "shared-sk"])
def test_mldsa_device_pointers_vs_oracle(L, ps, shared):
    import oracle
    mode = DSA_MODES[ps]
    pksz, sksz, sigsz = oracle.mldsa_sizes(mode)
    n = 67
    ppk, psk = mldsa_pool(mode, 6)
    idx = np.zeros(n, dtype=np.int64) if shared else np.arange(n) % len(psk)
    msgs = messages(n, ps.encode())
    msgs[0] = msgs[n // 2] = b""
    blob, off = pack_messages(msgs)
    nist = mode > 10
    ctx = b"device context" if nist else b""
    rnd = rand_bytes(ps.encode() + b"rnd", n, 32) if nist else np.zeros((n, 32), dtype=np.uint8)
    d_sk = dev(psk[0] if shared else psk[idx])
    d_blob, d_off, d_rnd = dev(blob), dev(off), dev(rnd)
    d_sig, d_st = dzeros(n * sigsz), dev(np.full(n, 0xAA, dtype=np.uint8))
    att = C.c_uint64(0)
    assert L.cb200_mldsa_sign(mode, ptr(d_sk), 0 if shared else sksz, ptr(d_blob), ptr(d_off), cstr(ctx), len(ctx),
                              ptr(d_rnd) if nist else None, ptr(d_sig), ptr(d_st), n, 0, u64_ptr(att)) == 0, \
        L.cb200_last_error()
    sig, st = host(d_sig, (n, sigsz)), host(d_st, (n,))
    assert not st.any()
    want = omap(lambda r: oracle.mldsa_sign(mode, psk[idx[r]].tobytes(), msgs[r], ctx, rnd[r].tobytes()), range(n))
    assert [sig[r].tobytes() for r in range(n)] == [w[0] for w in want]
    assert att.value == sum(w[1] for w in want)
    # verify, device pointers, some signatures tampered
    bad = sig.copy()
    tampered = [1, 2, n - 1]
    bad[tampered, 50] ^= 0x10
    d_pk, d_bad, d_ok = dev(ppk[0] if shared else ppk[idx]), dev(bad), dev(np.full(n, 0xAA, dtype=np.uint8))
    assert L.cb200_mldsa_verify(mode, ptr(d_pk), 0 if shared else pksz, ptr(d_blob), ptr(d_off), cstr(ctx), len(ctx),
                                ptr(d_bad), ptr(d_ok), n, 0) == 0, L.cb200_last_error()
    ok = host(d_ok, (n,))
    assert np.flatnonzero(ok != 1).tolist() == tampered and not ok[tampered].any()
    # keygen, device pointers
    seeds = rand_bytes(ps.encode() + b"seed", 9, 32)
    d_pk2, d_sk2 = dzeros(9 * pksz), dzeros(9 * sksz)
    assert L.cb200_mldsa_keygen(mode, ptr(dev(seeds)), ptr(d_pk2), ptr(d_sk2), 9) == 0
    pk2, sk2 = host(d_pk2, (9, pksz)), host(d_sk2, (9, sksz))
    assert [(pk2[i].tobytes(), sk2[i].tobytes()) for i in range(9)] == [oracle.mldsa_keygen(mode, s.tobytes()) for s in seeds]


def test_mldsa_device_pointer_misalignment_is_an_argument_error(L, cb):
    mode, pksz, sksz, sigsz = 65, 1952, 4032, 3309
    n = 4
    ppk, psk = mldsa_pool(mode)
    blob, off = pack_messages([b"a", b"bc", b"", b"def"])
    sk_buf, pk_buf = dev(np.concatenate([psk[:n].reshape(-1), np.zeros(64, np.uint8)])), dev(
        np.concatenate([ppk[:n].reshape(-1), np.zeros(64, np.uint8)]))
    off_buf = dev(np.concatenate([np.zeros(2, np.uint64), off]))  # off at +16 bytes; +8 is misaligned
    d_blob, d_sig, d_ok = dev(blob), dzeros(n * sigsz + 64), dzeros(64)
    import torch
    torch.cuda.synchronize()
    before = cb.launch_count()
    o16, o8 = ptr(off_buf) + 16, ptr(off_buf) + 8
    cases = [
        L.cb200_mldsa_sign(mode, ptr(sk_buf) + 1, sksz, ptr(d_blob), o16, None, 0, None, ptr(d_sig), None, n, 0, None),
        L.cb200_mldsa_sign(mode, ptr(sk_buf), sksz, ptr(d_blob), o8, None, 0, None, ptr(d_sig), None, n, 0, None),
        L.cb200_mldsa_sign(mode, ptr(sk_buf), sksz + 8, ptr(d_blob), o16, None, 0, None, ptr(d_sig), None, n - 1, 0, None),
        L.cb200_mldsa_verify(mode, ptr(pk_buf) + 4, pksz, ptr(d_blob), o16, None, 0, ptr(d_sig), ptr(d_ok), n, 0),
        L.cb200_mldsa_verify(mode, ptr(pk_buf), pksz, ptr(d_blob), o8, None, 0, ptr(d_sig), ptr(d_ok), n, 0),
        L.cb200_mldsa_verify(mode, ptr(pk_buf), pksz + 1, ptr(d_blob), o16, None, 0, ptr(d_sig), ptr(d_ok), n - 1, 0),
    ]
    assert cases == [ERR_ARG] * len(cases)
    assert cb.launch_count() == before  # rejected before anything was launched
    # the aligned call on the same buffers works
    assert L.cb200_mldsa_sign(mode, ptr(sk_buf), sksz, ptr(d_blob), o16, None, 0, None, ptr(d_sig), None, n, 0, None) == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------- 4. caller-stream order of device-pointer calls
SLEEP_CYCLES = 200_000_000  # about 0.1 s of a busy caller stream ahead of the call
SENTINEL = 0x5C
NS = 4 * 8192  # four ML-KEM sub-batches: both internal lanes finish work of their own


def _dsa_inputs(n):
    _, psk = mldsa_pool(65, 8)
    msgs = messages(n, b"stream")
    blob, off = pack_messages(msgs)
    return psk[np.arange(n) % 8], blob, off


def _stream_cases(L):
    """name -> builder() returning (inputs [(device buffer, device source)], outputs [device buffer], call(L))."""
    pek, pdk = mlkem_pool(3)
    idx = np.arange(NS) % len(pek)

    def kyber_ntt():
        p = np.random.default_rng(1).integers(-Q_KYBER, Q_KYBER, size=(1 << 16, 256), dtype=np.int16)
        buf = dzeros(p.nbytes)
        return [(buf, dev(p))], [buf], lambda L: L.cb200_kyber_ntt(ptr(buf), p.shape[0], 0)

    def dil_ntt():
        p = np.random.default_rng(2).integers(0, Q_DIL, size=(1 << 15, 256), dtype=np.uint32)
        buf = dzeros(p.nbytes)
        return [(buf, dev(p))], [buf], lambda L: L.cb200_dil_ntt(ptr(buf), p.shape[0], 0)

    def sha3():
        m = rand_bytes(b"s3", NS, 64)
        i, o = dzeros(m.nbytes), dzeros(NS * 32)
        return [(i, dev(m))], [o], lambda L: L.cb200_sha3(256, ptr(i), 64, 64, ptr(o), 32, NS)

    def mlkem_encaps(push=False):
        ek, s = dzeros(NS * 1184), dzeros(NS * 32)
        ct, ss, st = dzeros(NS * 1088), dzeros(NS * 32), dzeros(NS)
        ins = [(ek, dev(pek[idx])), (s, dev(rand_bytes(b"se", NS, 32)))]
        if not push:
            return ins, [ct, ss, st], lambda L: L.cb200_mlkem_encaps(3, ptr(ek), 1184, ptr(s), ptr(ct), ptr(ss), ptr(st), NS)
        pct, pss = dzeros(NS * 1088), dzeros(NS * 32)
        return ins, [ct, ss, st, pct, pss], lambda L: L.cb200_mlkem_encaps_push(
            3, ptr(ek), 1184, ptr(s), ptr(ct), ptr(ss), ptr(st), NS, ptr(pct), ptr(pss))

    def mlkem_decaps():
        dk, ct = dzeros(NS * 2400), dzeros(NS * 1088)
        ss, st = dzeros(NS * 32), dzeros(NS)
        return [(dk, dev(pdk[idx])), (ct, dev(rand_bytes(b"sd", NS, 1088)))], [ss, st], \
            lambda L: L.cb200_mlkem_decaps(3, ptr(dk), 2400, ptr(ct), ptr(ss), ptr(st), NS)

    def mlkem_keygen():
        s, ek, dk = dzeros(NS * 64), dzeros(NS * 1184), dzeros(NS * 2400)
        return [(s, dev(rand_bytes(b"sk", NS, 64)))], [ek, dk], lambda L: L.cb200_mlkem_keygen(3, ptr(s), ptr(ek), ptr(dk), NS)

    def kyber768_encaps():
        ek, s, ct, ss = dzeros(NS * 1184), dzeros(NS * 32), dzeros(NS * 1088), dzeros(NS * 32)
        return [(ek, dev(pek[idx])), (s, dev(rand_bytes(b"ke", NS, 32)))], [ct, ss], \
            lambda L: L.cb200_kyber_kem_encaps(3, ptr(ek), 1184, ptr(s), ptr(ct), ptr(ss), NS)

    def kyber768_decaps():
        dk, ct, ss = dzeros(NS * 2400), dzeros(NS * 1088), dzeros(NS * 32)
        return [(dk, dev(pdk[idx])), (ct, dev(rand_bytes(b"kd", NS, 1088)))], [ss], \
            lambda L: L.cb200_kyber_kem_decaps(3, ptr(dk), 2400, ptr(ct), ptr(ss), NS)

    def xwing_encaps():
        import oracle
        pool = np.stack([np.frombuffer(oracle.xwing_keygen(bytes([j]) * 32), dtype=np.uint8) for j in range(16)])
        pk, es = dzeros(NS * 1216), dzeros(NS * 64)
        ct, ss, st = dzeros(NS * 1120), dzeros(NS * 32), dzeros(NS)
        return [(pk, dev(pool[np.arange(NS) % 16])), (es, dev(rand_bytes(b"xe", NS, 64)))], [ct, ss, st], \
            lambda L: L.cb200_xwing_encaps(ptr(pk), 1216, ptr(es), ptr(ct), ptr(ss), ptr(st), NS)

    def xwing_decaps():
        sk, ct, ss = dzeros(NS * 32), dzeros(NS * 1120), dzeros(NS * 32)
        return [(sk, dev(rand_bytes(b"xs", NS, 32))), (ct, dev(rand_bytes(b"xc", NS, 1120)))], [ss], \
            lambda L: L.cb200_xwing_decaps(ptr(sk), 32, ptr(ct), ptr(ss), NS)

    def hybrid_keys():
        import oracle
        keys = [oracle.hybrid_keygen("X25519MLKEM768", bytes([j]) * 64) for j in range(16)]
        return (np.stack([np.frombuffer(p, dtype=np.uint8) for p, _ in keys]),
                np.stack([np.frombuffer(s, dtype=np.uint8) for _, s in keys]))

    def hybrid_encaps():
        pool, _ = hybrid_keys()
        pk, s = dzeros(NS * 1216), dzeros(NS * 32)
        ct, ss, st = dzeros(NS * 1120), dzeros(NS * 64), dzeros(NS)
        return [(pk, dev(pool[np.arange(NS) % 16])), (s, dev(rand_bytes(b"he", NS, 32)))], [ct, ss, st], \
            lambda L: L.cb200_hybrid_encaps(0, ptr(pk), 1216, ptr(s), ptr(ct), ptr(ss), ptr(st), NS)

    def hybrid_decaps():
        import oracle
        pool, skp = hybrid_keys()
        j = np.arange(NS) % 16
        cts = np.stack([np.frombuffer(oracle.hybrid_encaps("X25519MLKEM768", pool[i].tobytes(), bytes([i]) * 32)[0],
                                      dtype=np.uint8) for i in range(16)])
        sk, ct, ss, st = dzeros(NS * 2432), dzeros(NS * 1120), dzeros(NS * 64), dzeros(NS)
        return [(sk, dev(skp[j])), (ct, dev(cts[j]))], [ss, st], \
            lambda L: L.cb200_hybrid_decaps(0, ptr(sk), 2432, ptr(ct), ptr(ss), ptr(st), NS)

    def mldsa_sign():
        n = 2048
        sks, blob, off = _dsa_inputs(n)
        sk, b, o, rnd = dzeros(sks.nbytes), dzeros(blob.nbytes), dzeros(off.nbytes), dzeros(n * 32)
        sig, st = dzeros(n * 3309), dzeros(n)
        ctx = cstr(b"stream ctx")
        return [(sk, dev(sks)), (b, dev(blob)), (o, dev(off)), (rnd, dev(rand_bytes(b"sr", n, 32)))], [sig, st], \
            lambda L: L.cb200_mldsa_sign(65, ptr(sk), 4032, ptr(b), ptr(o), ctx, 10, ptr(rnd), ptr(sig), ptr(st), n, 0, None)

    def mldsa_verify():
        n = 2048
        sks, blob, off = _dsa_inputs(n)
        ppk, _ = mldsa_pool(65, 8)
        sig = hbuf((n, 3309))
        assert L.cb200_mldsa_sign(65, ptr(put(sks)), 4032, ptr(blob), ptr(off), None, 0, None, ptr(sig), None, n, 0,
                                  None) == 0
        sig[::7, 33] ^= 4
        pk, b, o, s, ok = dzeros(n * 1952), dzeros(blob.nbytes), dzeros(off.nbytes), dzeros(sig.nbytes), dzeros(n)
        return [(pk, dev(ppk[np.arange(n) % 8])), (b, dev(blob)), (o, dev(off)), (s, dev(sig))], [ok], \
            lambda L: L.cb200_mldsa_verify(65, ptr(pk), 1952, ptr(b), ptr(o), None, 0, ptr(s), ptr(ok), n, 0)

    return {"kyber_ntt": kyber_ntt, "dil_ntt": dil_ntt, "sha3": sha3, "mlkem_encaps": mlkem_encaps,
            "mlkem_decaps": mlkem_decaps, "mlkem_keygen": mlkem_keygen, "kyber768_encaps": kyber768_encaps,
            "kyber768_decaps": kyber768_decaps, "xwing_encaps": xwing_encaps, "xwing_decaps": xwing_decaps,
            "x25519mlkem768_encaps": hybrid_encaps, "x25519mlkem768_decaps": hybrid_decaps, "mldsa_sign": mldsa_sign,
            "mldsa_verify": mldsa_verify, "mlkem_encaps_push": lambda: mlkem_encaps(push=True)}


STREAM_CASES = ["kyber_ntt", "dil_ntt", "sha3", "mlkem_encaps", "mlkem_decaps", "mlkem_keygen", "kyber768_encaps",
                "kyber768_decaps", "xwing_encaps", "xwing_decaps", "x25519mlkem768_encaps", "x25519mlkem768_decaps",
                "mldsa_sign", "mldsa_verify", "mlkem_encaps_push"]


@pytest.mark.parametrize("case", STREAM_CASES)
def test_device_call_is_ordered_on_the_callers_stream(L, case):
    """Behind ~0.1 s of work on a fresh stream s: write the inputs on s, call on s, clone the outputs on s and overwrite
    them with a sentinel on s.  The clones must be the results, and nothing may write the outputs after s passed the
    call.  For encaps-push the pushed rows must equal ct / ss as well."""
    import torch
    ins, outs, call = _stream_cases(L)[case]()
    # expected results: the same call on the default stream, synchronised
    for dst, src in ins:
        dst.copy_(src)
    torch.cuda.synchronize()
    assert L.cb200_set_stream(None) == 0
    assert call(L) == 0, L.cb200_last_error()
    torch.cuda.synchronize()
    want = [o.clone() for o in outs]
    for dst, _ in ins:
        dst.zero_()
    for o in outs:
        o.fill_(0x77)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    assert L.cb200_set_stream(C.c_void_p(s.cuda_stream)) == 0
    try:
        with torch.cuda.stream(s):
            torch.cuda._sleep(SLEEP_CYCLES)
            for dst, src in ins:
                dst.copy_(src)
            rc = call(L)
            got = [o.clone() for o in outs]
            for o in outs[:3] if case == "mlkem_encaps_push" else outs:
                o.fill_(SENTINEL)
        s.synchronize()
    finally:
        L.cb200_set_stream(None)
        L.cb200_release_stream(C.c_void_p(s.cuda_stream))
    assert rc == 0, L.cb200_last_error()
    for i, (g, w) in enumerate(zip(got, want)):
        assert torch.equal(g, w), f"output {i} read before the call finished"
    for i, o in enumerate(outs[:3] if case == "mlkem_encaps_push" else outs):
        assert bool((o == SENTINEL).all()), f"output {i} written after the stream passed the call"
    if case == "mlkem_encaps_push":
        assert torch.equal(outs[3], want[0]) and torch.equal(outs[4], want[1])
