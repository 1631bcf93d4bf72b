"""The staging chunk sizes that tests/test_gpu_batch_paths.py sizes its batches by must be the ones in csrc/.

Those GPU tests pick 4C + 1 and 6C + 13 operations so that a host batch reuses every staging slot and runs the ramp
chunks.  If a chunk size changed and the table did not, the same tests would quietly run inside one or two chunks;
this CPU test fails instead.
"""
import importlib.util
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "circl_b200", "csrc")


def _table_module():
    spec = importlib.util.spec_from_file_location("_batch_paths_table",
                                                  os.path.join(ROOT, "tests", "test_gpu_batch_paths.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


T = _table_module()


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _eval(expr, consts):
    expr = re.sub(r"(\d+)u\b", r"\1", expr.strip())
    for k, v in consts.items():
        expr = expr.replace(k, str(v))
    assert re.fullmatch(r"[\d\s<>()]+", expr), expr
    return eval(expr, {"__builtins__": {}})


def _body(src, fn):
    """Source text from the definition of fn (the last one, after any forward declaration) onwards."""
    starts = [m.start() for m in re.finditer(r"^(?:static )?int " + re.escape(fn) + r"\(", src, re.M)]
    assert starts, fn
    return src[starts[-1]:]


CHUNK_RE = re.compile(r"hc\.chunk = ([^;]+);|run_host\(bufs, n, ([^,]+),|constexpr size_t kChunk = ([^;]+);")


def test_slot_count():
    m = re.search(r"static constexpr int kSlots = (\d+);", _src("context.h"))
    assert m and int(m.group(1)) == T.SLOTS["staged"]
    sign = _body(_src("mldsa.cu"), "cb200_mldsa_sign")
    m = re.search(r"const int nslots = nchunks < (\d+) \? \(int\)nchunks : (\d+);", sign)
    assert m and int(m.group(1)) == int(m.group(2)) == T.SLOTS["sign"]
    assert re.search(r"const int sl = \(int\)\(ci % " + str(T.SLOTS["sign"]) + r"\);", sign)
    verify = _body(_src("mldsa.cu"), "cb200_mldsa_verify")
    assert "cudaStream_t st = c.pipe[0];" in verify.split("constexpr size_t kChunk")[0]


@pytest.mark.parametrize("entry,src,fn,chunk,pipeline", T.CHUNK_TABLE, ids=[e[0] for e in T.CHUNK_TABLE])
def test_chunk_table_matches_sources(entry, src, fn, chunk, pipeline):
    api = _src("api.cu")
    consts = {"kPolyChunk": _eval(re.search(r"static constexpr size_t kPolyChunk = ([^;]+);", api).group(1), {})}
    m = CHUNK_RE.search(_body(_src(src), fn))
    assert m, f"no chunk size found in {fn}"
    expr = next(g for g in m.groups() if g)
    if entry in T.PER_K:
        assert expr.replace(" ", "").endswith("/k"), expr
        expr = expr.replace(" ", "")[:-2]
    assert _eval(expr, consts) == chunk
    assert (pipeline == "staged") == (m.group(3) is None)  # run_staged, or a pipeline of its own


@pytest.mark.parametrize("entry", [e[0] for e in T.CHUNK_TABLE if e[4] == "staged"])
def test_sizes_reuse_every_slot_and_run_the_ramp(entry):
    c = T.chunk_of(entry)
    s4 = T.schedule(T.SIZES["4C+1"](c), c)
    assert len(s4) == 5 and s4[-1][1:] == (1, 0)  # the fifth chunk: one row, back in slot 0
    n6 = T.SIZES["6C+13"](c)
    s6 = T.schedule(n6, c)
    assert [x[1] for x in s6] == [c // 4, c // 4, c // 2, c, c, c, c, 13, c // 2, c // 4, c // 4]
    assert [x[2] for x in s6] == [i % 4 for i in range(11)] and sum(x[1] for x in s6) == n6


def test_dot_product_chunk_is_not_a_multiple_of_four():
    c = T.chunk_of("cb200_kyber_dot", 3)
    assert c == 43690
    assert [x[1] for x in T.schedule(6 * c + 13, c)[:3]] == [10922, 10922, 21845]


def test_sign_and_verify_sizes_reuse_their_slots():
    c = T.chunk_of("cb200_mldsa_sign")
    s = T.schedule(3 * c + 5, c, "sign")
    assert [x[1:] for x in s] == [(c, 0), (c, 1), (c, 2), (5, 0)]
    v = T.chunk_of("cb200_mldsa_verify")
    assert [x[1] for x in T.schedule(2 * v + 3, v, "verify")] == [v, v, 3]


def test_boundary_rows():
    assert T.boundary_rows(10, 4) == [0, 1, 2, 3, 4, 5, 6, 7, 8, 9]
    rows = T.boundary_rows(4 * 4096 + 1, 4096)
    assert {0, 1, 4094, 4095, 4096, 4097, 16383, 16384} <= set(rows) and 2048 not in rows
