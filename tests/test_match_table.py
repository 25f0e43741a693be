"""k_match's per-position match table against match_search() of b200z_core.cuh, entry for entry.

The parse only reads the table, so a wrong entry can hide behind a parse that never visits its position; here every
(A, B) entry of every data position is compared, over the data and the hash-chain links the plan's SEARCH stage used.
The GPU tier runs it on the device; the CPU tier runs the same tests on the CUDA emulator (tests/cuda_emu)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import crafted_t8
from sharpziplib_b200 import datagen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K_MAX_DIST = 32506
K_SLIDE_FIRST = 65273


def _cases():
    """(name, history bytes, data bytes, pos_base or None); pos_base makes the stream a continuation whose window has seen
    pos_base bytes before its data, which moves the SlideWindow phase (trap T8) into the data"""
    rng = datagen.Rng(0x3A7C)
    out = [("run_of_one_byte", b"", bytes([7]) * 40000, None)]
    # period-d repeats: every position's first candidate is at distance d (or a multiple), the match runs to the 258 cap
    for d in (1, 2, 3, 257, 258, 259, K_MAX_DIST - 1, K_MAX_DIST, K_MAX_DIST + 1):
        block = rng.bytes(d).tobytes()
        n = max(6000, 2 * d + 3000)
        out.append(("period_%d" % d, b"", (block * (n // d + 1))[:n], None))
    # streams whose every position has maxlen < 10, and a repeat that runs into the end of the stream
    for n in range(3, 14):
        out.append(("tail_abc_%d" % n, b"", (b"abc" * 5)[:n], None))
    out.append(("tail_run_12", b"", b"a" * 12, None))
    # one tile, the tile boundary, multi-tile
    for i, n in enumerate((32767, 32768, 32769, 100000)):
        out.append(("mix_%d" % n, b"", datagen.silesia_mix(i, n, config=9).tobytes(), None))
    out.append(("t8", b"", crafted_t8(), None))
    text = datagen.gen_text(120000, 5).tobytes()
    out.append(("dictionary_5000", text[:5000], text[60000:90000], None))
    out.append(("dictionary_32506", text[:K_MAX_DIST], text[40000:50000], None))
    # continuations: a slide position inside the data, once on text and once where the only candidate sits at 32506
    out.append(("continue_text_slide", text[:1000], text[30000:70000], 1000 + K_SLIDE_FIRST - 33000))
    block = rng.bytes(K_MAX_DIST).tobytes()
    out.append(("continue_period_32506_slide", text[:2000], (block * 3)[:70000], 2000 + K_SLIDE_FIRST - 40000))
    return out


@pytest.fixture(scope="module")
def ref(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("match_ref") / "libmatch_ref.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", os.path.join(ROOT, "sharpziplib_b200", "csrc"),
                           "-o", so, os.path.join(ROOT, "tests", "cpu_model", "match_ref.cpp")])
    M = C.CDLL(so)
    M.ref_match_table.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p]
    return M


def _run_search(z, cases, level):
    """one plan over all cases, SEARCH stage only; returns [(links, table)] per case"""
    import torch
    from sharpziplib_b200 import _lib
    from sharpziplib_b200.batch import _Plan
    L = _lib.lib()
    lens = np.array([len(d) for _, _, d, _ in cases], dtype=np.int64)
    hist = np.array([len(h) for _, h, _, _ in cases], dtype=np.int64)
    pos_base = np.array([len(h) if pb is None else pb for _, h, _, pb in cases], dtype=np.int64)
    kind = _lib.HIST_CONTINUE if cases[0][3] is not None else _lib.HIST_DICTIONARY
    hs = _lib.History(kind, 0, hist.ctypes.data, pos_base.ctypes.data if kind == _lib.HIST_CONTINUE else None, None, None)
    h = C.c_void_p()
    _lib.raise_for(L.b200z_deflate_plan_create_ex(lens.size, lens.ctypes.data, level, 0, _lib.WRAP_RAW, _lib.END_FINISH,
                                                  C.addressof(hs), C.byref(h)))
    plan = _Plan(h, lens.size)
    blob = np.zeros(plan.in_bytes, np.uint8)
    for o, (_, hb, db, _) in zip(plan.in_offsets, cases):
        blob[o:o + len(hb) + len(db)] = np.frombuffer(hb + db, np.uint8)
    d_in = torch.from_numpy(blob).cuda()
    d_out = torch.zeros(plan.out_bytes, dtype=torch.uint8, device="cuda")
    d_len = torch.zeros(plan.n, dtype=torch.int64, device="cuda")
    d_st = torch.ones(plan.n, dtype=torch.int32, device="cuda")
    plan.run(d_in, d_out, d_len, d_st, stages=_lib.STAGE_SEARCH)
    res = []
    for i in range(plan.n):
        link = np.zeros(int(hist[i] + lens[i]), np.uint16)
        tab = np.zeros(2 * int(lens[i]), np.uint32)
        _lib.raise_for(L.b200z_plan_get_match_table(plan._h, i, link.ctypes.data, tab.ctypes.data,
                                                    torch.cuda.current_stream().cuda_stream))
        res.append((link, tab))
    plan.close()
    return res


def _fmt(e):
    return "0" if e == 0 else "len %d dist %d" % (e >> 16, e & 0xFFFF)


def _check(z, ref, level, cases):
    bad = []
    plain = [c for c in cases if c[3] is None]
    cont = [c for c in cases if c[3] is not None]
    for (name, hb, db, pb), (link, tab) in zip(plain + cont, _run_search(z, plain, level) + _run_search(z, cont, level)):
        data = np.frombuffer(hb + db, np.uint8)
        H = len(hb)
        bias = (len(hb) if pb is None else pb) - H
        want = np.zeros_like(tab)
        ref.ref_match_table(data.ctypes.data, link.ctypes.data, data.size, H, bias, level, want.ctypes.data)
        diff = np.nonzero(tab != want)[0]
        if diff.size:
            rows = sorted(set(int(k) // 2 for k in diff[:8]))
            bad.append("%s (%d entries differ): " % (name, diff.size) + "; ".join(
                "position %d: kernel (A %s, B %s), match_search (A %s, B %s)" % (
                    H + r, _fmt(tab[2 * r]), _fmt(tab[2 * r + 1]), _fmt(want[2 * r]), _fmt(want[2 * r + 1])) for r in rows))
    assert not bad, "level %d:\n" % level + "\n".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("level", [5, 6, 7, 8, 9])
def test_match_table_equals_match_search(z, ref, level):
    _check(z, ref, level, _cases())


def test_match_table_on_the_emulator():
    """the GPU-tier tests above, with the unmodified kernel sources on the CUDA emulator (in a subprocess: the emulator
    library never shares a process with tests of the real one)"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "cuda_emu", "run_emulated.py"), __file__], capture_output=True,
                       text=True, timeout=2400)
    assert r.returncode == 0, (r.stdout[-4000:], r.stderr[-4000:])
