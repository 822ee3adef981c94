"""CPU: the C-ABI library loads (no GPU needed) and exports every symbol include/tarok_b200.h declares."""
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "tarok_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tarok_[a-z0-9_]+)\s*\(", src)))


def test_library_is_built_and_exports_every_declared_symbol():
    import __graft_entry__ as G
    G.build()
    from tarok_b200 import _lib
    lib = _lib.load()
    names = _declared()
    assert len(names) >= 25
    for nm in names:
        assert hasattr(lib, nm), "libtarok_b200.so does not export %s" % nm
    assert set(names) == set(_lib.SIGNATURES), set(names) ^ set(_lib.SIGNATURES)


NO_DEVICE = r'''
import sys
sys.path.insert(0, %r)
from tarok_b200 import _lib
from tarok_b200.env import TarokEnv
try:
    TarokEnv(16)
except _lib.TarokLibraryError as ex:
    print(ex)
else:
    sys.exit("TarokEnv was created without a CUDA device")
'''


def test_no_gpu_fails_loudly_not_silently():
    """Without a CUDA device tarok_create must return an error (there is no CPU fallback).  Checked in a child process that
    sees no device (empty CUDA_VISIBLE_DEVICES), so that it runs on machines with a GPU as well."""
    out = subprocess.run([sys.executable, "-c", NO_DEVICE % ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "no CUDA device" in out.stdout or "CUDA" in out.stdout


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "tarok_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "oracle" not in txt.replace("the oracle", "").replace("oracle's", "") or f == "README.md", \
                    "%s mentions the oracle" % f


def test_c_consumer_compiles_against_the_header():
    """A plain-C program builds against include/tarok_b200.h and links the shared library (no GPU needed to link)."""
    import subprocess
    import tempfile
    import __graft_entry__ as G
    G.build()
    exe = os.path.join(tempfile.mkdtemp(), "c_abi_demo")
    cmd = ["/usr/bin/gcc", "-O2", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"),
           os.path.join(ROOT, "examples", "c_abi_demo.c"), "-o", exe, "-L" + os.path.join(ROOT, "tarok_b200"),
           "-ltarok_b200", "-Wl,-rpath," + os.path.join(ROOT, "tarok_b200")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    import torch
    out = subprocess.run([exe, "200000"], capture_output=True, text=True, timeout=120)
    if torch.cuda.is_available():
        assert out.returncode == 0, out.stdout + out.stderr
        assert 199900 <= int(out.stdout.split()[1]) <= 200000 and "kernel launches: 51" in out.stdout     # one graph replay: hand-over kernel + setup + 48 play_steps + score
    else:       # no GPU here: the program must fail loudly, not fall back
        assert out.returncode == 1 and "no CUDA device" in out.stderr


@pytest.mark.gpu
def test_c_consumer_runs_on_the_gpu():
    test_c_consumer_compiles_against_the_header()


def test_pack_records_is_the_documented_layout():
    """Host-side serialiser (CPU code in the library): decode the bit planes in numpy and compare with the rows."""
    import numpy as np
    from tarok_b200.env import pack_records
    rng = np.random.default_rng(3)
    n = 2000
    perm = np.stack([rng.permutation(54) for _ in range(n)]).astype(np.uint8)
    contract = rng.integers(0, 10, n).astype(np.uint8)
    declarer = rng.integers(0, 4, n).astype(np.uint8)
    king = rng.integers(0, 4, n).astype(np.uint8)
    rec, bad = pack_records(perm, contract, declarer, king)
    assert bad == 0
    raw = rec.numpy()
    assert raw.shape == (n, 20) and raw.dtype == np.uint8
    for g in range(n):
        w0 = int.from_bytes(raw[g, 0:8].tobytes(), "little")
        w1 = int.from_bytes(raw[g, 8:16].tobytes(), "little")
        w2 = int.from_bytes(raw[g, 16:20].tobytes(), "little")
        m = (w0 >> 54) | (w1 >> 54) << 10 | w2 << 20
        w0 &= (1 << 54) - 1; w1 &= (1 << 54) - 1
        assert m >> 45 == 0
        talon = [(m >> (6 * i)) & 63 for i in range(6)]
        assert talon == perm[g, 48:].tolist()
        code = [((w0 >> c) & 1) | ((w1 >> c) & 1) << 1 for c in range(54)]
        assert all(code[c] == 0 for c in talon)
        for s in range(4):
            assert sorted(c for c in range(54) if code[c] == s and c not in talon) == sorted(perm[g, 12 * s:12 * s + 12].tolist())
        assert (m >> 36) & 15 == contract[g]
        assert (m >> 40) & 3 == declarer[g]
        assert (m >> 42) & 7 == king[g]
    perm[0, 0] = perm[0, 1]
    assert pack_records(perm, contract, declarer, None)[1] == 1


def test_pack_records_vector_and_scalar_serialisers_agree():
    """The AVX-512 serialiser (taken at run time where the CPU has it) and the scalar one produce identical records and reject
    the same rows: duplicates, ids 54..63, ids >= 64, out-of-range contract / declarer -- also on several threads and on the
    very last row of a buffer (the vector code must not read past it)."""
    import numpy as np
    from tarok_b200 import _lib
    from tarok_b200.env import pack_records
    lib = _lib.load()
    rng = np.random.default_rng(11)
    n = 50021
    perm = np.stack([rng.permutation(54) for _ in range(n)]).astype(np.uint8)
    contract = rng.integers(0, 10, n).astype(np.uint8)
    declarer = rng.integers(0, 4, n).astype(np.uint8)
    king = rng.integers(0, 8, n).astype(np.uint8)
    perm[5, 3] = perm[5, 4]                     # duplicate inside a hand
    perm[77, 50] = 60                           # id 54..63 in the talon
    perm[99, 0] = 200                           # id >= 64
    perm[100, 47], perm[100, 48] = 53, 53       # duplicate across hand and talon
    perm[101, 49] = 130                         # id >= 64 in the talon
    perm[n - 1, 53] = perm[n - 1, 52]           # the last row
    contract[11] = 99
    declarer[12] = 7
    out = {}
    prev = lib.tarok_pack_force_scalar(0)
    try:
        for scalar in (0, 1):
            lib.tarok_pack_force_scalar(scalar)
            for threads in (1, 3):
                rec, bad = pack_records(perm, contract, declarer, king, threads=threads)
                out[(scalar, threads)] = (rec.numpy().copy(), bad)
        lib.tarok_pack_force_scalar(0)
        import torch
        for shift in (0, 4, 20, 33):             # 64-byte aligned output (non-temporal stores) and three unaligned ones
            buf = torch.zeros(n * 20 + 128, dtype=torch.uint8)
            off = (-buf.data_ptr() % 64) + shift
            view = buf[off:off + n * 20].view(n, 20)
            rec, bad = pack_records(perm, contract, declarer, king, out=view, threads=2)
            out[("vector, output shifted", shift)] = (rec.numpy().copy(), bad)
    finally:
        lib.tarok_pack_force_scalar(prev)
    ref, bad = out[(1, 1)]
    assert bad == 8
    for k, (rec, b) in out.items():
        assert b == bad and np.array_equal(rec, ref), k


def test_pack_pool_and_tapered_chunks_without_a_gpu(tmp_path):
    """The host half of tarok_rollout_host_packed -- tapered upload chunks, the block-scheduled pack pool whose chunks complete
    in order while later ones are still being packed -- compiled from the library's own source into a plain C++ harness
    and compared with the single-threaded serialiser (ragged sizes, 1..4 threads, 1..29 chunks, one invalid row)."""
    exe = str(tmp_path / "harness")
    cmd = ["g++", "-O2", "-std=c++17", "-pthread", os.path.join(ROOT, "tests", "host_pool_harness.cpp"),
           os.path.join(ROOT, "tarok_b200", "csrc", "tarok_host.cpp"), "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    for rows, threads in ((300007, 4), (1 << 18, 3), (5000, 2), (1, 1), (2049, 4), (700001, 1)):
        out = subprocess.run([exe, str(rows), str(threads)], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0 and out.stdout.startswith("ok"), (rows, threads, out.stdout, out.stderr)
