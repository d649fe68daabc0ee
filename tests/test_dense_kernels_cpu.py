"""The instance table of tests/test_dense_kernels_gpu.py against the launchers' sources (no GPU needed): every dense
kernel instance the library compiles is run by some parametrization there, and the table's rules are the launchers'."""
import os
import re

import numpy as np

from tests import test_dense_kernels_gpu as G

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "physicsbasedbayesianinference_b200",
                    "csrc")


def source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def compiled_k_dense():
    """(kernel, dtype, TN, MINB) of every k_dense instance launch_dense reaches (csrc/inst_dense.cuh, instantiated for
    float and double by inst_dense_f32.cu / inst_dense_f64.cu).  MINB > 1 sits behind the float-only occupancy switch."""
    src = source("inst_dense.cuh")
    body = src[src.index("int launch_dense(ehmc_ctx* c"):]
    body = body[:body.index("\n}\n")]
    assert "const bool two = sizeof(T) == 4 && c->dense_occupancy >= 2;" in body
    assert "if constexpr (sizeof(T) == 4) {" in body
    pairs = {(int(tn), int(mb)) for tn, mb in re.findall(r"launch_dense_tn<T, (\d+), (\d+)>", body)}
    assert pairs, "no launch_dense_tn instances found"
    assert "template int launch_dense<float>" in source("inst_dense_f32.cu")
    assert "template int launch_dense<double>" in source("inst_dense_f64.cu")
    out = set()
    for tn, mb in pairs:
        for dt in ("float32", "float64"):
            if mb == 1 or dt == "float32":
                out.add(("k_dense", dt, tn, mb))
    return out


def compiled_tc3():
    src = source("inst_dense_tc3.cu")
    cases = re.findall(r"case (\d+): return launch_tc3_c8<(\d+)>", src)
    assert cases and all(a == b for a, b in cases)
    return {("k_dense_tc3", "float32", int(c)) for c, _ in cases}


def test_dense_tn_matches_launcher():
    """dense_tn in the table is csrc/inst_dense_f32.cu's rule at every D the dense kernels serve."""
    m = re.search(r"int dense_tn\(int D\) \{ return (.*?); \}", source("inst_dense_f32.cu"))
    assert m, "dense_tn not found"
    steps = [(int(d), int(t)) for d, t in re.findall(r"D <= (\d+) \? (\d+)", m.group(1))]
    last = int(re.search(r": (\d+)$", m.group(1)).group(1))
    for D in range(17, 129):
        want = next((t for d, t in steps if D <= d), last)
        assert G.dense_tn(D) == want, D


def test_tc3_shape_rule():
    """C8 = ceil(D / 8) (pack_dense_tc3), and the tensor-core kernel serves every D the dense kernels serve."""
    assert "C8 = (D + 7) / 8" in source("inst_dense_tc3.cu")
    assert {G.tc3_c8(D) for D in range(17, 129)} == {i[2] for i in compiled_tc3()}


def test_every_instance_is_parametrized():
    """Every (kernel, dtype, TN, MINB) and every C8 the library compiles appears in the GPU file's cases, and no case
    names an instance that does not exist."""
    ran = {G.instance(c) for c in G.CASES}
    compiled = compiled_k_dense() | compiled_tc3()
    assert compiled - ran == set(), f"instances no test runs: {sorted(compiled - ran)}"
    assert ran - compiled == set(), f"cases for instances that do not exist: {sorted(ran - compiled)}"


def test_case_shapes():
    """The D values sit on each kernel's edges: k_dense at every TN edge in float32 (both occupancies at TN = 13) and
    float64; k_dense_tc3 with a full and a partly padded last chunk per C8, every padding width and every D mod 4."""
    kd = {(np.dtype(dt).name, D, occ) for k, dt, D, occ in G.CASES if k == "k_dense"}
    for D in (17, 32, 33, 64, 65, 104, 105, 128):
        assert ("float64", D, 2) in kd and ("float32", D, 2) in kd
        if G.dense_tn(D) == 13:
            assert ("float32", D, 1) in kd
    tc = [D for k, _, D, _ in G.CASES if k == "k_dense_tc3"]
    for c8 in range(3, 17):
        assert 8 * c8 in tc
        assert any(8 * c8 - 8 < D < 8 * c8 for D in tc), c8
    assert {D % 4 for D in tc} == {0, 1, 2, 3}
    assert {(8 - D % 8) % 8 for D in tc} == set(range(8))  # padding dims in the last chunk: 0 .. 7
    assert len(set(G.case_id(c) for c in G.CASES)) == len(G.CASES)


def test_schedule_model():
    """The tile schedule the persistent-scheduling test reasons with: contiguous tile ranges per CTA, alternating
    groups; every tile is dealt once."""
    S = 148
    for T in (1, S - 1, S, S + 1, 2 * S + 1, 5 * S + 3):
        P = 128 * (T - 1) + 1 + (37 * T) % 127
        assert G.tc3_tiles(P) == T and P % 128 != 0
        sched = G.tc3_schedule(P, S)
        assert sorted(sched) == list(range(T))
        counts = {}
        for b, g in sched.values():
            counts[(b, g)] = counts.get((b, g), 0) + 1
        assert max(counts.values()) - min(counts.values()) <= 2
