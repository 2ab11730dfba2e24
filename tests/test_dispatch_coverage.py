"""CPU side of tests/test_gpu_dispatch_coverage.py.

1. The coverage guard: the kernel instantiations the dispatchers can select are read out of the CUDA sources, and
   every one of them must be claimed by a parity case of the GPU file (and every claim must name a cell that exists
   and a case that exists).  A new instantiation without a parity case fails here, without a GPU.
2. The oracle those cases compare with, cross-checked against the independent numpy restatement at the new shapes:
   a (5,10) code with check degree 10 and an overcomplete code (m = 400 > n = 46, irregular checks), in exact and SFU
   arithmetic -- the same checks tests/test_oracle.py and tests/test_gnn_bp4.py run on the (3,6) codes."""
import os
import re

import numpy as np
import pytest

import test_gpu_dispatch_coverage as D

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "feedback-gnn_b200", "csrc")


def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _body(src, signature):
    """Text of the function whose definition starts with `signature` (up to its matching closing brace)."""
    i = src.index(signature)
    i = src.index("{", i)
    depth = 0
    for j in range(i, len(src)):
        depth += {"{": 1, "}": -1}.get(src[j], 0)
        if depth == 0:
            return src[i:j + 1]
    raise AssertionError(f"unbalanced braces after {signature!r}")


def _norm(s):
    return re.sub(r"\s+", "", s)


def dispatcher_cells():
    """Every kernel instantiation a dispatcher can select, in the spelling of CLAIMS."""
    bp, gnn, gbp = _source("fbgnn_bp.cu"), _source("fbgnn_gnn.cu"), _source("fbgnn_gbp.cu")
    cells = set()
    launch_bp4 = _body(bp, "int launch_bp4(fbgnn_ctx")
    cells |= {_norm(m) for m in re.findall(r"launch_bp4_m<[^>]*>(?=\()", launch_bp4)}
    cells |= {_norm(m) for m in re.findall(r"launch_bp4_gstate<[^>]*>(?=\()", launch_bp4)}
    cluster_d = _body(bp, "static int launch_bp4_cluster_d(")
    cells |= {f"launch_bp4_cluster_t<{n}>" for n in re.findall(r"launch_bp4_cluster_t<\s*\w+\s*,\s*\w+\s*,\s*(\d+)\s*>", cluster_d)}
    cells |= {_norm(m) for m in re.findall(r"launch_bp2_m<[^>]*>(?=\()", _body(bp, "int launch_bp2(fbgnn_ctx"))}
    launch_gnn = _body(gnn, "int launch_gnn(fbgnn_ctx")
    cells |= {_norm(m) for m in re.findall(r"launch_gnn_m<[^>]*>(?=\()", launch_gnn)}
    cells |= {_norm(m) for m in re.findall(r"(?:tc::)?k_gnn\w*<[^>]*>(?=<<<)", launch_gnn)}
    gbp_run = _body(gbp, "static int gbp_run(")
    cells |= {_norm(m) for m in re.findall(r"(?:tc::)?k_gbp\w*<[^>]*>(?=<<<)", gbp_run)}
    return cells


def test_extraction_finds_the_known_cells():
    """The regexes still see the dispatchers (a reformatted source must not make the guard vacuous)."""
    cells = dispatcher_cells()
    for c in ("launch_bp4_m<5,10>", "launch_bp4_m<0,0>", "launch_bp4_cluster_t<64>", "launch_bp4_gstate<MathSfu>",
              "launch_bp2_m<5,10>", "launch_gnn_m<64,32,0,false,false>", "k_gnn_deep<MathSfu>",
              "k_gbp_vn<20,40,20,MATH>", "tc::k_gbp_cn_tc<MATH>"):
        assert c in cells, c
    assert len(cells) >= 30


def test_every_dispatched_instantiation_has_a_parity_case():
    cells = dispatcher_cells()
    unclaimed = sorted(cells - set(D.CLAIMS))
    assert not unclaimed, f"kernel instantiations without a parity case in test_gpu_dispatch_coverage.py: {unclaimed}"
    stale = sorted(set(D.CLAIMS) - cells)
    assert not stale, f"CLAIMS names cells the dispatchers no longer select: {stale}"
    for cell, cases in D.CLAIMS.items():
        assert cases, cell
        for case in cases:
            assert callable(getattr(D, case, None)) and case.startswith("test_"), (cell, case)


def test_guard_catches_a_new_instantiation(monkeypatch):
    """A launch_bp4_m<6, 12> line added to the dispatcher is reported as unclaimed."""
    bp = _source("fbgnn_bp.cu")
    anchor = "    if (dv == 5 && dc == 10)"
    assert anchor in bp
    mutated = bp.replace(anchor, "    if (dv == 6 && dc == 12) return launch_bp4_m<6, 12>(ctx, a, grid, smem, threads, cp);\n" + anchor)
    real = _source
    monkeypatch.setitem(globals(), "_source", lambda name: mutated if name == "fbgnn_bp.cu" else real(name))
    assert "launch_bp4_m<6,12>" in dispatcher_cells() - set(D.CLAIMS)


# ------------------------------------------------------------------ routing restatement sanity (no GPU) ------------
def test_routing_of_the_coverage_codes(codes):
    import fbgnn as F
    import test_gpu_published as PUB
    assert D.bp4_cell(codes["c882"]) == "launch_bp4_m<3,6>" and D.bp4_cell(codes["gb48"]) == "launch_bp4_m<4,8>"
    gb254 = PUB._code(F, "GB_n254_k28", codes, None)
    oc = PUB._code(F, "GB_n46_k2_oc", codes, None)
    assert D.bp4_cell(gb254) == "launch_bp4_m<5,10>" and D.bp2_cell(gb254.hx) == "launch_bp2_m<5,10>"
    assert D.bp4_cell(oc) == "launch_bp4_m<0,0>" and D.max_node_degree(gb254) == 10
    # the [[7688,50]] (3,6) code of test_gpu_parity.py: over one SM, DCMAX = 8 in the cluster
    h = F.create_circulant_matrix(62, [0, 2, 5])
    big = F.hypergraph_product(h, h)
    assert D.bp4_state_bytes(big) > D.SMEM_OPTIN
    assert D.bp4_cell(big, large="cluster") == "launch_bp4_cluster_t<8>"
    assert D.bp4_cell(big, math="sfu") == "launch_bp4_gstate<MathSfu>"
    assert D.bp4_cell(big, early_stop=True) == "launch_bp4_gstate<MathExact>"


# ------------------------------------------------------------------ oracle cross-checks at the new shapes -----------
@pytest.fixture(scope="module")
def xcodes(codes, weights):
    import fbgnn as F
    import test_gpu_published as PUB
    c = dict(codes)
    c["GB_n254_k28"] = PUB._code(F, "GB_n254_k28", codes, None)
    c["GB_n46_k2_oc"] = PUB._code(F, "GB_n46_k2_oc", codes, None)
    return c


@pytest.fixture(params=["exact", "sfu"])
def arith(request, oracle, monkeypatch):
    """The oracle in each arithmetic; in SFU the cancellation bound of the teacher-forced check is doubled, as in
    tests/test_sfu_oracle.py."""
    import test_oracle as T
    oracle.set_math(request.param)
    if request.param == "sfu":
        monkeypatch.setattr(T, "_CANCEL", 8e-6)
    yield request.param
    oracle.set_math("exact")


NEW = ["GB_n254_k28", "GB_n46_k2_oc"]


@pytest.mark.parametrize("name", NEW)
@pytest.mark.parametrize("cn_type", ["boxplus-phi", "minsum", "boxplus"])
def test_c_oracle_vs_numpy_oracle_teacher_forced(oracle, xcodes, arith, name, cn_type, monkeypatch):
    """On the overcomplete code every qubit sits in about 87 checks per side: a variable-node sum of that many
    saturated messages (|S| up to ~1300) carries float32 rounding of ~1e-3 that depends on the summation order, and a
    check whose other inputs are saturated passes it on to a small outgoing message.  The noise model gets a relative
    term of that size there (measured worst case 3e-3); the (5,10) code keeps the model of tests/test_oracle.py."""
    import test_oracle as T
    if name.endswith("_oc"):
        tol = T._tol
        monkeypatch.setattr(T, "_tol", lambda ref, cn, got=None: tol(ref, cn, got) + 5e-3 * np.abs(ref))
    T.test_c_oracle_vs_numpy_oracle_teacher_forced(oracle, xcodes, None, name, cn_type)


@pytest.mark.parametrize("name", NEW)
def test_c_oracle_vs_numpy_oracle_gnn_and_bp2(oracle, xcodes, weights, arith, name):
    import test_oracle as T
    T.test_c_oracle_vs_numpy_oracle_gnn_and_bp2(oracle, xcodes, None, {name: weights["c882"]}, name)


@pytest.mark.parametrize("name", NEW)
@pytest.mark.parametrize("reduce_op", ["mean", "sum", "max", "min"])
def test_gnn_bp4_c_oracle_matches_numpy_restatement(oracle, xcodes, arith, name, reduce_op):
    import test_gnn_bp4 as G
    G.test_c_oracle_matches_numpy_restatement(oracle, xcodes, name, reduce_op)
