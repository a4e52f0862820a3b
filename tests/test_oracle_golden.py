"""The oracle (oracle/krylov_oracle.py) against the golden vectors produced by the unmodified reference
(oracle/pin_reference.py).  CPU only.  Bit-exact where the arithmetic is the same torch build; 1e-12 otherwise."""
import os

import pytest
import torch

from conftest import build_matrix, load_case, rel_diff
from oracle import krylov_oracle as orc

SLOW = {"gmres_ldc100_step0_incremental", "gmres_ldc100_step1_batched"}


@pytest.fixture(autouse=True)
def golden_threads(manifest):
    """torch's CPU reductions split their sums by the number of threads, so the oracle reproduces the reference's bits
    only with the thread count the goldens were pinned with, whatever the cores of the machine running the tests."""
    saved = torch.get_num_threads()
    torch.set_num_threads(manifest["torch_threads"])
    yield
    torch.set_num_threads(saved)


def _case_names():
    import json
    from conftest import GOLD
    with open(GOLD / "manifest.json") as f:
        return sorted(json.load(f)["cases"].keys())


@pytest.mark.parametrize("name", _case_names())
def test_oracle_matches_reference_golden(name, manifest):
    if name in SLOW and not os.environ.get("BK_SLOW_TESTS"):
        pytest.skip("slow oracle case (set BK_SLOW_TESTS=1)")
    entry = manifest["cases"][name]
    data = load_case(name)
    A = build_matrix(entry["gen"])
    n = entry["n"]
    if "b" in data:
        b = data["b"]
    else:  # digest cases: b = ones or manufactured
        if "rand" in name:
            from pytorch_sparse_solver import problems
            b, _ = problems.manufactured_rhs(A, 0)
        else:
            b = torch.ones(n, dtype=torch.float64)
    x0 = data.get("x0")
    kw = dict(entry["kwargs"])
    if entry.get("jacobi"):
        from pytorch_sparse_solver import problems
        d = problems.csr_diagonal(A)
        kw["M"] = lambda r: r / d
    x, info, stats = getattr(orc, entry["kind"])(A, b, x0, **kw)
    assert info == entry["info"]
    assert stats["matvecs"] + 1 == entry["matvecs_ref"]
    assert stats["iterations"] == entry["iterations"]
    if "x" in data:
        if torch.__version__ == manifest["torch"]:
            assert torch.equal(x, data["x"])
        else:
            assert rel_diff(x, data["x"]) <= 1e-12
    else:
        idx = data["x_sample_idx"]
        assert rel_diff(x[idx], data["x_sample"]) <= 1e-12
        assert abs(float(torch.linalg.norm(x)) - entry["x_norm"]) <= 1e-12 * entry["x_norm"]


@pytest.mark.parametrize("kind", ["cg", "bicgstab", "gmres"])
def test_oracle_adjoint_matches_reference_autograd(kind, manifest):
    entry = manifest["autograd"][f"autograd_{kind}"]
    data = load_case(f"autograd_{kind}")
    A = build_matrix(entry["gen"])
    x, info, _ = getattr(orc, kind)(A, data["b"], None, **entry["kwargs"])
    g = orc.adjoint_grad_b(kind, A, 2.0 * x, None, **entry["kwargs"])
    assert rel_diff(g, data["grad_b"]) <= 1e-12
    assert rel_diff(x, data["x"]) <= 1e-12


def test_oracle_adjoint_ldc_gmres(manifest):
    entry = manifest["autograd"]["autograd_gmres_ldc32"]
    data = load_case("autograd_gmres_ldc32")
    A = build_matrix(entry["gen"])
    x, info, _ = orc.gmres(A, data["b"], None, **entry["kwargs"])
    g = orc.adjoint_grad_b("gmres", A, 2.0 * x, None, **entry["kwargs"])
    assert info == entry["info"] and rel_diff(g, data["grad_b"]) <= 1e-12 and rel_diff(x, data["x"]) <= 1e-12


def test_oracle_tolerance_quirk_fp32():
    """torch.tensor(tol) is fp32 (reference :816): 1e-8 -> 9.99999993922529e-09, squared in fp32."""
    t = torch.tensor(1e-8)
    assert float(t) == pytest.approx(9.99999993922529e-09, rel=0, abs=1e-24)
    assert float(torch.square(t)) == pytest.approx(1.0000000168623835e-16, rel=1e-15)
