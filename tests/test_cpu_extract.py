"""CPU suite: extract.py's host logic around the kernels -- the eigensolver retry and the .pth layouts -- driven with
CPU tensors in place of device results."""
import numpy as np
import torch

from conftest import load_pkg


def _first_pass(B=5, K=3, N=8):
    g = torch.Generator().manual_seed(0)
    evals = torch.rand(B, K, generator=g).sort(dim=1).values
    evecs = torch.randn(B, K, N, generator=g)
    info = torch.tensor([[20, 1, 0, 0]] * B, dtype=torch.int32)
    return evals, evecs, info


def test_retry_replaces_converged_rows_and_reports_the_rest():
    """Rows 1, 2, 3 fail the first solve (1 and 2 did not converge, 3 has a NaN vector). On the retry row 1 converges,
    row 2 still does not, row 3 converges with finite vectors but a NaN eigenvalue: only row 1 is replaced."""
    ex = load_pkg("extract")
    evals, evecs, info = _first_pass()
    info[1, 1] = info[2, 1] = 0
    evecs[3, 2, 5] = float("nan")
    before = (evals.clone(), evecs.clone(), info.clone())
    calls = []

    def solve(rows, max_steps):
        calls.append((rows, max_steps))
        n = len(rows)
        ev = torch.arange(n * 3, dtype=torch.float32).reshape(n, 3) + 100.0
        vec = torch.full((n, 3, 8), 7.0) + torch.arange(n, dtype=torch.float32)[:, None, None]
        inf = torch.tensor([[7, 1, 0, 0]] * n, dtype=torch.int32)
        inf[rows.index(2), 1] = 0                    # row 2: still not converged
        ev[rows.index(3), 1] = float("nan")         # row 3: converged, finite vectors, NaN eigenvalue
        return ev, vec, inf

    replaced, failed, ev_new, vec_new = ex._retry_bad_rows(solve, evals, evecs, info)
    assert calls == [([1, 2, 3], 7)]                 # largest Krylov space: N - 1
    assert replaced == [1] and failed == [2, 3]
    assert torch.equal(ev_new, torch.tensor([[100.0, 101.0, 102.0]])) and torch.equal(vec_new, torch.full((1, 3, 8), 7.0))
    assert torch.equal(evals[1], ev_new[0]) and torch.equal(evecs[1], vec_new[0]) and info[1].tolist() == [7, 1, 0, 0]
    for i in (0, 2, 3, 4):                           # failed rows keep their first result; good rows are untouched
        assert torch.equal(evals[i], before[0][i]) and torch.equal(info[i], before[2][i])
        assert torch.equal(evecs[i].nan_to_num(), before[1][i].nan_to_num())


def test_retry_is_not_called_when_every_row_converged():
    ex = load_pkg("extract")
    evals, evecs, info = _first_pass()

    def solve(rows, max_steps):
        raise AssertionError("no row needs a retry")
    assert ex._retry_bad_rows(solve, evals, evecs, info) == ([], [], None, None)


def test_eigs_layout_saved_through_the_writer_helper(tmp_path):
    """which_matrix='affinity' keeps the reference's quirk (ascending numpy eigenvalues next to the descending
    eigenvectors the solver returned, vectors not flipped); 'laplacian' saves tensors that load with weights_only."""
    ex = load_pkg("extract")
    iop = load_pkg("io_pipeline")
    evals = torch.tensor([[3.0, 2.0, 0.5], [9.0, 4.0, 1.0]])            # descending, as the affinity solver returns them
    evecs = torch.randn(2, 3, 6, generator=torch.Generator().manual_seed(1))
    (tmp_path / "sub").mkdir()
    arrays, items = ex._eigs_batch(str(tmp_path), ["a", "sub/b"], evals, evecs, "affinity", skip=[0])
    assert [it[0] for it in items] == [str(tmp_path / "sub" / "b.pth")]
    for item in items:
        iop.save_item(arrays, item)
    assert sorted(p.name for p in (tmp_path / "sub").iterdir()) == ["b.pth"]   # the temporary file was renamed
    out = torch.load(tmp_path / "sub" / "b.pth", weights_only=False)
    assert set(out) == {"eigenvalues", "eigenvectors"}
    assert isinstance(out["eigenvalues"], np.ndarray) and out["eigenvalues"].tolist() == [1.0, 4.0, 9.0]
    assert torch.equal(out["eigenvectors"], evecs[1])
    arrays, items = ex._eigs_batch(str(tmp_path), ["a", "sub/b"], evals, evecs)
    iop.save_item(arrays, items[0])
    out = torch.load(tmp_path / "a.pth")
    assert torch.equal(out["eigenvalues"], evals[0]) and torch.equal(out["eigenvectors"], evecs[0])
