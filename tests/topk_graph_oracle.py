"""The pattern selection of the sparse graph generator (`pair_topk`, `gen(X_seq, k=k)`), restated in fp64 on the CPU --
test infrastructure, like oracle/.

S[n, m] = <U_n, V_m> - <V_n, U_m> for every m, with S[n, n] = 0 exactly; row n keeps the k columns with the largest
S[n, m], equal scores going to the smaller column, stored in ascending column order.  The full [N, N] score matrix is
formed here: fine at test sizes, and exactly what the CUDA path avoids."""
import torch

Tensor = torch.Tensor


def full_scores(U: Tensor, V: Tensor, rows: Tensor = None) -> Tensor:
    """S [N, N] (or the listed rows [len(rows), N]) in U's dtype, the diagonal exactly 0."""
    idx = torch.arange(U.shape[0], device=U.device) if rows is None else rows.long().to(U.device)
    S = U[idx] @ V.t() - V[idx] @ U.t()
    S[torch.arange(idx.numel(), device=U.device), idx] = 0
    return S


def select(S: Tensor, k: int) -> Tensor:
    """[R, k] int64: per row the k columns with the largest S (ties: the smaller column), ascending.  A stable sort of -S
    keeps equal scores in column order."""
    order = torch.sort(-S, dim=1, stable=True).indices[:, :k]
    return torch.sort(order, dim=1).values


def kth_margin(S: Tensor, k: int, rel: float = 1e-5):
    """(t, tau) per row: t the k-th largest score, tau = rel * max|S_row|.  A selection is right at rows where every
    column with S > t + tau is selected and none with S < t - tau."""
    t = torch.sort(S, dim=1, descending=True).values[:, k - 1]
    return t, rel * S.abs().amax(dim=1)


def check_selection(S: Tensor, cols: Tensor, k: int, rel: float = 1e-5):
    """Checks `cols` ([R, k], from the device) against the margin rule of `kth_margin`; returns the number of near-tie
    rows (a column within tau of t exists besides the k-th).  Raises AssertionError naming the first wrong row."""
    cols = cols.long().to(S.device)
    R, N = S.shape
    assert cols.shape == (R, k), cols.shape
    assert torch.all(cols[:, 1:] > cols[:, :-1]), "columns are not strictly ascending in every row"
    assert int(cols.min()) >= 0 and int(cols.max()) < N
    t, tau = kth_margin(S, k, rel)
    chosen = torch.zeros(R, N, dtype=torch.bool, device=S.device)
    chosen.scatter_(1, cols, True)
    must = S > (t + tau)[:, None]
    mustnt = S < (t - tau)[:, None]
    bad = (must & ~chosen).any(1) | (mustnt & chosen).any(1)
    if bad.any():
        r = int(bad.nonzero()[0, 0])
        raise AssertionError(f"row {r}: selected {cols[r].tolist()}, fp64 selection {select(S[r:r + 1], k)[0].tolist()}")
    near = ((S - t[:, None]).abs() <= tau[:, None]).sum(1) > 1
    return int(near.sum())
