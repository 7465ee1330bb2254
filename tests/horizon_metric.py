"""Error metrics for comparing a kernel's [R, T', C] output with a reference, one horizon at a time.

One relative L2 over the whole tensor dilutes an error confined to a single time slot: at T' = 52 a slot is 1/52 of the
elements, so a 5 % error in one slot moves the global figure by well under 1 %.  Tile, halo and level-offset bugs of the
denoiser and the LSTM kernels are confined to single slots (the last tile of a level, the seam between two half-horizon
lanes), so the tests also take the worst slot and the worst row."""
import torch


def rel(a, b):
    """Relative L2 of `a` against `b` over all elements (float64)."""
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def worst_row_rel(got, want):
    """Largest relative L2 of any single row (first dimension), taken over everything else in the row."""
    got, want = torch.as_tensor(got).double().cpu(), torch.as_tensor(want).double().cpu()
    R = want.shape[0]
    d = (got.reshape(R, -1) - want.reshape(R, -1)).norm(dim=1)
    return (d / (want.reshape(R, -1).norm(dim=1) + 1e-30)).max().item()


def worst_slot_rel(got, want, t_slots):
    """Reshapes both to [R, t_slots, C] and returns the largest relative L2 of any single time slot, taken over rows and
    channels."""
    got, want = torch.as_tensor(got).double().cpu(), torch.as_tensor(want).double().cpu()
    R = want.shape[0]
    g, w = got.reshape(R, t_slots, -1), want.reshape(R, t_slots, -1)
    d = (g - w).transpose(0, 1).reshape(t_slots, -1).norm(dim=1)
    n = w.transpose(0, 1).reshape(t_slots, -1).norm(dim=1)
    return (d / (n + 1e-30)).max().item()
