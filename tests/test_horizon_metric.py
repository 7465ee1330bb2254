"""CPU: the per-slot metric of the horizon tests sees an error confined to one time slot that the global relative L2 of the
same tensors does not."""
import torch

import cld_oracle as O
from horizon_metric import rel, worst_row_rel, worst_slot_rel

BF16_TOL = 1e-2          # global bound of the bf16 denoiser tests
SLOT_TOL = 3e-2          # worst-slot bound of the same tests


def test_one_wrong_slot_passes_the_global_bound_but_not_the_slot_bound(models_cpu):
    dm, _, _ = models_cpu(10)
    sd = {k: v.detach() for k, v in dm.model.state_dict().items()}
    torch.manual_seed(0)
    R = 8
    x, cond, t = torch.randn(R, 52, 4), torch.randn(R, 256), torch.randint(0, 10, (R,))
    taps = {}
    with torch.no_grad():
        O.unet_forward(sd, x, cond, t, taps=taps)
    want = taps["downs.0.1"]
    assert want.shape == (R, 52, 64)
    assert rel(want, want) == 0.0 and worst_slot_rel(want, want, 52) == 0.0 and worst_row_rel(want, want) == 0.0
    got = want.clone()
    got[:, 51] *= 1.05                               # the last slot: the one the overlapping last tile of level 0 writes
    g, s, r = rel(got, want), worst_slot_rel(got, want, 52), worst_row_rel(got, want)
    print("one slot of 52 off by 5 %%: global %.3e, worst slot %.3e, worst row %.3e" % (g, s, r))
    assert g < BF16_TOL
    assert s > SLOT_TOL
    assert abs(s - 0.05) < 1e-6                      # the slot's own error, undiluted (fp32 rounding of the scaling)
    # the metric takes [R, T', C] in the row-major layout of the kernels' outputs: a flattened [R, T'*C] tensor gives the same
    assert worst_slot_rel(got.reshape(R, -1), want.reshape(R, -1), 52) == s


def test_worst_slot_is_the_largest_over_slots():
    torch.manual_seed(1)
    want = torch.randn(5, 12, 3)
    got = want.clone()
    got[:, 3] += 0.01 * want[:, 3]
    got[:, 7] += 0.02 * want[:, 7]
    assert abs(worst_slot_rel(got, want, 12) - 0.02) < 1e-6
    got[2] = want[2] * 1.5
    assert abs(worst_row_rel(got, want) - 0.5) < 1e-6
