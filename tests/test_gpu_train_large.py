"""GPU (-m gpu): the denoiser training step (cld_unet_train_forward / cld_unet_backward / cld_ppo_grad) at the row counts where its
kernels switch tiles and reduction paths.  The other training tests stay at <= 37 rows; the choices below exist only for large batches:

  * GroupNorm forward / backward with one warp per group (gn_mish_fwd_mw_kernel<1>, gn_mish_bwd_kernel<1>) above 2 x SMs rows;
  * the two-stage column sum (colsum_kernel + colsum_final_kernel) of the per-row GroupNorm partials and of the time-bias gradient
    above 512 rows;
  * the CUDA-core implicit GEMM with 64- and 128-row tiles (fp32 mode);
  * the tensor-pipe convolution with N tiles of 64 / 128 / 256 columns, its shallower stage ring, the accumulate-mode epilogue of wide
    tiles, and the tensor-pipe weight gradient with several row boxes per CTA (tf32 mode).

The reference is torch autograd of the oracle in float64 on the CPU, in row chunks (GroupNorm is per row and the loss is a sum over
rows, so chunking is exact).  A dropped or doubled row box moves a gradient summed over 4 097 rows by only ~1 / 4 097, so besides the
whole-tensor figures the tests take the worst row and the worst time slot, and a sparse-row probe puts the whole loss on a few rows
that sit in first, last-full and last-partial boxes."""
import json
import re

import pytest
import torch

import cld_oracle as O
from horizon_metric import rel, worst_row_rel, worst_slot_rel
from ppo_cases import assert_graph_replay_equals_eager, clip_regions, ppo_case, ppo_oracle

pytestmark = pytest.mark.gpu

T = 52
N_T = 16                                   # diffusion steps of the model; t is drawn from 1 .. N_T - 1
CHUNK = 256                                # rows per float64 autograd graph (~1.4 GB of host memory)
EPS_TOL = {"fp32": 2e-5, "tf32": 1e-2}     # relative L2 of eps
GRAD_TOL = {"fp32": 1e-4, "tf32": 1e-2}    # relative L2 of dx and of every parameter gradient
LOCAL = 3.0                                # a single row or time slot averages fewer elements: LOCAL x the whole-tensor budget
# (mode, row count).  fp32 mode at 4 097 rows reaches no branch that 1 031 rows does not.
CASES = [("fp32", "gn"), ("tf32", "gn"), ("fp32", "mid"), ("tf32", "mid"), ("tf32", "big")]


def num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def row_count(which):
    """gn: the first row count on the one-warp GroupNorm path.  mid: odd, a partial last box at every box height the kernels use
    (2 / 4 / 9 rows in the tensor-pipe forward, 2 / 4 / 8 in its weight gradient, 128 in the time projection).  big: N tiles of 256
    at level 2 and many row boxes per weight-gradient CTA."""
    return {"gn": 2 * num_sms() + 1, "mid": 1031, "big": 4097}[which]


def _inputs(R, seed):
    g = torch.Generator().manual_seed(seed)
    x, cond = torch.randn(R, T, 4, generator=g), torch.randn(R, 256, generator=g)
    t = torch.randint(1, N_T, (R,), generator=g)
    d_eps = torch.randn(R, T, 4, generator=g)
    return x, cond, t, d_eps


def _oracle(sd64, x, cond, t, d_eps):
    """float64 autograd of loss = sum(eps * d_eps) through the oracle's U-Net, CHUNK rows at a time -> (eps, [parameter gradients
    summed over the chunks], dx)."""
    params = list(sd64.values())
    grads = [torch.zeros_like(p) for p in params]
    eps, dx = [], []
    for lo in range(0, x.shape[0], CHUNK):
        xs = x[lo:lo + CHUNK].double().requires_grad_(True)
        e = O.unet_forward(sd64, xs, cond[lo:lo + CHUNK].double(), t[lo:lo + CHUNK])
        g = torch.autograd.grad((e * d_eps[lo:lo + CHUNK].double()).sum(), params + [xs])
        for acc, gi in zip(grads, g[:-1]):
            acc += gi
        eps.append(e.detach())
        dx.append(g[-1])
    return torch.cat(eps), grads, torch.cat(dx)


def _free(dm):
    if dm._train_eng is not None:
        dm._train_eng.close()
        dm._train_eng = None
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def dm(models_cpu):
    m, _, _ = models_cpu(N_T)
    m = m.cuda()
    yield m
    _free(m)


@pytest.fixture()
def fresh(dm):
    """The module's model without a training engine before and after the test (the engine of 4 097 rows holds ~6 GB)."""
    _free(dm)
    yield dm
    dm.train_precision = "fp32"
    _free(dm)


@pytest.fixture(scope="module")
def sd64(dm):
    return {k: v.detach().cpu().double().requires_grad_(True) for k, v in dm.model.state_dict().items()}


@pytest.fixture(scope="module")
def reference(sd64):
    """(R, seed) -> inputs and the float64 reference, computed once and shared by the fp32 and tf32 cases."""
    cache = {}

    def get(R, seed):
        if (R, seed) not in cache:
            x, cond, t, d_eps = _inputs(R, seed)
            eps, grads, dx = _oracle(sd64, x, cond, t, d_eps)
            cache[(R, seed)] = dict(x=x, cond=cond, t=t, d_eps=d_eps, eps=eps, grads=grads, dx=dx)
        return cache[(R, seed)]
    return get


def _step(dm, mode, x, cond, t, d_eps):
    """Training forward + backward on the model's training engine (grown to x.shape[0] rows if needed) -> (eps, grads, dx)."""
    dm.train_precision = mode
    eng = dm.train_engine(x.shape[0])
    eps = eng.unet_train_forward(x.cuda(), cond.cuda(), t.cuda())
    grads = [torch.empty_like(p) for p in dm.model.parameters()]
    dx = eng.unet_backward(d_eps.cuda(), grads, want_dx=True)
    torch.cuda.synchronize()
    return eps, grads, dx


# --------------------------------------------------------------------------------------------------------------------------
# 1. forward and backward against the float64 oracle
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,which", CASES)
def test_train_step_vs_float64_oracle(fresh, reference, mode, which):
    R = row_count(which)
    ref = reference(R, 1000 + R)
    eps, grads, dx = _step(fresh, mode, ref["x"], ref["cond"], ref["t"], ref["d_eps"])
    e = {"eps": rel(eps, ref["eps"]), "eps_row": worst_row_rel(eps, ref["eps"]), "eps_slot": worst_slot_rel(eps, ref["eps"], T),
         "dx": rel(dx, ref["dx"]), "dx_row": worst_row_rel(dx, ref["dx"]), "dx_slot": worst_slot_rel(dx, ref["dx"], T)}
    errs = {k: rel(g, w) for k, g, w in zip(fresh.model.state_dict(), grads, ref["grads"])}
    worst = max(errs, key=errs.get)
    print("R=%4d %s: eps rel %.2e row %.2e slot %.2e | dx rel %.2e row %.2e slot %.2e | worst gradient %.2e (%s)" % (
        R, mode, e["eps"], e["eps_row"], e["eps_slot"], e["dx"], e["dx_row"], e["dx_slot"], errs[worst], worst))
    et, gt = EPS_TOL[mode], GRAD_TOL[mode]
    assert e["eps"] < et and e["eps_row"] < LOCAL * et and e["eps_slot"] < LOCAL * et, e
    assert e["dx"] < gt and e["dx_row"] < LOCAL * gt and e["dx_slot"] < LOCAL * gt, e
    assert len(errs) == 148
    bad = {k: v for k, v in errs.items() if not v < gt}
    assert not bad, bad


# --------------------------------------------------------------------------------------------------------------------------
# 2. sparse-row probe: the loss on a few rows in first, last-full and last-partial boxes
# --------------------------------------------------------------------------------------------------------------------------
def probe_rows(R):
    """Row 0, row 2 x SMs, the last row (in the last partial box of every box height that does not divide R) and the last row of
    the last full box of 9 rows (tensor-pipe forward at level 2) and of 8 rows (its weight gradient; also the 128-row box of the
    time projection when R % 128 < 8)."""
    rows = {0, 2 * num_sms(), R - 1}
    for b in (9, 8):
        if R % b:
            rows.add(R - R % b - 1)
    return sorted(r for r in rows if r < R)


@pytest.mark.parametrize("mode,which", CASES)
def test_sparse_row_probe(fresh, sd64, mode, which):
    """d_eps is zero except on the probe rows, so those rows carry every weight, GroupNorm and bias gradient: a kernel that drops or
    double-counts a row box, a split or a column-sum block shows as an O(1) error of that tensor, not as 1 / R."""
    R = row_count(which)
    rows = probe_rows(R)
    idx = torch.tensor(rows)
    x, cond, t, d_all = _inputs(R, 2000 + R)
    d_eps = torch.zeros_like(d_all)
    d_eps[idx] = d_all[idx]
    _, want, dx_want = _oracle(sd64, x[idx], cond[idx], t[idx], d_eps[idx])      # the other rows contribute exactly nothing
    _, grads, dx = _step(fresh, mode, x, cond, t, d_eps)
    dx = dx.cpu()
    others = torch.ones(R, dtype=torch.bool)
    others[idx] = False
    assert torch.count_nonzero(dx[others]) == 0                                   # rows without a loss gradient get none
    e_dx, e_row = rel(dx[idx], dx_want), worst_row_rel(dx[idx], dx_want)
    errs = {k: rel(g, w) for k, g, w in zip(fresh.model.state_dict(), grads, want)}
    worst = max(errs, key=errs.get)
    print("R=%4d %s probe rows %s: dx rel %.2e worst row %.2e | worst gradient %.2e (%s)" % (R, mode, rows, e_dx, e_row, errs[worst], worst))
    gt = GRAD_TOL[mode]
    assert e_dx < gt and e_row < LOCAL * gt, (e_dx, e_row)
    bad = {k: v for k, v in errs.items() if not v < gt}
    assert not bad, bad


# --------------------------------------------------------------------------------------------------------------------------
# 3. one handle across row counts: arena reuse and the tensor-map cache
# --------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_row_count_history_is_bit_reproducible(fresh, mode):
    """One engine whose training arena is sized by a 4 097-row step runs 1 031, 2 x SMs + 1, 1 031 and 12 rows.  The two 1 031-row
    steps are bit-identical, and the 2 x SMs + 1 and 12-row steps equal those of an engine made for exactly that row count: the
    arena carved for more rows and the tensor maps cached by (pointer, shape) change nothing."""
    dm = fresh
    R_gn, R_mid, R_big = row_count("gn"), row_count("mid"), row_count("big")
    seeds = {R_big: 31, R_mid: 32, R_gn: 33, 12: 34}
    run = lambda R: _step(dm, mode, *_inputs(R, seeds[R]))                       # noqa: E731
    run(R_big)
    eng = dm._train_eng
    history = [run(R) for R in (R_mid, R_gn, R_mid, 12)]
    assert dm._train_eng is eng                                                   # every step ran on the one handle

    def same(a, b):
        return torch.equal(a[0], b[0]) and torch.equal(a[2], b[2]) and all(torch.equal(p, q) for p, q in zip(a[1], b[1]))
    assert same(history[0], history[2])
    for R, got in ((R_gn, history[1]), (12, history[3])):
        _free(dm)
        assert same(got, run(R)), R
        assert dm._train_eng is not eng


# --------------------------------------------------------------------------------------------------------------------------
# 4. the PPO minibatch at 1 031 rows
# --------------------------------------------------------------------------------------------------------------------------
CLIP = 0.2


@pytest.fixture(scope="module")
def ppo_ref(dm, sd64):
    """The 1 031-row PPO minibatch (tests/ppo_cases.py) and its float64 reference, built once for both modes and the graph test."""
    R = row_count("mid")
    sched = {k: v.detach().cpu().double() for k, v in dm.named_buffers()}
    case = ppo_case(sched, sd64, R, 77, T=T, n_t=N_T, clip=CLIP)
    baseline = 0.05
    loss, lp, grads = ppo_oracle(sd64, sched, *case, baseline, CLIP)
    return dict(R=R, sched=sched, case=case, baseline=baseline, loss=loss, lp=lp, grads=grads)


@pytest.fixture()
def own_model(models_cpu):
    """-> make(): a fresh CUDA model (seed 0, like the module's); every model made is closed after the test, whatever its outcome."""
    made = []

    def make():
        m, _, _ = models_cpu(N_T)
        made.append(m.cuda())
        return made[-1]
    yield make
    for m in made:
        _free(m)


def _head_d_eps64(eps, x1, x0, t, sched, lp_old, reward, baseline):
    """d(loss)/d(eps) of DmModel.log_prob's tail + the clipped surrogate (O.ppo_loss) in float64, at a given eps."""
    e = eps.detach().cpu().double().requires_grad_(True)
    c = lambda k: sched[k][t].view(-1, 1, 1)                                      # noqa: E731
    mean = c("x_t_cof") * x1.double() - c("noise_cof") * e
    sigma = (0.5 * c("posterior_log_variance_clipped")).exp()
    lp = torch.distributions.Normal(mean, sigma).log_prob(x0.double()).mean(dim=(1, 2))
    return torch.autograd.grad(O.ppo_loss(lp, lp_old.double(), reward.double(), baseline, CLIP), e)[0]


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_ppo_minibatch_vs_float64_oracle(own_model, sd64, ppo_ref, mode):
    """cld_ppo_grad (forward, log-prob head, clipped surrogate, backward) at 1 031 rows against O.ppo_grads in float64: log_p_new, the
    loss and all 148 gradients.

    tf32 mode: the head's d_eps is proportional to x_{t-1} - mean with mean = c1 x_t - c2 eps, so an eps error reaches d_eps scaled by
    c2 / sigma -- 0.69 .. 1.75 for t = 1 .. 14 of the 16-step schedule, but 32 at t = 15 (beta clipped to 0.999) -- and gradients such as
    the output bias (a sum of d_eps whose terms largely cancel) amplify it further: end to end, tf32's 1.6e-3 eps error puts gradients
    2e-2 .. 4e-2 away from float64.  That figure is printed; what is asserted is each stage against float64 at the kernel's own input --
    the head's d_eps at the kernel's eps (1e-5), and the gradients against float64 autograd of the backward driven by the kernel's d_eps
    (1e-2) -- plus log_p_new and the loss end to end (1e-2)."""
    R, sched, baseline = ppo_ref["R"], ppo_ref["sched"], ppo_ref["baseline"]
    x1, x0, cond, t, lp_old, reward = ppo_ref["case"]
    loss_want, lp_want, g_want = ppo_ref["loss"], ppo_ref["lp"], ppo_ref["grads"]
    inside, cut = clip_regions(lp_want, lp_old, reward, baseline, CLIP)
    ratio = (lp_want - lp_old.double()).exp()
    assert inside.any() and cut.any() and (~inside & ~cut).any() and (ratio > 1 + CLIP).any() and (ratio < 1 - CLIP).any()
    dm = own_model()
    dm.train_precision = mode
    c = lambda v: v.cuda()                                                        # noqa: E731
    loss, lp = dm.ppo_minibatch_grad(c(x1), c(x0), c(cond), c(t), c(lp_old), c(reward), baseline, CLIP)
    torch.cuda.synchronize()
    grads = [g.clone() for g in dm._flat_views[1]]
    names = list(dm.model.state_dict())
    e_lp, e_loss = rel(lp, lp_want), abs(float(loss) - loss_want)
    errs = {k: rel(gr, w) for k, gr, w in zip(names, grads, g_want)}
    worst = max(errs, key=errs.get)
    print("R=%4d %s PPO minibatch: log_p_new rel %.2e max abs %.2e, loss %.4f error %.2e, worst gradient vs float64 PPO %.2e (%s); "
          "rows inside / cut %d / %d" % (R, mode, e_lp, (lp.cpu().double() - lp_want).abs().max().item(), loss_want, e_loss, errs[worst], worst,
                                         int(inside.sum()), int(cut.sum())))
    tol = {"fp32": 1e-5, "tf32": 1e-2}[mode]
    assert e_lp < tol and e_loss < tol * max(1.0, abs(loss_want)), (e_lp, e_loss)
    assert len(errs) == 148
    if mode == "tf32":
        # the same step in its stages: forward -> head (d_eps) -> backward, each against float64 at the kernel's own input
        eng = dm.train_engine(R)
        eps = eng.unet_train_forward(c(x1), c(cond), c(t))
        _, _, d_eps = eng.ppo_head(eps, c(x1), c(x0), c(t), c(lp_old), c(reward), baseline, CLIP)
        staged = [torch.empty_like(p) for p in dm.model.parameters()]
        eng.unet_backward(d_eps, staged)
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(grads, staged))             # cld_ppo_grad == the three calls
        e_head = rel(d_eps, _head_d_eps64(eps, x1, x0, t, sched, lp_old, reward, baseline))
        _, g_stage, _ = _oracle(sd64, x1, cond, t, d_eps.cpu())
        errs = {k: rel(gr, w) for k, gr, w in zip(names, grads, g_stage)}
        worst = max(errs, key=errs.get)
        print("R=%4d tf32 PPO minibatch in stages: head d_eps rel %.2e, worst gradient vs float64 backward of the kernel's d_eps %.2e (%s)" % (
            R, e_head, errs[worst], worst))
        assert e_head < 1e-5, e_head
    bad = {k: v for k, v in errs.items() if not v < GRAD_TOL[mode]}
    assert not bad, bad


def test_graph_replay_equals_eager_updates_1031_rows(own_model, ppo_ref):
    """GraphedPPOStep at 1 031 rows (tf32 mode): two eager warm-up calls, then three graph replays, reproduce the parameters and
    losses of five un-captured updates bit for bit.  At this size the parameter-gradient stream inside the graph overlaps the
    data-gradient chain for much longer than at the 12 rows of test_gpu_train.py."""
    assert_graph_replay_equals_eager(own_model, *ppo_ref["case"], baseline=0.0, clip=CLIP, iters=5)


# --------------------------------------------------------------------------------------------------------------------------
# 5. coverage guard: the large-batch kernels are really launched
# --------------------------------------------------------------------------------------------------------------------------
def _kernels(fn, path):
    """-> the CUDA kernel events (name, grid, stream, ts) of fn(), from torch.profiler's exported trace, in launch order."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        ev = json.load(f)["traceEvents"]
    ks = [e for e in ev if e.get("cat") == "kernel"]
    return sorted(ks, key=lambda e: e["ts"])


def test_large_batch_kernels_are_launched(fresh, tmp_path):
    """fp32 mode at 1 031 rows: the one-warp GroupNorm kernels, the two-stage column sum (colsum_kernel is its first stage and runs
    nowhere else) and the 64- and 128-row GEMM tiles all run (down- and upsampling GEMMs take 64-row tiles, the level-0 and level-2
    convolutions 128-row tiles).  If a dispatch threshold moves, this fails instead of the tests above silently checking the
    small-batch kernels again."""
    dm = fresh
    R = row_count("mid")
    x, cond, t, d_eps = _inputs(R, 5)
    dm.train_precision = "fp32"
    eng = dm.train_engine(R)
    grads = [torch.empty_like(p) for p in dm.model.parameters()]

    def step():
        eng.unet_train_forward(x.cuda(), cond.cuda(), t.cuda())
        eng.unet_backward(d_eps.cuda(), grads, want_dx=True)
    names = sorted({e["name"] for e in _kernels(step, tmp_path / "fp32.json")})
    # template arguments as the demangler prints them: <1> or <(int)1>, <false, 64> or <(bool)0, (int)64>
    want = {"gn_mish_fwd_mw_kernel<1>": r"gn_mish_fwd_mw_kernel<(\(int\))?1>", "gn_mish_bwd_kernel<1>": r"gn_mish_bwd_kernel<(\(int\))?1>",
            "colsum_kernel": r"\bcolsum_kernel\(",
            "tgemm_kernel BM 64": r"tgemm_kernel<(\(bool\))?\w+, (\(int\))?64>", "tgemm_kernel BM 128": r"tgemm_kernel<(\(bool\))?\w+, (\(int\))?128>"}
    seen = {k: [n for n in names if re.search(p, n)] for k, p in want.items()}
    print("R=%d fp32 training step, %d distinct kernels:\n  %s" % (R, len(names), "\n  ".join(names)))
    missing = [k for k, v in seen.items() if not v]
    assert not missing, (missing, names)


def _tf32_forward_convs(dims, T, D):
    """(N, T') of every convolution of the training forward that runs on the tensor pipe, in launch order: all but those reading the
    4-channel input or writing the 4-channel output (channels not a multiple of 32 / 16)."""
    d0, d1, d2 = dims
    T2, T4 = T // 2, T // 4
    seq = [(2 * (d0 + d1 + d2) + 2 * d2 + 2 * (d1 + d0), 1)]                       # time / cond projection of the 12 blocks
    def block(cin, cout, Tp):                                                      # noqa: E306
        ok = all(c % 32 == 0 for c in cin)
        seq.extend([(cout, Tp)] * (int(ok) + 1 + int(ok and sum(cin) != cout)))   # blocks[0] conv, blocks[1] conv, residual 1x1
    block((D,), d0, T); block((d0,), d0, T); seq.append((d0, T2))                  # downs.0, Downsample1d    # noqa: E702
    block((d0,), d1, T2); block((d1,), d1, T2); seq.append((d1, T4))               # downs.1, Downsample1d    # noqa: E702
    block((d1,), d2, T4); block((d2,), d2, T4)                                     # downs.2                  # noqa: E702
    block((d2,), d2, T4); block((d2,), d2, T4)                                     # mid blocks               # noqa: E702
    block((d2, d2), d1, T4); block((d1,), d1, T4); seq += [(d1, T4)] * 2           # ups.0, Upsample1d phases # noqa: E702
    block((d1, d1), d0, T2); block((d0,), d0, T2); seq += [(d0, T2)] * 2           # ups.1, Upsample1d phases # noqa: E702
    seq.append((d0, T))                                                            # final Conv1dBlock
    return seq


def test_tf32_forward_tile_widths(fresh, tmp_path):
    """tf32 mode: the N tile of the tensor-pipe convolution is a runtime parameter, seen in the trace as grid.y = N / BN (grid.x =
    row tiles of 128 // T' rows).  The launches of one training forward are matched to the layer list, their row tiling is checked,
    and the N tile widths per row count are printed."""
    dm = fresh
    seq = _tf32_forward_convs(dm.model.dims[1:], T, 4)
    for which in ("gn", "mid", "big"):
        R = row_count(which)
        x, cond, t, _ = _inputs(R, 6)
        dm.train_precision = "tf32"
        eng = dm.train_engine(R)
        ks = [e for e in _kernels(lambda: eng.unet_train_forward(x.cuda(), cond.cuda(), t.cuda()), tmp_path / ("tf32_%d.json" % R))
              if "tf32_conv_kernel" in e["name"]]
        assert len(ks) == len(seq), (R, len(ks), len(seq))
        widths = {}
        for (N, Tp), e in zip(seq, ks):
            gx, gy = e["args"]["grid"][:2]
            assert gx == -(-R // min(128 // Tp, R)), (R, N, Tp, e["args"]["grid"])
            assert N % gy == 0, (R, N, Tp, e["args"]["grid"])
            widths.setdefault((Tp, N), set()).add(N // gy)
        print("R=%4d tf32 forward, N tile per (T', N): %s" % (
            R, ", ".join("(%d, %d): %s" % (Tp, N, "/".join(str(b) for b in sorted(v))) for (Tp, N), v in sorted(widths.items()))))
        _free(dm)
