"""Thin, typed wrapper around the C ABI: owns a CldHandle, converts torch tensors to raw device
pointers, raises RuntimeError(cld_last_error()) on failure.  PyTorch is plumbing only (device
memory + streams); all arithmetic of the path happens inside libcld_b200.so."""
import ctypes as C

import torch

from . import _lib
from ._lib import CldConfig, CldGuidanceConfig, CldScene, lib

from .keys import DECODER_KEYS, NORM_MEAN, NORM_STD, default_guidance  # noqa: F401  (re-exported)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _f32(t, dev):
    if t is None:
        return None
    return t.to(device=dev, dtype=torch.float32).contiguous()


def _u8(t, dev):
    if t is None:
        return None
    t = t.to(device=dev)
    if t.dtype == torch.bool:
        t = t.to(torch.uint8)
    return t.to(torch.uint8).contiguous()


def _grad_steps(v):
    """The guidance dict's `grad_steps`: an integer >= 1 (a bool or a float is refused rather than rounded)."""
    import numbers
    if isinstance(v, bool) or not isinstance(v, numbers.Integral) or int(v) < 1:
        raise ValueError("guidance grad_steps must be an integer >= 1, got %r" % (v,))
    return int(v)


def _on_device(fn):
    """Run a method with the engine's device current: the handle's buffers, the kernels and the caller's stream all
    belong to `self.device`, whatever device the calling thread had selected."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *a, **k):
        if torch.cuda.current_device() == self.device.index:
            return fn(self, *a, **k)
        with torch.cuda.device(self.device):
            return fn(self, *a, **k)
    return wrapped


class Engine:
    def __init__(self, *, horizon=52, latent_dim=4, cond_dim=256, base_dim=32, dims=(64, 128, 256), hidden=64,
                 n_timesteps=100, max_rows=4096, precision="fp32", dt=0.1, acce_bound=(-10.0, 8.0),
                 vbound=(-10.0, 30.0), max_steer=0.5, max_yawvel=6.283185307179586, norm_mean=NORM_MEAN,
                 norm_std=NORM_STD, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("cld_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        cfg = CldConfig()
        cfg.horizon, cfg.latent_dim, cfg.cond_dim, cfg.base_dim = horizon, latent_dim, cond_dim, base_dim
        cfg.dims = (C.c_int32 * 3)(*[int(d) for d in dims])
        cfg.hidden, cfg.n_timesteps, cfg.max_rows = hidden, int(n_timesteps), int(max_rows)
        cfg.precision = {"fp32": _lib.CLD_PREC_FP32, "bf16": _lib.CLD_PREC_BF16}[precision]
        cfg.dt = dt
        cfg.acce_lo, cfg.acce_hi = float(acce_bound[0]), float(acce_bound[1])
        cfg.v_lo, cfg.v_hi = float(vbound[0]), float(vbound[1])
        cfg.max_steer, cfg.max_yawvel = float(max_steer), float(max_yawvel)
        cfg.norm_mean = (C.c_float * 6)(*[float(v) for v in norm_mean])
        cfg.norm_std = (C.c_float * 6)(*[float(v) for v in norm_std])
        self.cfg = cfg
        self.precision = precision
        self.T, self.D, self.Cc = horizon, latent_dim, cond_dim
        self.max_rows = int(max_rows)
        self._h = C.c_void_p(0)
        with torch.cuda.device(self.device):
            rc = lib.cld_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            raise RuntimeError("cld_create failed (%d): %s" % (rc, lib.cld_last_error(None).decode()))
        self._keep = []

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            lib.cld_destroy(self._h)
            self._h = C.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise RuntimeError("%s failed (%d): %s" % (what, rc, lib.cld_last_error(self._h).decode()))

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ measurement
    def launch_count(self):
        return int(lib.cld_launch_count(self._h))

    @_on_device
    def profile_begin(self):
        self._check(lib.cld_profile_begin(self._h), "cld_profile_begin")

    @_on_device
    def profile_end(self):
        """-> {kind: (total_ms, brackets)} for kinds denoiser / step / guidance / decode."""
        ms, cnt = (C.c_double * 4)(), (C.c_int * 4)()
        self._check(lib.cld_profile_end(self._h, ms, cnt, 4), "cld_profile_end")
        names = ["denoiser", "step", "guidance", "decode"]
        return {n: (ms[i], cnt[i]) for i, n in enumerate(names)}

    # ------------------------------------------------------------------ weights / schedule
    @_on_device
    def load_unet(self, state_dict):
        """state_dict: DmModel.model.state_dict() (reference key order, SURVEY.md sec. 8b)."""
        ts = [_f32(v.detach(), self.device) for v in state_dict.values()]
        n = len(ts)
        ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in ts])
        numels = (C.c_int64 * n)(*[t.numel() for t in ts])
        with torch.cuda.device(self.device):
            self._check(lib.cld_load_unet(self._h, ptrs, numels, n, self._stream()), "cld_load_unet")

    @_on_device
    def load_decoder(self, state_dict):
        """state_dict: VaeModel.lstmvae.lstm_dec.state_dict() (keys DECODER_KEYS)."""
        ts = [_f32(state_dict[k].detach(), self.device) for k in DECODER_KEYS]
        ptrs = (C.c_void_p * 12)(*[t.data_ptr() for t in ts])
        with torch.cuda.device(self.device):
            self._check(lib.cld_load_decoder(self._h, ptrs, 12, self._stream()), "cld_load_decoder")

    @_on_device
    def set_schedule(self, bufs):
        names = ["x_t_cof", "noise_cof", "posterior_log_variance_clipped", "sqrt_recip_alphas_cumprod",
                 "sqrt_recipm1_alphas_cumprod", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod"]
        arrs = []
        for k in names:
            v = bufs[k].detach().to("cpu", torch.float32).contiguous()
            arrs.append((C.c_float * v.numel())(*v.tolist()))
        n = int(bufs["x_t_cof"].numel())
        self._check(lib.cld_set_schedule(self._h, *arrs, n), "cld_set_schedule")

    # ------------------------------------------------------------------ scene / guidance structs
    @_on_device
    def make_scene(self, batch, num_scenes, agents_per_scene, num_samp):
        """batch: the reference's data_batch dict (extent, world_from_agent, raster_from_agent, curr_speed,
        drivable_map, [target_pos], [all_other_agents_future_positions/_availability])."""
        d = self.device
        # the drivable map may arrive bit-packed ("drivable_map_bits" [B,H,W/8] uint8, synthetic.pack_drivable_map): 1/8 of the bytes
        bits = batch.get("drivable_map_bits")
        keep = {
            "extent": _f32(batch.get("extent"), d), "wfa": _f32(batch.get("world_from_agent"), d),
            "rfa": _f32(batch.get("raster_from_agent"), d), "speed": _f32(batch.get("curr_speed"), d),
            "dmap": _u8(bits if bits is not None else batch.get("drivable_map"), d), "target": _f32(batch.get("target_pos"), d),
            "others": _f32(batch.get("all_other_agents_future_positions"), d),
            "avail": _u8(batch.get("all_other_agents_future_availability"), d),
            "tspeed": _f32(batch.get("target_speed"), d),
            # waypoint guidance (cld_b200.waypoints.*.scene_entries): per-agent local target, branch, time step, goal distance, multiplier
            "wp_target": _f32(batch.get("wp_target"), d), "wp_dist": _f32(batch.get("wp_dist"), d), "wp_weight": _f32(batch.get("wp_weight"), d),
            "wp_mode": batch["wp_mode"].to(d, torch.int32).contiguous() if batch.get("wp_mode") is not None else None,
            "wp_time": batch["wp_time"].to(d, torch.int32).contiguous() if batch.get("wp_time") is not None else None,
        }
        sc = CldScene()
        sc.num_scenes, sc.agents_per_scene, sc.num_samp = int(num_scenes), int(agents_per_scene), int(num_samp)
        sc.extent, sc.world_from_agent, sc.raster_from_agent = _ptr(keep["extent"]), _ptr(keep["wfa"]), _ptr(keep["rfa"])
        sc.curr_speed, sc.drivable_map = _ptr(keep["speed"]), _ptr(keep["dmap"])
        sc.map_packed = 1 if bits is not None else 0
        if keep["dmap"] is not None:
            sc.map_h = int(keep["dmap"].shape[-2])
            sc.map_w = int(batch.get("drivable_map_width", keep["dmap"].shape[-1] * 8)) if bits is not None else int(keep["dmap"].shape[-1])
        sc.target_pos, sc.others_pos, sc.others_avail = _ptr(keep["target"]), _ptr(keep["others"]), _ptr(keep["avail"])
        sc.num_others = int(keep["others"].shape[1]) if keep["others"] is not None else 0
        sc.target_speed = _ptr(keep["tspeed"])
        sc.wp_target, sc.wp_mode, sc.wp_time = _ptr(keep["wp_target"]), _ptr(keep["wp_mode"]), _ptr(keep["wp_time"])
        sc.wp_dist, sc.wp_weight = _ptr(keep["wp_dist"]), _ptr(keep["wp_weight"])
        if keep["tspeed"] is not None and tuple(keep["tspeed"].shape[-1:]) != (self.T,):
            raise ValueError("target_speed must be [B, T=%d]" % self.T)
        if keep["others"] is not None and keep["others"].shape[2] != self.T:
            raise ValueError("all_other_agents_future_positions must cover the horizon T=%d" % self.T)
        sc._keep = keep
        return sc

    @staticmethod
    def make_guidance(g):
        gc = CldGuidanceConfig()
        gc.w_agent_collision = float(g.get("agent_collision", 0.0))
        gc.w_map_collision = float(g.get("map_collision", 0.0))
        gc.w_target_pos = float(g.get("target_pos", 0.0))
        gc.num_disks = int(g.get("num_disks", 2))
        gc.buffer_dist = float(g.get("buffer_dist", 0.2))
        gc.decay_rate = float(g.get("decay", 0.9))
        npts = g.get("num_points", (10, 10))
        gc.num_points_l, gc.num_points_w = int(npts[0]), int(npts[1])
        gc.speed_th = float(g.get("speed_th", 0.5))
        gc.min_target_time = float(g.get("min_target_time", 0.0))
        gc.optimizer = {"adam": _lib.CLD_OPT_ADAM, "sgd": _lib.CLD_OPT_SGD}[g.get("optimizer", "adam")]
        gc.lr = float(g.get("lr", 0.3))
        gc.w_target_speed = float(g.get("target_speed", 0.0))
        gc.w_acc_limit, gc.acc_limit = float(g.get("acc_limit", 0.0)), float(g.get("acc_limit_value", 0.0))
        gc.w_speed_limit, gc.speed_limit = float(g.get("speed_limit", 0.0)), float(g.get("speed_limit_value", 0.0))
        gc.w_waypoint = float(g.get("waypoint", 0.0))
        gc.grad_steps = _grad_steps(g.get("grad_steps", 1))
        return gc

    # ------------------------------------------------------------------ kernels
    @_on_device
    def unet_forward(self, x, cond, t, debug_stage=None):
        x, cond = _f32(x, self.device), _f32(cond, self.device)
        t = t.to(self.device, torch.int64).contiguous()
        R = x.shape[0]
        eps = torch.empty_like(x)
        dbg = None
        if debug_stage is not None:
            n = lib.cld_unet_debug_stage(self._h, int(debug_stage), C.c_void_p(1), R, self._stream())
            if n < 0:
                raise ValueError("bad debug stage %r" % (debug_stage,))
            dbg = torch.empty(R, n, device=self.device, dtype=torch.float32)
            lib.cld_unet_debug_stage(self._h, int(debug_stage), _ptr(dbg), R, self._stream())
        try:
            self._check(lib.cld_unet_forward(self._h, _ptr(x), _ptr(cond), _ptr(t), _ptr(eps), R, self._stream()),
                        "cld_unet_forward")
        finally:
            if dbg is not None:
                lib.cld_unet_debug_stage(self._h, -1, C.c_void_p(0), R, self._stream())
        return (eps, dbg) if debug_stage is not None else eps

    # ------------------------------------------------------------------ denoiser training (SURVEY.md sec. 8 f-2)
    def set_train_precision(self, mode):
        """"fp32": every training GEMM on the CUDA cores (1e-4 parity mode); "tf32": the stride-1 convolutions (forward and data
        gradient) on the tensor pipe (tcgen05 kind::tf32)."""
        self._check(lib.cld_train_set_precision(self._h, {"fp32": 0, "tf32": 1}[mode]), "cld_train_set_precision")

    @_on_device
    def unet_train_forward(self, x, cond, t):
        """eps like `unet_forward` on the fp32 kernels; the handle keeps the activations for `unet_backward`."""
        x, cond = _f32(x, self.device), _f32(cond, self.device)
        t = t.to(self.device, torch.int64).contiguous()
        eps = torch.empty_like(x)
        self._train_keep = (x, cond, t)            # the backward reads x and t again
        self._check(lib.cld_unet_train_forward(self._h, _ptr(x), _ptr(cond), _ptr(t), _ptr(eps), x.shape[0], self._stream()),
                    "cld_unet_train_forward")
        return eps

    @staticmethod
    def _grad_ptrs(grads):
        for g in grads:
            if g.dtype != torch.float32 or not g.is_contiguous():
                raise ValueError("gradient tensors must be contiguous fp32")
        return (C.c_void_p * len(grads))(*[g.data_ptr() for g in grads])

    @_on_device
    def unet_backward(self, d_eps, grads, want_dx=False):
        """d_eps [R,T,D] -> the parameter gradients, written into `grads` (state-dict order and shapes); -> dx or None."""
        d_eps = _f32(d_eps, self.device)
        dx = torch.empty_like(d_eps) if want_dx else None
        self._check(lib.cld_unet_backward(self._h, _ptr(d_eps), self._grad_ptrs(grads), len(grads), _ptr(dx), d_eps.shape[0],
                                          self._stream()), "cld_unet_backward")
        return dx

    @_on_device
    def ppo_head(self, eps, x_t, x_tm1, t, logp_old, reward, baseline, clip_eps=0.2, want_grad=True, baseline_dev=None):
        """-> (logp_new [R], loss [1], d_eps [R,T,D] or None): DmModel.log_prob's tail + the clipped surrogate and its gradient."""
        eps, x_t, x_tm1 = _f32(eps, self.device), _f32(x_t, self.device), _f32(x_tm1, self.device)
        logp_old, reward = _f32(logp_old, self.device), _f32(reward, self.device)
        t = t.to(self.device, torch.int64).contiguous()
        R = eps.shape[0]
        logp, loss = torch.empty(R, device=self.device), torch.empty(1, device=self.device)
        d_eps = torch.empty_like(eps) if want_grad else None
        self._check(lib.cld_ppo_head(self._h, _ptr(eps), _ptr(x_t), _ptr(x_tm1), _ptr(t), _ptr(logp_old), _ptr(reward), float(baseline),
                                     _ptr(baseline_dev), float(clip_eps), _ptr(logp), _ptr(loss), _ptr(d_eps), R, self._stream()), "cld_ppo_head")
        return logp, loss, d_eps

    @_on_device
    def mse_head(self, eps, noise, want_grad=True):
        eps, noise = _f32(eps, self.device), _f32(noise, self.device)
        loss = torch.empty(1, device=self.device)
        d_eps = torch.empty_like(eps) if want_grad else None
        self._check(lib.cld_mse_head(self._h, _ptr(eps), _ptr(noise), _ptr(loss), _ptr(d_eps), eps.shape[0], self._stream()),
                    "cld_mse_head")
        return loss, d_eps

    @_on_device
    def ppo_grad(self, x_t, x_tm1, cond, t, logp_old, reward, baseline, grads, clip_eps=0.2, baseline_dev=None):
        """One minibatch of ppo_update up to `opt.step()`: -> (logp_new [R], loss [1]); the gradients land in `grads`."""
        x_t, x_tm1, cond = _f32(x_t, self.device), _f32(x_tm1, self.device), _f32(cond, self.device)
        logp_old, reward = _f32(logp_old, self.device), _f32(reward, self.device)
        t = t.to(self.device, torch.int64).contiguous()
        R = x_t.shape[0]
        logp, loss = torch.empty(R, device=self.device), torch.empty(1, device=self.device)
        self._check(lib.cld_ppo_grad(self._h, _ptr(x_t), _ptr(x_tm1), _ptr(cond), _ptr(t), _ptr(logp_old), _ptr(reward), float(baseline),
                                     _ptr(baseline_dev), float(clip_eps), self._grad_ptrs(grads), len(grads), _ptr(logp), _ptr(loss), R,
                                     self._stream()), "cld_ppo_grad")
        return logp, loss

    @_on_device
    def adam_step(self, params, grads, exp_avg, exp_avg_sq, step, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        """torch.optim.Adam on one flat fp32 vector (in place)."""
        for v in (params, grads, exp_avg, exp_avg_sq):
            if v.dtype != torch.float32 or not v.is_contiguous() or v.numel() != params.numel():
                raise ValueError("adam_step needs four contiguous fp32 vectors of equal length")
        self._check(lib.cld_adam_step(self._h, _ptr(params), _ptr(grads), _ptr(exp_avg), _ptr(exp_avg_sq), params.numel(), float(lr),
                                      float(betas[0]), float(betas[1]), float(eps), float(weight_decay), int(step), self._stream()),
                    "cld_adam_step")

    @_on_device
    def adam_step_dev(self, params, grads, exp_avg, exp_avg_sq, lr_dev, step_dev, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        """Adam with the step counter (int64 [1], incremented by the call) and the learning rate (float64 [1]) on the device: replayable
        inside a CUDA graph."""
        self._check(lib.cld_adam_step_dev(self._h, _ptr(params), _ptr(grads), _ptr(exp_avg), _ptr(exp_avg_sq), params.numel(), _ptr(lr_dev),
                                          _ptr(step_dev), float(betas[0]), float(betas[1]), float(eps), float(weight_decay), self._stream()),
                    "cld_adam_step_dev")

    @_on_device
    def posterior_step(self, x, eps, noise, t, t_next=-1, sampler="ddpm", want_mean=False):
        x, eps, noise = _f32(x, self.device), _f32(eps, self.device), _f32(noise, self.device)
        out = torch.empty_like(x)
        mean = torch.empty_like(x) if want_mean else None
        smp = _lib.CLD_SAMPLER_DDPM if sampler == "ddpm" else _lib.CLD_SAMPLER_DDIM
        self._check(lib.cld_posterior_step(self._h, _ptr(x), _ptr(eps), _ptr(noise), int(t), int(t_next), smp,
                                           _ptr(out), _ptr(mean), x.shape[0], self._stream()), "cld_posterior_step")
        return (out, mean) if want_mean else out

    @_on_device
    def decode_rollout(self, z, cond, curr):
        z, cond, curr = _f32(z, self.device), _f32(cond, self.device), _f32(curr, self.device)
        R = z.shape[0]
        act = torch.empty(R, self.T, 2, device=self.device)
        traj = torch.empty(R, self.T, 6, device=self.device)
        self._check(lib.cld_decode_rollout(self._h, _ptr(z), _ptr(cond), _ptr(curr), _ptr(act), _ptr(traj), R,
                                           self._stream()), "cld_decode_rollout")
        return act, traj

    @_on_device
    def unicycle(self, curr, u):
        curr, u = _f32(curr, self.device), _f32(u, self.device)
        R = u.shape[0]
        st = torch.empty(R, self.T, 4, device=self.device)
        self._check(lib.cld_unicycle(self._h, _ptr(curr), _ptr(u), _ptr(st), R, self._stream()), "cld_unicycle")
        return st

    @_on_device
    def indicators(self, traj, scene):
        traj = _f32(traj, self.device)
        R = traj.shape[0]
        off = torch.empty(R, self.T, device=self.device, dtype=torch.uint8)
        coll = torch.empty(R, device=self.device)
        rew = torch.empty(R, device=self.device)
        self._check(lib.cld_indicators(self._h, _ptr(traj), C.byref(scene), _ptr(off), _ptr(coll), _ptr(rew), R,
                                       self._stream()), "cld_indicators")
        return off.bool(), coll, rew

    @_on_device
    def guidance_step(self, z_mean, cond_rows, curr_rows, scene, guidance):
        z, cond, curr = _f32(z_mean, self.device), _f32(cond_rows, self.device), _f32(curr_rows, self.device)
        R = z.shape[0]
        gc = self.make_guidance(guidance)
        z_out, grad = torch.empty_like(z), torch.empty_like(z)
        loss = torch.empty(7, R, device=self.device)      # agent_collision, map_collision, target_pos, target_speed, acc_limit, speed_limit, waypoint
        self._check(lib.cld_guidance_step(self._h, _ptr(z), _ptr(cond), _ptr(curr), C.byref(scene), C.byref(gc),
                                          _ptr(z_out), _ptr(grad), _ptr(loss), R, self._stream()), "cld_guidance_step")
        return z_out, grad, loss

    @_on_device
    def sample(self, x_init, cond_rows, *, noises=None, seed=0, row_offset=0, curr_rows=None, scene=None, guidance=None,
               stride=1, sampler="ddpm", want_traj=False, want_indicators=False):
        """x_init None (with seed != 0): the initial state is drawn in-kernel; row_offset: global id of row 0 (sharded calls)."""
        x_init, cond = _f32(x_init, self.device), _f32(cond_rows, self.device)
        noises, curr = _f32(noises, self.device), _f32(curr_rows, self.device)
        R = cond.shape[0]
        x0 = torch.empty(R, self.T, self.D, device=self.device)
        x1 = torch.empty_like(x0)
        x1_valid = C.c_int(0)
        traj = torch.empty(R, self.T, 6, device=self.device) if (want_traj or want_indicators) else None
        off = torch.empty(R, self.T, device=self.device, dtype=torch.uint8) if want_indicators else None
        coll = torch.empty(R, device=self.device) if want_indicators else None
        gc = self.make_guidance(guidance) if guidance is not None else None
        smp = _lib.CLD_SAMPLER_DDPM if sampler == "ddpm" else _lib.CLD_SAMPLER_DDIM
        self._check(lib.cld_sample(self._h, _ptr(x_init), _ptr(noises), C.c_uint64(int(seed)), C.c_int64(int(row_offset)), _ptr(cond),
                                   _ptr(curr),
                                   C.byref(scene) if scene is not None else None,
                                   C.byref(gc) if gc is not None else None, int(stride), smp, _ptr(x0), _ptr(x1),
                                   C.byref(x1_valid), _ptr(traj), _ptr(off), _ptr(coll), R, self._stream()),
                    "cld_sample")
        return {"x0": x0, "x1": x1 if x1_valid.value else None, "traj": traj,
                "offroad": off.bool() if off is not None else None, "coll": coll}
