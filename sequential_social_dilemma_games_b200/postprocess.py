"""Advantages and value targets of a trajectory on the device: what the rollout worker of the reference's trainers
(algorithms/{ppo,a3c,impala}_causal.py) computes between `env.step` and the learner, over [T, B, N] buffers already in HBM.

    compute_advantages   RLlib's compute_advantages: GAE (use_gae=True) -> (advantages, value_targets), or discounted returns
                         (use_gae=False) -> (advantages, None)
    vtrace               V-trace's from_importance_weights -> VTrace(vs, pg_advantages)

Both add the weighted intrinsic reward first (r = rewards + intrinsic_weight * intrinsic, in fp32: the curriculum-weighted
influence reward of the MOA trainers), and treat a done as the end of an episode: nothing of a later step reaches an earlier
episode, so each episode fragment gets what RLlib computes for it alone with last_r = 0, and the last fragment of a column
bootstraps from `bootstrap` (RLlib's last_r).  One CUDA call (csrc/ssd_advantages.cu, `ssd_advantages` / `ssd_vtrace`) on the
current torch stream; no gradients.  The formulas are those of include/ssd_b200.h.

Inputs are [T, B, N] or [T, M] (then N = M / B from dones [T, B]), all on one CUDA device and contiguous:
    rewards   int32 (what BatchedSSDEnv.step returns) or float32;   values, intrinsic, target_logp, behaviour_logp   float32;
    dones     uint8 or bool [T, B];   bootstrap   float32 shaped like one step of values.
Outputs are float32 and shaped like values."""
import collections
import ctypes as C

import torch

from . import _lib

VTrace = collections.namedtuple("VTrace", "vs pg_advantages")
VTrace.__doc__ = """V-trace targets of a trajectory: vs float32 (the value targets) and pg_advantages float32, shaped like values."""


def _check(name, t, dtypes, shape, device):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch tensor" % name)
    if t.device != device:
        raise ValueError("%s is on %s, values on %s" % (name, t.device, device))
    if t.dtype not in dtypes:
        raise TypeError("%s has dtype %s, expected %s" % (name, t.dtype, " or ".join(str(d) for d in dtypes)))
    if tuple(t.shape) != tuple(shape):
        raise ValueError("%s has shape %s, expected %s" % (name, tuple(t.shape), tuple(shape)))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    return C.c_void_p(t.data_ptr())


def _prepare(rewards, values, dones, bootstrap, intrinsic, intrinsic_weight, logps=()):
    """-> (T, M, N, device, ctypes arguments from `rewards` through `bootstrap`, the logp pointers)."""
    if not isinstance(values, torch.Tensor) or values.device.type != "cuda":
        raise ValueError("values must be a float32 CUDA tensor")
    if values.dim() not in (2, 3):
        raise ValueError("values must be [T, B, N] or [T, M], not %s" % (tuple(values.shape),))
    device = values.device
    if not isinstance(dones, torch.Tensor) or dones.dim() != 2:
        raise ValueError("dones must be a [T, B] tensor")
    t_count, b = dones.shape
    if values.dim() == 3:
        n = values.shape[2]
        if tuple(values.shape[:2]) != (t_count, b):
            raise ValueError("values has shape %s, dones %s: expected [T, B, N] with [T, B] = %s" % (tuple(values.shape),
                             tuple(dones.shape), (t_count, b)))
    else:
        if values.shape[0] != t_count or b == 0 or values.shape[1] % b != 0:
            raise ValueError("values has shape %s, dones %s: expected [T, M] with M a multiple of B" % (tuple(values.shape),
                             tuple(dones.shape)))
        n = values.shape[1] // b
    if t_count == 0 or b * n == 0:
        raise ValueError("empty trajectory: T = %d, M = %d" % (t_count, b * n))
    shape, f32 = tuple(values.shape), (torch.float32,)
    if dones.dtype == torch.bool:
        dones = dones.view(torch.uint8)
    args = [_check("rewards", rewards, (torch.int32, torch.float32), shape, device),
            _lib.DTYPE_I32 if rewards.dtype == torch.int32 else _lib.DTYPE_F32,
            None if intrinsic is None else _check("intrinsic", intrinsic, f32, shape, device),
            float(intrinsic_weight),
            _check("values", values, f32, shape, device),
            _check("dones", dones, (torch.uint8,), (t_count, b), device),
            _check("bootstrap", bootstrap, f32, shape[1:], device)]
    ptrs = [_check(name, t, f32, shape, device) for name, t in logps]
    return t_count, b * n, n, device, args, ptrs


def _run(fn, t_count, m, device, args):
    with torch.cuda.device(device):
        nbytes = _lib.lib.ssd_advantages_workspace_bytes(t_count, m)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=device) if nbytes else None   # chunk carries, when time is split
        stream = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
        _lib.check(fn(*args, None if ws is None else C.c_void_p(ws.data_ptr()), nbytes, stream))


def compute_advantages(rewards, values, dones, bootstrap, *, gamma, lambda_, use_gae=True, intrinsic=None, intrinsic_weight=0.0):
    """RLlib's compute_advantages over a trajectory -> (advantages, value_targets), value_targets None for use_gae=False.

    use_gae=True:  delta_t = r_t + gamma V_{t+1} - V_t, advantages = the gamma*lambda-discounted sum of delta within the
                   episode, value_targets = advantages + values;
    use_gae=False: advantages = the gamma-discounted return within the episode (RLlib writes zeros as value targets; none here).
    V_T = bootstrap, and a done at t drops every t+1 term.  gamma and lambda_ in [0, 1] (lambda_ is not used for use_gae=False)."""
    t_count, m, n, device, args, _ = _prepare(rewards, values, dones, bootstrap, intrinsic, intrinsic_weight)
    adv = torch.empty_like(values)
    vt = torch.empty_like(values) if use_gae else None
    mode = _lib.ADV_GAE if use_gae else _lib.ADV_RETURNS
    _run(_lib.lib.ssd_advantages, t_count, m, device,
         [mode, t_count, m, n] + args + [float(gamma), float(lambda_), C.c_void_p(adv.data_ptr()),
                                         None if vt is None else C.c_void_p(vt.data_ptr())])
    return adv, vt


def vtrace(rewards, values, dones, bootstrap, target_logp, behaviour_logp, *, gamma, clip_rho_threshold, clip_pg_rho_threshold,
           intrinsic=None, intrinsic_weight=0.0):
    """V-trace's from_importance_weights over a trajectory -> VTrace(vs, pg_advantages).

    rho = exp(target_logp - behaviour_logp); rho_bar = min(clip_rho_threshold, rho), c = min(1, rho),
    rho_pg = min(clip_pg_rho_threshold, rho); vs_t - V_t = rho_bar_t delta_t + gamma c_t (vs_{t+1} - V_{t+1}) with
    delta_t = r_t + gamma V_{t+1} - V_t; pg_advantages_t = rho_pg_t (r_t + gamma vs_{t+1} - V_t); vs_T = V_T = bootstrap, and a
    done at t drops every t+1 term.  A threshold of float('inf') disables its clip (None in RLlib); gamma in [0, 1]."""
    t_count, m, n, device, args, ptrs = _prepare(rewards, values, dones, bootstrap, intrinsic, intrinsic_weight,
                                                  (("target_logp", target_logp), ("behaviour_logp", behaviour_logp)))
    vs, pg = torch.empty_like(values), torch.empty_like(values)
    _run(_lib.lib.ssd_vtrace, t_count, m, device,
         [t_count, m, n] + args + ptrs + [float(gamma), float(clip_rho_threshold), float(clip_pg_rho_threshold),
                                          C.c_void_p(vs.data_ptr()), C.c_void_p(pg.data_ptr())])
    return VTrace(vs, pg)
