"""`GreenLight` -- mirror of the reference's pybind11 class (greenlight_model.cpp:130-136):
`GreenLight(nx, nu, nd, np, dt).evalF(x, u, d, p) -> list[float]`, executed by the CUDA evalF kernel.

`evalF_batch` is the batched form the B200 path is built for (B independent evalF calls in one launch).
The integrator is classical RK4 with zero-order hold on `n_sub` nominal substeps (BASELINE.json north_star): "graded" (default,
grid refined at the start of the interval, DESIGN.md "Integrator contract") or "fixed" (equal substeps); the reference's CVODES
(abstol=reltol=1e-6) is a third-party solver that is not available here.
"""
import numpy as np
import torch

from . import _lib


class GreenLight:
    def __init__(self, nx=28, nu=6, nd=10, np_=208, dt=900.0, n_sub=None, device=0, integrator=None):
        if (nx, nu, nd, np_) != (_lib.NX, _lib.NU, _lib.ND, _lib.NP):
            raise ValueError("GreenLight model dimensions are fixed: nx=28, nu=6, nd=10, np=208")
        self.dt = float(dt)
        if integrator is None:
            from .vec_env import DEFAULT_INTEGRATOR
            integrator = DEFAULT_INTEGRATOR
        if integrator not in ("fixed", "graded"):
            raise ValueError("integrator must be 'fixed' or 'graded'")
        self.integrator = integrator  # "graded": DESIGN.md "Graded integrator" (default n_sub 300)
        self.n_sub = int(n_sub) if n_sub is not None else (600 if integrator == "fixed" else 260)
        self.device = int(device)
        self._lib = _lib.load()

    def _inputs(self, x, u, d, p):
        dev = torch.device("cuda", self.device)
        as_t = lambda a: torch.as_tensor(np.asarray(a, dtype=np.float64) if not torch.is_tensor(a) else a,
                                         dtype=torch.float64, device=dev).contiguous()
        x, u, d, p = as_t(x), as_t(u), as_t(d), as_t(p)
        B = x.shape[0]
        assert x.shape == (B, 28) and u.shape == (B, 6) and d.shape == (B, 10)
        p_stride = 0 if p.dim() == 1 else _lib.NP
        assert p.shape[-1] == _lib.NP and (p.dim() == 1 or p.shape[0] == B)
        return dev, x, u, d, p, B, p_stride

    def evalF_batch(self, x, u, d, p, return_bad=False):
        """x [B,28], u [B,6], d [B,10], p [208] or [B,208]; torch CUDA float64 tensors or array-likes.
        Returns x_next [B,28] as a CUDA float64 tensor."""
        dev, x, u, d, p, B, p_stride = self._inputs(x, u, d, p)
        out = torch.empty_like(x)
        bad = torch.zeros(B, dtype=torch.uint8, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = self._lib.glg_evalf_batch_ex(x.data_ptr(), u.data_ptr(), d.data_ptr(), p.data_ptr(), p_stride, out.data_ptr(),
                                          bad.data_ptr(), B, self.dt, self.n_sub, 0 if self.integrator == "fixed" else 1,
                                          self.device, stream)
        _lib.check(rc, None, "glg_evalf_batch_ex")
        return (out, bad) if return_bad else out

    def rhs_jacobian_batch(self, x, u, d, p):
        """Continuous-time right-hand side and its exact Jacobians (forward-mode differentiation of the model, fp64).
        Inputs as evalF_batch.  Returns (f [B,28], df/dx [B,28,28], df/du [B,28,6]) as CUDA float64 tensors."""
        dev, x, u, d, p, B, p_stride = self._inputs(x, u, d, p)
        f = torch.empty_like(x)
        jx = torch.empty((B, 28, 28), dtype=torch.float64, device=dev)
        ju = torch.empty((B, 28, 6), dtype=torch.float64, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = self._lib.glg_rhs_jacobian_batch(x.data_ptr(), u.data_ptr(), d.data_ptr(), p.data_ptr(), p_stride, f.data_ptr(),
                                              jx.data_ptr(), ju.data_ptr(), B, self.device, stream)
        _lib.check(rc, None, "glg_rhs_jacobian_batch")
        return f, jx, ju

    def jacobian_batch(self, x, u, d, p, return_bad=False):
        """One control interval (evalF_batch) and its exact Jacobians on the executed integration grid.  Inputs as evalF_batch.
        Returns (x_next [B,28], dx_next/dx [B,28,28], dx_next/du [B,28,6]) as CUDA float64 tensors, plus the uint8 [B]
        non-finite flags when return_bad is set."""
        dev, x, u, d, p, B, p_stride = self._inputs(x, u, d, p)
        xn = torch.empty_like(x)
        jx = torch.empty((B, 28, 28), dtype=torch.float64, device=dev)
        ju = torch.empty((B, 28, 6), dtype=torch.float64, device=dev)
        bad = torch.zeros(B, dtype=torch.uint8, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = self._lib.glg_evalf_jacobian_batch(x.data_ptr(), u.data_ptr(), d.data_ptr(), p.data_ptr(), p_stride, xn.data_ptr(),
                                                jx.data_ptr(), ju.data_ptr(), bad.data_ptr(), B, self.dt, self.n_sub,
                                                0 if self.integrator == "fixed" else 1, self.device, stream)
        _lib.check(rc, None, "glg_evalf_jacobian_batch")
        return (xn, jx, ju, bad) if return_bad else (xn, jx, ju)

    def evalF(self, x, u, d, p):
        """Single-env call with the reference's signature; returns a list of 28 floats. Raises RuntimeError if the
        integration produced a non-finite state (the reference raises from CVODES; tomato_env.py:119-123 catches)."""
        out, bad = self.evalF_batch(np.asarray(x, dtype=np.float64)[None], np.asarray(u, dtype=np.float64)[None],
                                    np.asarray(d, dtype=np.float64)[None], np.asarray(p, dtype=np.float64), True)
        if int(bad[0]) != 0:
            raise RuntimeError("GreenLight.evalF: non-finite state")
        return out[0].cpu().tolist()
