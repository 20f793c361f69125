"""Minimal LMS discrete scheduler with the diffusers-0.10.0 `LMSDiscreteScheduler` call surface used at
paint_with_words.py:197-202, 431-476, 506 and paint_with_words_inpaint.py:180-197, 266.

diffusers is a third-party dependency that is not vendored under /root/reference (requirements.txt:1
pins 0.10.0) and is not installed here, so the published algorithm is restated: scaled-linear betas
0.00085..0.012 over 1000 train steps, Karras-style sigmas = sqrt((1-abar)/abar) interpolated at
linspace(0,999,n)[::-1] with a trailing 0, epsilon prediction, order-4 linear multistep with
coefficients from scipy.integrate.quad(epsrel=1e-4).

B200-first change: the multistep coefficients of every step are integrated once in `set_timesteps`
(the stock implementation calls scipy.quad on the host inside every `step`, stalling the stream), and
`step_index_of` avoids the `.nonzero().item()` device sync of paint_with_words.py:473.

Euler, Euler ancestral and DPM-Solver++(2M) (below) use the same sigma parametrisation and call surface; each step
is one row of coefficients, which `PwWSampler` applies on the GPU in one fused kernel.
"""
from __future__ import annotations

import math
from typing import List, Optional, Tuple

import numpy as np
import torch
from scipy import integrate


class _StepOutput:
    def __init__(self, prev_sample, pred_original_sample):
        self.prev_sample = prev_sample
        self.pred_original_sample = pred_original_sample


class LMSDiscreteScheduler:
    order = 1

    def __init__(self, beta_start: float = 0.0001, beta_end: float = 0.02, beta_schedule: str = "linear",
                 num_train_timesteps: int = 1000):
        if beta_schedule == "linear":
            betas = np.linspace(beta_start, beta_end, num_train_timesteps, dtype=np.float32)
        elif beta_schedule == "scaled_linear":
            betas = np.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=np.float32) ** 2
        else:
            raise NotImplementedError(beta_schedule)
        self.config = {"num_train_timesteps": num_train_timesteps, "beta_start": beta_start,
                       "beta_end": beta_end, "beta_schedule": beta_schedule}
        self.betas = torch.from_numpy(betas)
        self.alphas_cumprod = torch.cumprod(1.0 - self.betas, dim=0)
        sig = self._train_sigmas()
        self.sigmas = torch.from_numpy(np.concatenate([sig[::-1], [0.0]]).astype(np.float32))
        self.init_noise_sigma = self.sigmas.max()
        self.timesteps = torch.from_numpy(
            np.linspace(0, num_train_timesteps - 1, num_train_timesteps, dtype=float)[::-1].copy())
        self.num_inference_steps: Optional[int] = None
        self.derivatives: List[torch.Tensor] = []
        self._coeffs: Optional[List[List[float]]] = None
        self._t_list: List[float] = self.timesteps.tolist()

    def _train_sigmas(self) -> np.ndarray:
        ac = self.alphas_cumprod.numpy()
        return np.array(((1 - ac) / ac) ** 0.5)

    # ---- schedule ------------------------------------------------------------------------
    def set_timesteps(self, num_inference_steps: int, device=None):
        self.num_inference_steps = num_inference_steps
        n_train = self.config["num_train_timesteps"]
        timesteps = np.linspace(0, n_train - 1, num_inference_steps, dtype=float)[::-1].copy()
        sig = self._train_sigmas()
        sig = np.interp(timesteps, np.arange(0, len(sig)), sig)
        sig = np.concatenate([sig, [0.0]]).astype(np.float32)
        self.sigmas = torch.from_numpy(sig)            # host copy: sigma is host scalar math (pww.py:402-405)
        self.timesteps = torch.from_numpy(timesteps).to(device=device)
        self._t_list = timesteps.tolist()
        self.derivatives = []
        self._coeffs = [self._lms_coeffs(i, min(i + 1, 4)) for i in range(num_inference_steps)]

    def get_lms_coefficient(self, order: int, t: int, current_order: int) -> float:
        sig = self.sigmas

        def lms_derivative(tau):
            prod = 1.0
            for k in range(order):
                if current_order == k:
                    continue
                prod *= (tau - sig[t - k]) / (sig[t - current_order] - sig[t - k])
            return prod

        return integrate.quad(lms_derivative, sig[t], sig[t + 1], epsrel=1e-4)[0]

    def _lms_coeffs(self, step_index: int, order: int) -> List[float]:
        return [float(self.get_lms_coefficient(order, step_index, o)) for o in range(order)]

    def step_index_of(self, timestep) -> int:
        """Host lookup of the schedule position of `timestep` (no device sync)."""
        t = float(timestep)
        for i, v in enumerate(self._t_list):
            if v == t:
                return i
        raise ValueError(f"timestep {t} is not on the schedule")

    # ---- per-step ------------------------------------------------------------------------
    def scale_model_input(self, sample: torch.Tensor, timestep) -> torch.Tensor:
        sigma = float(self.sigmas[self.step_index_of(timestep)])
        return sample / ((sigma ** 2 + 1) ** 0.5)

    def step(self, model_output: torch.Tensor, timestep, sample: torch.Tensor, order: int = 4):
        i = self.step_index_of(timestep)
        sigma = float(self.sigmas[i])
        pred_original_sample = sample - sigma * model_output       # epsilon prediction
        derivative = (sample - pred_original_sample) / sigma
        self.derivatives.append(derivative)
        if len(self.derivatives) > order:
            self.derivatives.pop(0)
        order = min(i + 1, order)
        coeffs = self._coeffs[i][:order] if (self._coeffs is not None and order == min(i + 1, 4)) \
            else self._lms_coeffs(i, order)
        prev_sample = sample + sum(c * d for c, d in zip(coeffs, reversed(self.derivatives)))
        return _StepOutput(prev_sample, pred_original_sample)

    def add_noise(self, original_samples: torch.Tensor, noise: torch.Tensor, timesteps) -> torch.Tensor:
        idx = [self.step_index_of(t) for t in timesteps]
        sigma = self.sigmas[idx].flatten().to(original_samples.device, original_samples.dtype)
        while sigma.dim() < original_samples.dim():
            sigma = sigma.unsqueeze(-1)
        return original_samples + noise * sigma


# ---------------------------------------------------------------------------------------------
# single-evaluation sigma samplers: Euler, Euler ancestral, DPM-Solver++(2M)
# ---------------------------------------------------------------------------------------------
class _CoefficientScheduler:
    """Sigma (VE) parametrisation shared with `LMSDiscreteScheduler`: `scale_model_input` divides by sqrt(sigma^2+1),
    `add_noise` adds sigma * noise, `init_noise_sigma` is the train schedule's largest sigma.

    Per step i (sigma = sigmas[i], sigma' = sigmas[i+1]) with x0 = x - sigma * eps every update here has the form
        x' = a*x + b*eps + c*x0 + d*x0_prev + s*noise
    and `coefficients(i, first)` returns (a, b, c, d, s).  `first` marks the first step of a run (a run may start
    mid-schedule, as img2img does).  The same row drives `step` here and the device kernel of `PwWSampler`.

    `use_karras_sigmas=True` spaces sigma as Karras et al. (2022), rho = 7, between the train schedule's sigma_min and
    sigma_max; the timesteps are then the fractional positions of those sigmas on the train schedule (log-sigma
    interpolation), which the UNet's sinusoidal embedding takes as floats.
    """
    order = 1
    ancestral = False

    def __init__(self, num_train_timesteps: int = 1000, beta_start: float = 0.0001, beta_end: float = 0.02,
                 beta_schedule: str = "linear", use_karras_sigmas: bool = False):
        if beta_schedule == "linear":
            betas = np.linspace(beta_start, beta_end, num_train_timesteps, dtype=np.float32)
        elif beta_schedule == "scaled_linear":
            betas = np.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=np.float32) ** 2
        else:
            raise NotImplementedError(beta_schedule)
        self.config = {"num_train_timesteps": num_train_timesteps, "beta_start": beta_start,
                       "beta_end": beta_end, "beta_schedule": beta_schedule, "use_karras_sigmas": bool(use_karras_sigmas)}
        self.use_karras_sigmas = bool(use_karras_sigmas)
        self.betas = torch.from_numpy(betas)
        self.alphas_cumprod = torch.cumprod(1.0 - self.betas, dim=0)
        ac = self.alphas_cumprod.numpy()
        self._train_sig = np.array(((1 - ac) / ac) ** 0.5)
        self.sigmas = torch.from_numpy(np.concatenate([self._train_sig[::-1], [0.0]]).astype(np.float32))
        self.init_noise_sigma = self.sigmas.max()
        self.timesteps = torch.from_numpy(
            np.linspace(0, num_train_timesteps - 1, num_train_timesteps, dtype=float)[::-1].copy())
        self.num_inference_steps: Optional[int] = None
        self._t_list: List[float] = self.timesteps.tolist()
        self._prev_index: Optional[int] = None       # host `step` state: schedule index and x0 of the previous step
        self._x0_prev: Optional[torch.Tensor] = None

    @classmethod
    def from_config(cls, config, **kwargs):
        """diffusers idiom `NewScheduler.from_config(pipe.scheduler.config)`: keys this class does not take are ignored."""
        import inspect
        accepted = set(inspect.signature(cls.__init__).parameters) - {"self"}
        args = {k: v for k, v in dict(config).items() if k in accepted}
        args.update(kwargs)
        return cls(**args)

    # ---- schedule ------------------------------------------------------------------------
    def set_timesteps(self, num_inference_steps: int, device=None):
        self.num_inference_steps = num_inference_steps
        n_train = self.config["num_train_timesteps"]
        sig_train = self._train_sig
        if self.use_karras_sigmas:
            rho = 7.0
            smin, smax = float(sig_train[0]), float(sig_train[-1])
            ramp = np.linspace(0, 1, num_inference_steps)
            sig = (smax ** (1 / rho) + ramp * (smin ** (1 / rho) - smax ** (1 / rho))) ** rho
            timesteps = np.interp(np.log(sig), np.log(sig_train), np.arange(0, len(sig_train), dtype=float))
        else:
            timesteps = np.linspace(0, n_train - 1, num_inference_steps, dtype=float)[::-1].copy()
            sig = np.interp(timesteps, np.arange(0, len(sig_train)), sig_train)
        self.sigmas = torch.from_numpy(np.concatenate([sig, [0.0]]).astype(np.float32))
        self.timesteps = torch.from_numpy(np.ascontiguousarray(timesteps, dtype=float)).to(device=device)
        self._t_list = self.timesteps.tolist()
        self._prev_index, self._x0_prev = None, None

    def step_index_of(self, timestep) -> int:
        """Host lookup of the schedule position of `timestep` (no device sync)."""
        t = float(timestep)
        for i, v in enumerate(self._t_list):
            if v == t:
                return i
        raise ValueError(f"timestep {t} is not on the schedule")

    def coefficients(self, step_index: int, first: bool) -> Tuple[float, float, float, float, float]:
        raise NotImplementedError

    # ---- per-step ------------------------------------------------------------------------
    def scale_model_input(self, sample: torch.Tensor, timestep) -> torch.Tensor:
        sigma = float(self.sigmas[self.step_index_of(timestep)])
        return sample / ((sigma ** 2 + 1) ** 0.5)

    def step(self, model_output: torch.Tensor, timestep, sample: torch.Tensor, noise: Optional[torch.Tensor] = None,
             generator: Optional[torch.Generator] = None, return_dict: bool = True):
        """One update.  Ancestral samplers add `noise` (drawn from `generator` when not given)."""
        i = self.step_index_of(timestep)
        first = self._prev_index is None or self._prev_index != i - 1
        a, b, c, d, s = self.coefficients(i, first)
        sigma = float(self.sigmas[i])
        x0 = sample - sigma * model_output
        prev = a * sample + b * model_output + c * x0
        if d != 0.0:
            prev = prev + d * self._x0_prev
        if s != 0.0:
            if noise is None:
                noise = torch.randn(sample.shape, generator=generator, dtype=sample.dtype).to(sample.device)
            prev = prev + s * noise.to(sample.device, sample.dtype)
        self._prev_index, self._x0_prev = i, x0
        out = _StepOutput(prev, x0)
        return out if return_dict else (prev,)

    def add_noise(self, original_samples: torch.Tensor, noise: torch.Tensor, timesteps) -> torch.Tensor:
        idx = [self.step_index_of(t) for t in timesteps]
        sigma = self.sigmas[idx].flatten().to(original_samples.device, original_samples.dtype)
        while sigma.dim() < original_samples.dim():
            sigma = sigma.unsqueeze(-1)
        return original_samples + noise * sigma


class EulerDiscreteScheduler(_CoefficientScheduler):
    """Euler (k-diffusion `sample_euler`; diffusers 0.10 `EulerDiscreteScheduler` with s_churn = 0):
    x' = x + (sigma' - sigma) * eps."""

    def coefficients(self, step_index, first):
        s0, s1 = float(self.sigmas[step_index]), float(self.sigmas[step_index + 1])
        return 1.0, s1 - s0, 0.0, 0.0, 0.0


class EulerAncestralDiscreteScheduler(_CoefficientScheduler):
    """Euler ancestral (k-diffusion `sample_euler_ancestral`, eta = 1; diffusers 0.10
    `EulerAncestralDiscreteScheduler`): sigma_up = sqrt(sigma'^2 (sigma^2 - sigma'^2) / sigma^2),
    sigma_down = sqrt(sigma'^2 - sigma_up^2), x' = x + (sigma_down - sigma) * eps + sigma_up * noise."""
    ancestral = True

    def coefficients(self, step_index, first):
        s0, s1 = float(self.sigmas[step_index]), float(self.sigmas[step_index + 1])
        up = math.sqrt(s1 * s1 * (s0 * s0 - s1 * s1) / (s0 * s0))
        down = math.sqrt(max(s1 * s1 - up * up, 0.0))
        return 1.0, down - s0, 0.0, 0.0, up


class DPMSolverMultistepScheduler(_CoefficientScheduler):
    """DPM-Solver++(2M) (Lu et al. 2022; k-diffusion `sample_dpmpp_2m`) in the sigma parametrisation, rho = sigma'/sigma:
      first step of a run, or sigma' = 0:  x' = rho*x + (1 - rho)*x0
      otherwise, h = ln(sigma/sigma'), r = ln(sigma_prev/sigma)/h:
          x' = rho*x + (1 - rho)*((1 + 1/(2r))*x0 - x0_prev/(2r))
    The final step (sigma' = 0) is first order as in k-diffusion, which not every diffusers release does.  Only
    algorithm_type="dpmsolver++" with solver_order=2 is implemented."""

    def __init__(self, num_train_timesteps: int = 1000, beta_start: float = 0.0001, beta_end: float = 0.02,
                 beta_schedule: str = "linear", use_karras_sigmas: bool = False, solver_order: int = 2,
                 algorithm_type: str = "dpmsolver++"):
        if algorithm_type != "dpmsolver++":
            raise ValueError(f"algorithm_type={algorithm_type!r} is not implemented (only 'dpmsolver++')")
        if solver_order != 2:
            raise ValueError(f"solver_order={solver_order} is not implemented (only 2)")
        super().__init__(num_train_timesteps, beta_start, beta_end, beta_schedule, use_karras_sigmas)
        self.config.update(solver_order=solver_order, algorithm_type=algorithm_type)

    def coefficients(self, step_index, first):
        s0, s1 = float(self.sigmas[step_index]), float(self.sigmas[step_index + 1])
        rho = s1 / s0
        if first or s1 == 0.0 or step_index == 0:
            return rho, 0.0, 1.0 - rho, 0.0, 0.0
        h = math.log(s0 / s1)
        r = math.log(float(self.sigmas[step_index - 1]) / s0) / h
        return rho, 0.0, (1.0 - rho) * (1.0 + 1.0 / (2.0 * r)), -(1.0 - rho) / (2.0 * r), 0.0


SIGMA_SAMPLERS = (EulerDiscreteScheduler, EulerAncestralDiscreteScheduler, DPMSolverMultistepScheduler)
