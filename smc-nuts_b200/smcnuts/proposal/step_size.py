"""Dual-averaging step-size adaptation for the NUTS proposal.

Not in the reference: its step size is a constant of the run (nuts.py:31) and README.md:66-67 lists "step-size
adaptation" under future updates (SURVEY.md section 8 f4).  Off by default; `SMCSampler(..., adapt_step_size=K_adapt)`
turns it on for the first K_adapt iterations, after which the averaged step size is frozen.

The statistic is the one of Hoffman & Gelman (2014), Algorithm 6: for every particle the mean over the leaves of its tree
of min(1, exp(joint_leaf - joint_0)), accumulated inside the NUTS kernel (csrc/nuts_lane.cuh, `accept_stat`), summed over
the particles by smcb_sum_f64 and, when the particles are sharded, all-reduced.  An SMC iteration therefore yields ONE
very low-noise observation (N trees), so a handful of iterations is enough.  Constants are Stan's defaults.
"""
import math


class DualAveragingStepSize:
    def __init__(self, step_size, target_accept=0.8, gamma=0.05, t0=10.0, kappa=0.75):
        if not (0.0 < target_accept < 1.0):
            raise ValueError("target_accept must lie in (0, 1)")
        self.step_size = float(step_size)
        self.target_accept, self.gamma, self.t0, self.kappa = float(target_accept), float(gamma), float(t0), float(kappa)
        self.mu = math.log(10.0 * self.step_size)
        self.t = 0
        self.h_bar = 0.0
        self.log_eps_bar = 0.0

    def update(self, accept_mean):
        """One observation of the mean acceptance statistic at the current step size -> the next step size."""
        a = float(accept_mean)
        if not (a == a):        # NaN: every tree of the iteration diverged at its first leaf
            a = 0.0
        a = min(1.0, max(0.0, a))
        self.t += 1
        w = 1.0 / (self.t + self.t0)
        self.h_bar = (1.0 - w) * self.h_bar + w * (self.target_accept - a)
        log_eps = self.mu - math.sqrt(self.t) / self.gamma * self.h_bar
        eta = self.t ** (-self.kappa)
        self.log_eps_bar = eta * log_eps + (1.0 - eta) * self.log_eps_bar
        self.step_size = math.exp(log_eps)
        return self.step_size

    def rescale(self, factor):
        """The metric changed: a step of eps in the old z-units is one of eps * factor in the new ones.  The averaging
        state moves with it (centre, current and averaged log step), and what has been learned about the acceptance
        (h_bar, t) is kept.  Restarting instead would set mu = log(10 eps) again, and the first update after a restart
        multiplies the step by 2.3 even at acceptance 0: with the metric changing every iteration, the step grew
        geometrically while every tree diverged."""
        d = math.log(float(factor))
        self.mu += d
        self.log_eps_bar += d if self.t else 0.0
        self.step_size *= float(factor)
        return self.step_size

    def averaged(self):
        """The step size to freeze once adaptation ends (the initial one if there was no observation)."""
        return math.exp(self.log_eps_bar) if self.t else self.step_size
