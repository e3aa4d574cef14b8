"""Estimate -- importance-sampling mean/variance (reference: smcnuts/estimate/estimate.py).

mean = wn' c(x), var = wn' (c(x) - mean)^2 in constrained space when the target has `constrained_dim`
(estimate.py:25-28,91-95); the constrain transform (bridgestan.py:93-120: exp on the last coordinate for
the shipped models) is fused into the moment kernel instead of N BridgeStan calls.
"""
from .. import _cabi, _device as dev
from ..parallel import ShardContext

MOMENT_COLS = 256     # widest row smcb_weighted_moment reduces in one launch


class Estimate:
    def __init__(self, target, shard: ShardContext = None):
        self.target = target
        self.shard = shard or ShardContext()
        if hasattr(self.target, "constrained_dim"):
            self._constrain = getattr(self.target, "constrain_kind", _cabi.CONSTRAIN_EXP_LAST)
        else:
            self._constrain = _cabi.CONSTRAIN_NONE

    def return_estimate(self, x, wn, center=None):
        """center (device tensor [D], optional): a point near the mean, e.g. the previous iteration's estimate -- the two
        moments then come from ONE pass over the particles and one collective (same estimates to rounding)."""
        if center is not None and self._constrain != _cabi.CONSTRAIN_MODEL and 2 * x.shape[1] <= 256 and not dev.is_host(x):
            return self._estimate_one_pass(x, wn, self._constrain, center)
        return self._estimate(x, wn, self._constrain)

    def _estimate_one_pass(self, x, wn, constrain, center):
        N, D = x.shape
        sums, mean, var = dev.empty(2 * D), dev.empty(D), dev.empty(D)
        st = dev.stream_ptr()
        _cabi.call("smcb_weighted_moments12", dev.ptr(x), dev.ptr(wn), N, D, constrain, dev.ptr(center), dev.ptr(sums),
                   dev.ptr(dev.reduce_ws()), st)
        self.shard.all_reduce_sum_(sums)
        _cabi.call("smcb_moments12_finalize", dev.ptr(sums), dev.ptr(center), D, dev.ptr(mean), dev.ptr(var), st)
        return mean, var

    def return_estimate_unconstrained(self, x, wn):
        return self._estimate(x, wn, _cabi.CONSTRAIN_NONE)

    def _estimate(self, x, wn, constrain=_cabi.CONSTRAIN_NONE):
        xd, wd = dev.to_device(x), dev.to_device(wn)
        if constrain == _cabi.CONSTRAIN_MODEL:     # generated models: [N, dim] -> [N, constrained_dim] through the plug-in
            xd, constrain = self.target.constrain(xd), _cabi.CONSTRAIN_NONE
        N, D = xd.shape
        if D > MOMENT_COLS:      # wide rows (generated quantities): column blocks, the exp-on-last in the last one only
            mean, var = dev.empty(D), dev.empty(D)
            for j in range(0, D, MOMENT_COLS):
                k = min(j + MOMENT_COLS, D)
                m, v = self._moments(xd[:, j:k].contiguous(), wd, constrain if k == D else _cabi.CONSTRAIN_NONE)
                mean[j:k].copy_(m)
                var[j:k].copy_(v)
        else:
            mean, var = self._moments(xd, wd, constrain)
        return dev.like_input(mean, x), dev.like_input(var, x)

    def _moments(self, xd, wd, constrain):
        N, D = xd.shape
        mean, var = dev.empty(D), dev.empty(D)
        ws, st = dev.reduce_ws(), dev.stream_ptr()
        _cabi.call("smcb_weighted_moment", dev.ptr(xd), dev.ptr(wd), N, D, constrain, 0, 1, dev.ptr(mean),
                   dev.ptr(ws), st)
        self.shard.all_reduce_sum_(mean)
        _cabi.call("smcb_weighted_moment", dev.ptr(xd), dev.ptr(wd), N, D, constrain, dev.ptr(mean), 2, dev.ptr(var),
                   dev.ptr(ws), st)
        self.shard.all_reduce_sum_(var)
        return mean, var
