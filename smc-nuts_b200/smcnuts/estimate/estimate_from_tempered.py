"""EstimateFromTempered (reference: smcnuts/estimate/estimate_from_tempered.py:24-55): for every saved
iteration k, resample x_saved[k] by logw_saved[k], re-weight by pi(x)/pi(x, phi_k) = exp((1-phi_k)*loglik)
and form mean/variance estimates."""
import numpy as np

from .. import _cabi, _device as dev
from ..parallel import ShardContext
from ..samples.samples import Resampler, normalise
from .estimate import Estimate


class EstimateFromTempered(Estimate):
    def __init__(self, target, N, K, rng, shard: ShardContext = None, resampling="multinomial"):
        super().__init__(target, shard)
        self.N, self.K, self.rng = N, K, rng
        self.seed = dev.seed_from_rng(rng)
        self.resampler = Resampler(N, self.seed, self.shard, stream=_cabi.STREAM_ESTIMATE, scheme=resampling)

    def estimate_from_tempered(self, x_saved, logw_saved, phi):
        D = getattr(self.target, "constrained_dim", self.target.dim)     # estimates are on the constrained scale
        host = dev.is_host(x_saved)
        mean_e, var_e = np.zeros([self.K + 1, D]), np.zeros([self.K + 1, D])
        for k in range(self.K + 1):
            xk, lwk = dev.to_device(x_saved[k]), dev.to_device(logw_saved[k])
            wn, _, _, scan = normalise(lwk, self.shard, scan=True)
            x = self.resampler.resample_rows(xk, wn, iteration=k, scan=scan)
            A, B = self.target.split(x)
            lw = dev.empty(x.shape[0])
            # logpdf(x, 1) - logpdf(x, phi_k)  (estimate_from_tempered.py:47)
            zero = dev.zeros(x.shape[0])
            _cabi.call("smcb_reweight_asymptotic", dev.ptr(zero), dev.ptr(A), dev.ptr(B), 1.0, float(phi[k]),
                       x.shape[0], dev.ptr(lw), dev.stream_ptr())
            wn2, _, _ = normalise(lw, self.shard)
            m, v = self.return_estimate(x, wn2)
            mean_e[k], var_e[k] = m.cpu().numpy(), v.cpu().numpy()
        del host
        return mean_e, var_e
