"""GaussianApproxLKernel (reference: smcnuts/lkernel/gaussian_lkernel.py:24-84).

Unweighted mean/covariance of X = [-r_new, x_new], conditional Gaussian of -r_new given x_new with a 1e-6
ridge, evaluated per particle -- as four CUDA kernels (csrc/gauss_lkernel.cu) instead of a Python loop with a
pinv and an eigendecomposition per particle.  When particles are sharded over ranks the moment sums are
all-reduced (the only collective of this L-kernel)."""
from .. import _cabi, _device as dev
from ..parallel import ShardContext


class GaussianApproxLKernel:
    RIDGE = 1e-6  # gaussian_lkernel.py:68

    def __init__(self, target, N: int, shard: ShardContext = None):
        self.D = target.dim
        self.N = N            # GLOBAL particle count (np.cov ddof = 1 uses it)
        self.shard = shard or ShardContext()
        self.last_status = None   # device tensor [logdet, path] of the last call: path 0 Cholesky, 1 pinv fallback, -1 failed

    def calculate_L(self, r_new, x_new):
        D = self.D
        r = dev.to_device(r_new).reshape(-1, D)
        x = dev.to_device(x_new).reshape(-1, D)
        n = r.shape[0]
        st = dev.stream_ptr()
        n_total = int(self.shard.all_reduce_sum_scalar(n))
        sums = dev.empty(2 * D)
        _cabi.call("smcb_gaussL_sums", dev.ptr(r), dev.ptr(x), n, D, dev.ptr(sums), st)
        self.shard.all_reduce_sum_(sums)
        mean = dev.empty(2 * D)
        _cabi.call("smcb_affine", dev.ptr(sums), 2 * D, 1.0 / n_total, 0.0, dev.ptr(mean), st)
        gram = dev.zeros(2 * D, 2 * D)
        _cabi.call("smcb_gaussL_gram", dev.ptr(r), dev.ptr(x), n, D, dev.ptr(mean), dev.ptr(gram), st)
        self.shard.all_reduce_sum_(gram)
        G, logdet, scratch = dev.empty(D, 2 * D), dev.empty(2), dev.empty(6 * D * D)
        _cabi.call("smcb_gaussL_factor", dev.ptr(gram), n_total, D, self.RIDGE, dev.ptr(G), dev.ptr(logdet),
                   dev.ptr(scratch), st)
        self.last_status = logdet
        out = dev.empty(n)
        nfrag = _cabi.lib().smcb_gaussL_logpdf_scratch_bytes(D) // 8
        frag = dev.empty(nfrag) if nfrag else None   # None: D > 104 takes the scalar kernel, which needs no scratch
        _cabi.call("smcb_gaussL_logpdf", dev.ptr(r), dev.ptr(x), n, D, dev.ptr(mean), dev.ptr(G), dev.ptr(logdet),
                   dev.ptr(out), dev.ptr(frag), st)
        return dev.like_input(out, x_new)
