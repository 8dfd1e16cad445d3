"""GaussianProcess -- API shell, same as the reference's gaussian_proc/gaussian_process/gaussian_process.py:21-59, plus
prediction at new points (gaussian_proc/_predict.py)."""

from .._likelihood import Likelihood

__all__ = ['GaussianProcess']


class GaussianProcess(object):
    """Gaussian process for regression: ``GaussianProcess(X, K, likelihood_method='direct').train(z)``, then
    ``predict(test_points, X_test)``. ``K`` may be a NumPy array / SciPy CSR matrix (copied to the GPU) or a device handle
    returned by ``generate_correlation(..., device=True)``."""

    def __init__(self, X, K, likelihood_method='direct', imate_method=None, imate_options={}):
        self.X = X
        self.K = K
        self.likelihood = Likelihood(X, K, likelihood_method=likelihood_method, imate_method=imate_method,
                                     imate_options=imate_options)
        self.results = None
        self.z = None

    def train(self, z, plot=False, interval_eta=None):
        """Finds the hyperparameters; prints the result dict like the reference (:52-59) and also returns it.
        ``interval_eta``: search interval of the profiled method (default: the reference's [1e-4, 1e3])."""
        results = self.likelihood.maximize_log_likelihood(z, plot=plot, interval_eta=interval_eta)
        self.results = results
        self.z = z
        print(results)
        return results

    def predict(self, test_points, X_test, return_var=True, return_cov=False, noise=False, chunk_size=8192):
        """Kriging mean at ``test_points`` (m* x d) with basis rows ``X_test`` (m* x m), at the trained sigma and eta; plus
        the variance (``return_var``) and the covariance (``return_cov``) of the latent values, or of new observations with
        ``noise=True``. Returns ``mean``, ``(mean, var)``, ``(mean, cov)`` or ``(mean, var, cov)``. Needs a dense K that
        knows its points, correlation_scale and nu (see ``Predictor``)."""
        return self._predictor('predict').predict(test_points, X_test, return_var=return_var, return_cov=return_cov,
                                                  noise=noise, chunk_size=chunk_size)

    def predict_gradient(self, test_points, X_test, X_test_grad, return_var=True, noise=False, chunk_size=8192):
        """Kriging mean at ``test_points`` and its gradient with respect to the test-point coordinates, at the trained
        sigma and eta; ``X_test_grad`` (m* x d x m) is the Jacobian of the basis rows, d X_test[j] / d test_points[j, k].
        Returns ``(mean, mean_grad)`` or, with ``return_var``, ``(mean, var, mean_grad, var_grad)``; the gradients are
        m* x d, and mean and var equal those of ``predict`` (see ``Predictor.predict_gradient``)."""
        return self._predictor('predict_gradient').predict_gradient(test_points, X_test, X_test_grad, return_var=return_var,
                                                                    noise=noise, chunk_size=chunk_size)

    def _predictor(self, what):
        if self.results is None:
            raise RuntimeError('train(z) must be called before %s().' % what)
        from .._predict import Predictor
        return Predictor(self.likelihood.K_mixed, self.X, self.z, self.results['eta'], sigma=self.results['sigma'])
