"""GP prior base classes — the reference's `gpr_lib/GP_prior/GP_prior.py` surface for the rollout hot path.

Same class names, constructor arguments, parameter names (`sigma_n_log`) and method signatures as the reference
(GP_prior :22-257, Combine_GP :260-296, Sum_Independent_GP :299-347), so reference `state_dict`s load unchanged
and callers need no edits.  What differs is where the arithmetic runs: a kernel tree is flattened once into a
POD `McpGpSpec` (`_fill_spec`) and every covariance / factorisation / posterior is one call into
libmcpilco_b200.so (CUDA, float64).  CPU tensors are rejected: there is no fallback.

Out of scope here (SURVEY.md §2 row 1): `fit_model` (hyper-parameter training), `Multiply_GP_prior`, `Scale_GP_prior`.
"""
import time

import numpy as np
import torch

from ... import _native as _N
from ... import _ops as ops
from ... import _pack as P


class GP_prior(torch.nn.Module):
    """Superclass of the GP models (reference GP_prior.py:22-257)."""

    def __init__(self, active_dims, sigma_n_init=None, flg_train_sigma_n=True, name="", dtype=torch.float64, sigma_n_num=None,
                 device=None):
        super().__init__()
        self.name = name
        self.dtype = dtype
        self.device = torch.device("cpu") if device is None else device
        self.active_dims = None if active_dims is None else torch.tensor(active_dims, requires_grad=False, device=device, dtype=torch.long)
        self.GP_with_noise = sigma_n_init is not None
        if self.GP_with_noise:
            self.sigma_n_log = torch.nn.Parameter(torch.tensor(np.log(sigma_n_init), dtype=self.dtype, device=self.device),
                                                  requires_grad=flg_train_sigma_n)
        self.sigma_n_num = torch.as_tensor(0.0 if sigma_n_num is None else sigma_n_num, dtype=self.dtype, device=self.device)
        self._spec_cache = {}

    # ---- bookkeeping identical in behaviour to the reference -------------------------------------------------
    def to(self, dev):
        super().to(dev)
        self.device = dev
        self.sigma_n_num = self.sigma_n_num.to(dev)
        if self.active_dims is not None:
            self.active_dims = self.active_dims.to(dev)

    def set_eval_mode(self):
        self.flg_trainable_list = []
        for p in self.parameters():
            self.flg_trainable_list.append(p.requires_grad)
            p.requires_grad = False

    def set_training_mode(self):
        for i, p in enumerate(self.parameters()):
            p.requires_grad = self.flg_trainable_list[i]

    def get_sigma_n_2(self):
        return torch.exp(self.sigma_n_log) ** 2 + self.sigma_n_num ** 2

    def print_model(self):
        print(self.name + " parameters:")
        for par_name, par_value in self.named_parameters():
            print("-", par_name, ":", par_value.data)

    # ---- flattening ----------------------------------------------------------------------------------------
    # A kernel is described ONCE, as differentiable torch expressions of its parameters (`_kernel_terms`); the POD spec the
    # CUDA kernels take is their value, and the hyper-parameter gradients of the training objective are obtained by pushing
    # the native gradient w.r.t. the spec fields back through those same expressions (tiny tensors, torch autograd).
    def _kernel_terms(self, D):
        """{"inv_ls": Tensor[D] | None, "lam": 0-dim Tensor, "mean": 0-dim Tensor | None, "polys": [Tensor[deg, D + 1], ...]}:
        k(x,x') = lam exp(-sum_j ((x_j - x'_j) inv_ls_j)^2) + sum_p prod_f (sum_j W_p[f, j] x_j x'_j + W_p[f, D])."""
        raise NotImplementedError()

    def _noise_term(self):
        return self.get_sigma_n_2().reshape(()) if self.GP_with_noise else None

    def _scatter(self, values, D, extra=0):
        """Place per-active-dimension values into a length D (+extra) vector (zeros elsewhere), differentiably."""
        out = torch.zeros(D + extra, dtype=self.dtype, device=values.device)
        return out.index_put((self.active_dims.to(values.device),), values)

    def gp_spec(self, D):
        """McpGpSpec of this kernel for a D-dimensional gp input; rebuilt only when a parameter changed."""
        key = (int(D),) + tuple((id(p), p._version, p.data_ptr(), tuple(p.shape)) for p in self.parameters())  # `p.data = ...` keeps _version
        hit = self._spec_cache.get("k")
        if hit is not None and hit[0] == key:
            return hit[1]
        with torch.no_grad():
            t = self._kernel_terms(int(D))
            sn2 = self._noise_term()
        spec = P.new_gp_spec(int(D))
        if t.get("inv_ls") is not None:
            spec.has_se = 1
            spec.lambda_ = float(t["lam"])
            for j, v in enumerate(P._np(t["inv_ls"]).reshape(-1)):
                spec.inv_ls[j] = float(v)
        polys = t.get("polys", [])
        if len(polys) > _N.MAX_POLY:
            raise NotImplementedError("more than %d polynomial terms" % _N.MAX_POLY)
        for p, W in enumerate(polys):
            W = P._np(W)
            if W.shape[0] > _N.MAX_DEG:
                raise NotImplementedError("polynomial degree above %d" % _N.MAX_DEG)
            spec.poly_deg[p] = W.shape[0]
            for f in range(W.shape[0]):
                for j in range(int(D)):
                    spec.poly_w2[p][f][j] = float(W[f, j])
                spec.poly_w2[p][f][_N.MAX_D] = float(W[f, int(D)])
        spec.n_poly = len(polys)
        if not spec.has_se and not spec.n_poly:
            raise RuntimeError("empty kernel")
        spec.mean0 = float(t["mean"]) if t.get("mean") is not None else 0.0
        spec.sigma_n2 = float(sn2) if sn2 is not None else 0.0
        self._spec_cache["k"] = (key, spec)
        return spec

    # ---- arithmetic: all native ------------------------------------------------------------------------------
    def get_mean(self, X):
        """Constant prior mean in X, [N, 1]."""
        return torch.full((X.shape[0], 1), self.gp_spec(X.shape[1]).mean0, dtype=self.dtype, device=X.device)

    def get_covariance(self, X1, X2=None, flg_noise=False):
        """k(X1, X2); the noise variance is added on the diagonal only for X2=None, flg_noise and a noisy GP."""
        return ops.gp_covariance(self.gp_spec(X1.shape[1]), X1, X2, add_noise=bool(flg_noise) and self.GP_with_noise and X2 is None)

    def get_diag_covariance(self, X, flg_noise=False):
        d = ops.gp_diag_covariance(self.gp_spec(X.shape[1]), X)
        if flg_noise and self.GP_with_noise:
            d = d + self.gp_spec(X.shape[1]).sigma_n2
        return d

    def forward(self, X):
        """(m_X, K_X, K_X^-1, log det K_X) through the blocked Cholesky of the precompute (reference :91-115).  While
        hyper-parameters are being trained (grad enabled and some parameter requires grad) the four outputs are produced
        lazily: Marginal_log_likelihood consumes the handle directly and evaluates loss + analytic gradient in one native call."""
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            return PriorOutput(self, X)
        return self._forward_values(X)

    def _forward_values(self, X):
        spec = self.gp_spec(X.shape[1])
        K_X = ops.gp_covariance(spec, X, None, add_noise=self.GP_with_noise)
        zero = torch.zeros(X.shape[0], 1, dtype=self.dtype, device=X.device)
        _, K_X_inv, L = ops.gp_precompute(spec, X, zero, want_L=True)
        log_det = 2 * torch.sum(torch.log(torch.diagonal(L)))
        return self.get_mean(X), K_X, K_X_inv, log_det

    def get_alpha(self, X, Y):
        """alpha = K_X^-1 (Y - m_X)  (reference :130-135)."""
        alpha, K_X_inv, Linv = ops.gp_precompute(self.gp_spec(X.shape[1]), X, Y, want_Linv=True)
        # the triangular factor rides along on the K_X_inv tensor object (the reference's return signature has no slot for it):
        # forward-only posteriors built from THIS tensor use it; any other K_X_inv (a loaded log, a modified copy) takes the full product
        ops.attach_linv(K_X_inv, Linv)
        return alpha, self.get_mean(X), K_X_inv

    def get_estimate_from_alpha(self, X, X_test, alpha, m_X, K_X_inv=None, Y_test=None):
        """Posterior mean (and variance when K_X_inv is given) at X_test (reference :137-155).

        Differentiable (once) w.r.t. X_test in both forms; the GP's parameters, X, alpha and K_X_inv receive no gradient.  With grad
        mode on and X_test requiring grad the posterior takes the Jacobian path (the full product with K_X_inv, never the triangular
        factor; without K_X_inv, a zero [N, N] matrix stands in for it and only the mean is returned)."""
        spec = self.gp_spec(X.shape[1])
        if K_X_inv is None and torch.is_grad_enabled() and X_test.requires_grad:
            Y_hat, _ = ops.gp_predict([ops.FittedGp(spec, X, alpha, X.new_zeros(X.shape[0], X.shape[0]))], X_test)
            var = None
        elif K_X_inv is None:
            Y_hat = self.get_mean(X_test) + ops.gp_covariance(spec, X_test, X) @ alpha.reshape(-1, 1)
            var = None
        else:
            mean, var = ops.gp_predict([ops.FittedGp(spec, X, alpha, K_X_inv)], X_test)
            Y_hat, var = mean, var[:, 0]
        if Y_test is not None:
            print("MSE:", torch.sum((Y_test - Y_hat) ** 2) / Y_test.size()[0])
        return Y_hat if var is None else (Y_hat, var)

    def get_estimate(self, X, Y, X_test, Y_test=None, flg_return_K_X_inv=False):
        """Fit on (X, Y), predict at X_test (reference :157-171)."""
        alpha, m_X, K_X_inv = self.get_alpha(X, Y)
        Y_hat, var = self.get_estimate_from_alpha(X, X_test, alpha, m_X, K_X_inv=K_X_inv, Y_test=Y_test)
        if flg_return_K_X_inv:
            return Y_hat, var, alpha, m_X, K_X_inv
        return Y_hat, var, alpha

    def get_SOD(self, X, Y, threshold, flg_permutation=False):
        """Greedy subset of data: a point joins the subset when the predictive std of the GP fitted on the current subset exceeds
        `threshold` at it (reference :232-257; the first sample always seeds the subset, the rest are visited in order or in a random
        permutation).  One native call: the Cholesky factor of the subset is grown row by row on the device instead of refitting per
        candidate (the prior mean does not enter the variance, so Y is not needed)."""
        n = X.shape[0]
        order = None
        if flg_permutation:
            order = [0] + (1 + torch.randperm(n - 1)).tolist()
        thr = float(P._np(threshold).reshape(-1)[0])
        return ops.gp_sod_select(self.gp_spec(X.shape[1]), X, thr, order)

    def nlml(self, X, Y):
        """0.5 ((Y - m)^T K^-1 (Y - m) + log det K) as a [1, 1] tensor whose backward fills the hyper-parameter gradients."""
        params = [p for p in self.parameters() if p.requires_grad]
        return _Nlml.apply(self, X, Y, *params)

    def fit_model(self, trainloader=None, optimizer=None, criterion=None, N_epoch=1, N_epoch_print=1, f_saving_model=None, f_print=None):
        """Hyper-parameter optimisation (reference :179-230): for every epoch and batch, loss = criterion(self(inputs), labels),
        backward, optimizer step."""
        print("\nInitial parameters:")
        self.print_model()
        t_start = time.time()
        for epoch in range(N_epoch):
            running_loss, n_btc = 0.0, 0
            optimizer.zero_grad()
            for inputs, labels in trainloader:
                optimizer.zero_grad()
                loss = criterion(self(inputs), labels)
                loss.backward()
                optimizer.step()
                running_loss, n_btc = running_loss + loss.detach(), n_btc + 1
            if epoch % N_epoch_print == 0:
                print("\nEPOCH:", epoch)
                self.print_model()
                print("Running loss:", float(running_loss) / n_btc, "| time elapsed:", time.time() - t_start)
                t_start = time.time()
                if f_saving_model is not None:
                    f_saving_model(epoch)
                if f_print is not None:
                    f_print()
        print("\nFinal parameters:")
        self.print_model()


class PriorOutput:
    """Handle returned by GP_prior.forward in training mode.  Unpacks like the reference's 4-tuple (values, no graph);
    Marginal_log_likelihood takes the fused route through `gp.nlml`."""

    def __init__(self, gp, X):
        self.gp, self.X = gp, X
        self._vals = None

    def _values(self):
        if self._vals is None:
            with torch.no_grad():
                self._vals = self.gp._forward_values(self.X)
        return self._vals

    def __iter__(self):
        return iter(self._values())

    def __getitem__(self, i):
        return self._values()[i]

    def __len__(self):
        return 4


class _Nlml(torch.autograd.Function):
    """loss = NLML(parameters): forward is one native call returning the value and the gradient w.r.t. the spec fields;
    backward pushes that gradient through the kernel's own `_kernel_terms` expressions."""

    @staticmethod
    def forward(ctx, gp, X, Y, *params):
        D = X.shape[1]
        out = ops.gp_nlml(gp.gp_spec(D), X, Y)
        ctx.gp, ctx.D, ctx.params = gp, D, params
        ctx.save_for_backward(out)
        return out[0].reshape(1, 1).clone()

    @staticmethod
    def backward(ctx, g):
        out, = ctx.saved_tensors
        gp, D = ctx.gp, ctx.D
        with torch.enable_grad():
            t = gp._kernel_terms(D)
            sn2 = gp._noise_term()
            outs, gouts = [], []
            if t.get("inv_ls") is not None:
                outs += [t["inv_ls"], t["lam"].reshape(())]
                gouts += [out[ops.NLML_ILS:ops.NLML_ILS + D], out[ops.NLML_LAMBDA]]
            for p, W in enumerate(t.get("polys", [])):
                rows = []
                for f in range(W.shape[0]):
                    o = ops.nlml_poly_offset(p, f)
                    rows.append(torch.cat([out[o:o + D], out[o + _N.MAX_D:o + _N.MAX_D + 1]]))
                outs.append(W)
                gouts.append(torch.stack(rows))
            if t.get("mean") is not None:
                outs.append(t["mean"].reshape(()))
                gouts.append(out[ops.NLML_MEAN])
            if sn2 is not None:
                outs.append(sn2)
                gouts.append(out[ops.NLML_SN2])
            keep = [(o, go) for o, go in zip(outs, gouts) if o.requires_grad]
            grads = torch.autograd.grad([o for o, _ in keep], ctx.params, [go.reshape(o.shape) * g.reshape(()) for o, go in keep],
                                        allow_unused=True)
        return (None, None, None) + tuple(grads)


class Combine_GP(GP_prior):
    """Common part of kernels built from several GP priors (reference :260-296)."""

    def __init__(self, *gp_priors_obj):
        super().__init__(active_dims=None, sigma_n_num=gp_priors_obj[0].sigma_n_num, dtype=gp_priors_obj[0].dtype,
                         device=gp_priors_obj[0].device)
        self.gp_list = torch.nn.ModuleList(gp_priors_obj)
        self.GP_with_noise = any(gp.GP_with_noise for gp in self.gp_list)

    def to(self, dev):
        super().to(dev)
        for gp in self.gp_list:
            gp.to(dev)

    def print_model(self):
        for gp in self.gp_list:
            gp.print_model()

    def get_sigma_n_2(self):
        s = torch.zeros(1, dtype=self.dtype, device=self.device)
        for gp in self.gp_list:
            if gp.GP_with_noise:
                s = s + gp.get_sigma_n_2()
        return s


class Sum_Independent_GP(Combine_GP):
    """Sum of independent GP priors: covariances add (reference :299-347).  The prior mean is the FIRST child's only —
    the reference's get_mean returns from inside its loop (:306-312) — and that is reproduced."""

    def _kernel_terms(self, D):
        out = {"inv_ls": None, "lam": None, "mean": None, "polys": []}
        for k, gp in enumerate(self.gp_list):
            t = gp._kernel_terms(D)
            if t.get("inv_ls") is not None:
                if out["inv_ls"] is not None:
                    raise NotImplementedError("only one squared-exponential term per GP is supported on the CUDA path")
                out["inv_ls"], out["lam"] = t["inv_ls"], t["lam"]
            out["polys"] += list(t.get("polys", []))
            if k == 0:
                out["mean"] = t.get("mean")  # the first child's mean only (reference :306-312)
        return out


class Multiply_GP_prior(Combine_GP):
    def __init__(self, *a, **k):
        raise NotImplementedError("Multiply_GP_prior is not used by any MC-PILCO configuration and is outside the hot path")


def Scale_GP_prior(*a, **k):
    raise NotImplementedError("Scale_GP_prior is not used by any MC-PILCO configuration and is outside the hot path")
