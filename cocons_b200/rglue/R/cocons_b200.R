# R side of the drop-in: these definitions replace R/RcppExports.R (the four dense entry points
# and sumsmoothlone keep their names, argument names and order) and the dense halves of
# R/neg2loglikelihood.R.  Everything else in the package (coco(), cocoOptim(), getModelLists(),
# getScale(), .cocons.getPen(), ...) stays as it is and keeps calling these.
#
# Not executable in this repository's build image (no R there); see INTEGRATION.md.

# ---- R/RcppExports.R:10-46 ---------------------------------------------------------------
sumsmoothlone <- function(x, lambda, alpha = 1e6) {
  .Call(`_cocons_sumsmoothlone`, x, lambda, alpha)
}

cov_rns <- function(theta, locs, x_covariates, smooth_limits) {
  .Call(`_cocons_cov_rns`, theta, locs, x_covariates, smooth_limits)
}

cov_rns_pred <- function(theta, locs, locs_pred, x_covariates, x_covariates_pred, smooth_limits) {
  .Call(`_cocons_cov_rns_pred`, theta, locs, locs_pred, x_covariates, x_covariates_pred, smooth_limits)
}

cov_rns_classic <- function(theta, locs, x_covariates) {
  .Call(`_cocons_cov_rns_classic`, theta, locs, x_covariates)
}

# R/RcppExports.R:59-74 (sparse / tapered model)
cov_rns_taper_pred <- function(theta, locs, locs_pred, x_covariates, x_covariates_pred, colindices, rowpointers,
                               smooth_limits) {
  .Call(`_cocons_cov_rns_taper_pred`, theta, locs, locs_pred, x_covariates, x_covariates_pred, colindices,
        rowpointers, smooth_limits)
}

cov_rns_taper <- function(theta, locs, x_covariates, colindices, rowpointers, smooth_limits) {
  .Call(`_cocons_cov_rns_taper`, theta, locs, x_covariates, colindices, rowpointers, smooth_limits)
}

# ---- fused objectives --------------------------------------------------------------------
# kind: 0 ML, 1 profile, 2 REML (include/cocons_b200.h).  The device returns
# c(status, logdet, logdet_w, rank, quad_1..quad_r); n*log(2*pi), the penalty and the `safe`
# logic stay here, exactly as in R/neg2loglikelihood.R.
.cocons.n2ll.device <- function(kind, theta_list, locs, x_covariates, smooth.limits, z, x_betas = NULL) {
  tryCatch(
    .Call(`_cocons_n2ll_dense`, as.integer(kind), theta_list[-1], locs, as.matrix(x_covariates),
          smooth.limits, as.matrix(z), if (is.null(x_betas)) NULL else as.matrix(x_betas), theta_list$mean),
    error = function(e) e)
}

.cocons.chol.failed <- function(out, safe) {
  # status > 0: the leading minor of that order is not positive definite - what base::chol
  # reports as an error at R/neg2loglikelihood.R:200
  if (inherits(out, "error")) stop(out)
  if (out[1] > 0) {
    if (safe) return(TRUE)
    stop("Cholesky error")
  }
  FALSE
}

# R/neg2loglikelihood.R:183-222
GetNeg2loglikelihood <- function(theta, par.pos, locs, x_covariates, smooth.limits, z, n, lambda, safe = TRUE) {
  theta_list <- cocons::getModelLists(theta = theta, par.pos = par.pos, type = "diff")
  out <- .cocons.n2ll.device(0L, theta_list, locs, x_covariates, smooth.limits, z)
  if (.cocons.chol.failed(out, safe)) return(1e+06)
  logdet <- out[2]
  quad <- out[-(1:4)]
  sum_logliks <- sum(n * log(2 * pi) + 2 * logdet + quad)
  sum_logliks + .cocons.getPen(n * dim(z)[2], lambda, theta_list, smooth.limits)
}

# R/neg2loglikelihood.R:127-165
GetNeg2loglikelihoodProfile <- function(theta, par.pos, locs, x_covariates, smooth.limits, z, n, x_betas,
                                        lambda, safe = TRUE) {
  theta_list <- cocons::getModelLists(theta = theta, par.pos = par.pos, type = "diff")
  out <- .cocons.n2ll.device(1L, theta_list, locs, x_covariates, smooth.limits, z, x_betas)
  if (.cocons.chol.failed(out, safe)) return(1e+06)
  sum_logliks <- sum(n * log(2 * pi) + 2 * out[2] + out[-(1:4)])
  sum_logliks + .cocons.getPen(n * dim(z)[2], lambda, theta_list, smooth.limits)
}

# R/neg2loglikelihood.R:241-291
GetNeg2loglikelihoodREML <- function(theta, par.pos, locs, x_covariates, x_betas, smooth.limits, z, n,
                                     lambda, safe = TRUE) {
  theta_list <- cocons::getModelLists(theta = theta, par.pos = par.pos, type = "diff")
  out <- .cocons.n2ll.device(2L, theta_list, locs, x_covariates, smooth.limits, z)
  if (.cocons.chol.failed(out, safe)) return(1e+06)
  p <- out[4]
  sum_logliks <- sum((n - p) * log(2 * pi) + 2 * out[2] + 2 * out[3] + out[-(1:4)])
  sum_logliks + .cocons.getPen((n - p) * dim(z)[2], lambda, theta_list, smooth.limits)
}

# ---- many points per call: the finite-difference points of cocoOptim, the points of getHessian ----------------
# One .Call evaluates every point of `thetas` (a list of parameter vectors) on a batch context, up to `batch` points
# per launch of the assembly and the factorisation (n <= 16 256 sites).  The values are those of the closures above,
# bit for bit, including `safe` -> 1e6 per point; with safe = FALSE the first point that is not PD stops.
#   bctx <- .Call(`_cocons_ctx_new_batch`, locs, as.matrix(x_covariates), as.matrix(z), 8L, 0L)
#   on.exit(.Call(`_cocons_ctx_free`, bctx))
#   (PROFILE: .Call(`_cocons_ctx_set_xbetas`, bctx, as.matrix(x_betas)); REML: z are the contrasts)
GetNeg2loglikelihoodBatch <- function(kind, thetas, par.pos, bctx, smooth.limits, n, r, lambda, safe = TRUE) {
  lists <- lapply(thetas, function(theta) cocons::getModelLists(theta = theta, par.pos = par.pos, type = "diff"))
  p <- length(lists[[1]]$scale)
  means <- if (kind == 0L) lapply(lists, function(l) l$mean) else NULL
  out <- .Call(`_cocons_ctx_n2ll_batch`, bctx, as.integer(kind), lapply(lists, function(l) l[-1]), p, r,
               smooth.limits, means)
  names(out) <- c("logdet", "quad", "logdet_w", "rank_x", "status")
  vapply(seq_along(lists), function(i) {
    if (out$status[i] < 0) stop("cocons_b200: evaluation ", i, " failed with status ", out$status[i])
    if (out$status[i] > 0) {
      if (safe) return(1e+06)
      stop("Cholesky error")
    }
    quad <- out$quad[, i]
    if (kind == 2L) {
      np <- out$rank_x
      sum((n - np) * log(2 * pi) + 2 * out$logdet[i] + 2 * out$logdet_w[i] + quad) +
        .cocons.getPen((n - np) * r, lambda, lists[[i]], smooth.limits)
    } else {
      sum(n * log(2 * pi) + 2 * out$logdet[i] + quad) + .cocons.getPen(n * r, lambda, lists[[i]], smooth.limits)
    }
  }, numeric(1))
}

# ---- tapered objectives (R/neg2loglikelihood.R:20-108) -----------------------------------
# The tapered matrix is factored densely on the device instead of by spam's sparse Cholesky, so `cholS`
# is accepted and unused.  A context per call keeps the closures drop-in; cocoOptim's sparse branch
# (R/optim.R:480-531) can build it once, attach the taper once and pass it through `ctx`.  For large n it can
# build a tiled context instead, which stores only the tiles of the factor that can be nonzero (n = 200 000 fits
# one GPU) and is passed through `ctx` the same way:
#   ctx <- .Call(`_cocons_ctx_new_taper_tiled`, locs, as.matrix(x_covariates), as.matrix(z),
#                ref_taper@colindices, ref_taper@rowpointers, ref_taper@entries, 0L)
#   on.exit(.Call(`_cocons_ctx_free`, ctx))
.cocons.n2ll.taper.device <- function(theta_list, ref_taper, locs, x_covariates, smooth.limits, z, ctx = NULL) {
  tryCatch({
    if (is.null(ctx)) {
      ctx <- .Call(`_cocons_ctx_new`, locs, as.matrix(x_covariates), as.matrix(z), 0L)
      on.exit(.Call(`_cocons_ctx_free`, ctx))
      .Call(`_cocons_ctx_set_taper`, ctx, ref_taper@colindices, ref_taper@rowpointers, ref_taper@entries)
    }
    .Call(`_cocons_ctx_n2ll_taper`, ctx, theta_list[-1], ncol(as.matrix(x_covariates)), ncol(as.matrix(z)),
          smooth.limits, theta_list$mean)
  }, error = function(e) e)
}

GetNeg2loglikelihoodTaper <- function(theta, par.pos, ref_taper, locs, x_covariates, smooth.limits, cholS, z, n,
                                      lambda, safe = TRUE, ctx = NULL) {
  theta_list <- cocons::getModelLists(theta = theta, par.pos = par.pos, type = "diff")
  out <- .cocons.n2ll.taper.device(theta_list, ref_taper, locs, x_covariates, smooth.limits, z, ctx)
  if (.cocons.chol.failed(out, safe)) return(1e+06)
  sumlogs <- sum(n * log(2 * pi) + 2 * out[2] + out[-(1:2)])
  sumlogs + .cocons.getPen(n * dim(z)[2], lambda, theta_list, smooth.limits)
}

GetNeg2loglikelihoodTaperProfile <- function(theta, par.pos, ref_taper, locs, x_covariates, smooth.limits, cholS,
                                             z, n, lambda, safe = TRUE, ctx = NULL) {
  theta_list <- cocons::getModelLists(theta = theta, par.pos = par.pos, type = "diff")
  theta_list$std.dev[1] <- 0
  out <- .cocons.n2ll.taper.device(theta_list, ref_taper, locs, x_covariates, smooth.limits, z, ctx)
  if (.cocons.chol.failed(out, safe)) return(1e+06)
  r <- dim(z)[2]
  sum_in <- sum(out[-(1:2)])
  r * n * log(2 * pi) + r * n + r * 2 * out[2] + r * n * log(sum_in / (r * n)) +
    .cocons.getPen(n * r, lambda, theta_list, smooth.limits)
}

# ---- factor reuse for cocoPredict / cocoSim ----------------------------------------------
# Replace R/predict.R:136-159 by
#   ctx  <- .Call(`_cocons_ctx_new`, coco.object@locs, X_std$std.covs, coco.object@z, 0L)
#   .Call(`_cocons_ctx_factor`, ctx, 0L, adjusted_eff_values[-1], ncol(X_std$std.covs), smooth.limits)
#   pr   <- .Call(`_cocons_ctx_predict`, ctx, newlocs, X_pred_std$std.covs, coco.resid)
#   stochastic_part <- pr[[1]];  rowSums(cov_pred * t(inv_cov)) == pr[[2]]        (:159, :173)
# and R/sim.R:162-172 by
#   draws <- .Call(`_cocons_ctx_sim`, ctx, iiderrors)        # == t(t(iiderrors) %*% cholS)
# with iiderrors still produced by set.seed()/rnorm() in R so that seeds reproduce.
#
# Sparse branches (R/predict.R:219-275, R/sim.R:193-218): with taper_two / pred_taper still holding the
# TAPER values (before `@entries * cov_rns_taper*()`),
#   .Call(`_cocons_ctx_set_taper`, ctx, taper_two@colindices, taper_two@rowpointers, taper_two@entries)
#   .Call(`_cocons_ctx_factor_taper`, ctx, adjusted_eff_values[-1], ncol(X_std$std.covs), smooth.limits)
#   pr <- .Call(`_cocons_ctx_predict_taper`, ctx, newlocs, X_pred_std$std.covs, pred_taper@colindices,
#               pred_taper@rowpointers, pred_taper@entries, coco.resid)
#   stochastic_part <- pr[[1]];  spam::rowSums(pred_taper * t(inv_cov)) == pr[[2]]   (:259, :274)
# and `_cocons_ctx_sim_taper` (or `_cocons_ctx_sim`) for the marginal draws (same distribution as
# t(iiderrors) %*% cholS un-permuted).  At sizes whose dense matrix does not fit, the same sequence runs on a tiled
# context, which takes no `_cocons_ctx_set_taper` (its pattern is fixed at creation):
#   ctx <- .Call(`_cocons_ctx_new_taper_tiled`, locs, X_std$std.covs, as.matrix(z), taper_two@colindices,
#                taper_two@rowpointers, taper_two@entries, 0L)
#   .Call(`_cocons_ctx_factor_taper`, ctx, ...);  pr <- .Call(`_cocons_ctx_predict_taper`, ctx, ...)
#   draws <- .Call(`_cocons_ctx_sim_taper`, ctx, iiderrors)
