# ldsr_b200.R -- drop-in R wrappers that route ldsr's EM fan-out through ONE batched GPU call.
#
# NOT EXERCISED IN THIS REPOSITORY (no R in the build image); the Python mirror ldsr_b200/api.py
# implements the same logic and is what the tests run.  Source these definitions after
# library(ldsr) (or paste them over the originals in R/LDS_reconstruction.R) -- names, arguments
# and return values are the reference's.
#
# Random numbers: make_init() is called here, on the R side, in the order the reference's
# workers would call it under registerDoSEQ() (fold-major, then ensemble member), so set.seed()
# gives the same initial values -- and hence the same selected restarts -- as the reference.

.theta_vec <- function(th) c(th$A, th$B, th$C, th$D, th$Q, th$R, th$mu1, th$V1)

.theta_list <- function(vec, p, q) {
  th <- list(A = matrix(vec[1]), B = matrix(vec[2:(p + 1)], 1, p), C = matrix(vec[p + 2]),
             D = matrix(vec[(p + 3):(p + q + 2)], 1, q), Q = matrix(vec[p + q + 3]),
             R = matrix(vec[p + q + 4]), mu1 = matrix(vec[p + q + 5]), V1 = matrix(vec[p + q + 6]))
  class(th) <- 'theta'
  th
}

# One batched call: `jobs` is a list of list(series = index, held = 1-based steps, init = list of theta)
.em_batch <- function(series, jobs, niter, tol, n.devices = 0L) {
  stride <- max(sapply(series, function(s) nrow(s$u) + nrow(s$v) + 6L))
  theta0 <- do.call(cbind, lapply(jobs, function(j) sapply(j$init, function(th) {
    v <- .theta_vec(th); c(v, rep(0, stride - length(v)))
  })))
  .Call('_ldsr_em_batch', series, as.integer(sapply(jobs, `[[`, 'series')),
        lapply(jobs, function(j) as.integer(j$held)),
        rep(seq_along(jobs), sapply(jobs, function(j) length(j$init))),
        theta0, as.integer(niter), as.numeric(tol), as.integer(n.devices), PACKAGE = 'ldsr')
}

.pick <- function(res, g, series, jobs) {
  b <- res$best[g]
  if (is.na(b)) stop('no restart produced a finite likelihood')
  s <- series[[jobs[[g]]$series]]
  first <- sum(sapply(jobs[seq_len(g - 1)], function(j) length(j$init)))
  list(theta = .theta_list(res$theta[, b], nrow(s$u), nrow(s$v)),
       fit = list(X = res$X[[g]], Y = res$Y[[g]], V = res$V[[g]], J = res$J[[g]], lik = res$lik[b]),
       lik = res$lik[b], init = jobs[[g]]$init[[b - first]])
}

# R/LDS_reconstruction.R:42-62
LDS_EM_restart <- function(y, u, v, init, niter = 1000, tol = 1e-5, return.init = TRUE) {
  series <- list(list(y = y, u = u, v = v))
  jobs <- list(list(series = 1L, held = integer(0), init = init))
  res <- .em_batch(series, jobs, niter, tol, 1L)
  if (any(res$status == 1L)) stop('inv(): matrix is singular')
  ans <- .pick(res, 1L, series, jobs)
  if (!return.init) ans$init <- NULL
  ans
}

# R/LDS_reconstruction.R:270-285 (kept for callers that use it directly)
one_lds_cv <- function(z, instPeriod, mu, y, u, v, method = 'EM', num.restarts = 20,
                       ub = NULL, lb = NULL, num.islands = 4, pop.per.island = 100,
                       niter = 1000, tol = 1e-6, use.raw = FALSE) {
  stopifnot(method == 'EM')
  y[instPeriod][z] <- NA
  result <- LDS_EM_restart(y, u, v, make_init(nrow(u), nrow(v), num.restarts), niter, tol, FALSE)
  if (use.raw) c(propagate(result$theta, u, v, y)$Y[instPeriod]) + mu
  else c(result$fit$Y[instPeriod]) + mu
}

# The fold loop of cvLDS (R/LDS_reconstruction.R:372-382) as one batch.  Call it in place of the
# `Ycv <- if (single) foreach(...) else foreach(...) %:% foreach(...)` block; everything before
# (:308-370) and after (:384-409) stays as it is.  use.raw = TRUE: the fold output is the selected
# fit's open-loop propagate(theta, u, v, y_fold)$Y[instPeriod] + mu (:279-281).
cv_folds_batched <- function(Z, instPeriod, mu, y, u, v, num.restarts, niter, tol, n.devices = 0L,
                             use.raw = FALSE) {
  single <- is.matrix(u)
  if (single) { u <- list(u); v <- list(v) }
  series <- lapply(seq_along(u), function(i) list(y = y, u = u[[i]], v = v[[i]]))
  jobs <- list()
  for (z in Z) for (i in seq_along(u))   # fold-major, member-minor: the reference's nested foreach order
    jobs[[length(jobs) + 1L]] <- list(series = i, held = instPeriod[z],
                                      init = make_init(nrow(u[[i]]), nrow(v[[i]]), num.restarts))
  res <- .em_batch(series, jobs, niter, tol, n.devices)
  if (any(res$status == 1L)) stop('inv(): matrix is singular')
  .fold_outputs(res, series, jobs, seq_along(jobs), length(u), instPeriod, mu, use.raw)
}

# Ycv of one station from a batch result: `gs` are its groups (fold-major, member-minor, nm members).
.fold_outputs <- function(res, series, jobs, gs, nm, instPeriod, mu, use.raw) {
  lapply(seq_len(length(gs) %/% nm), function(k) {
    cols <- sapply(seq_len(nm), function(i) {
      g <- gs[(k - 1L) * nm + i]
      if (is.na(res$best[g])) stop('no restart produced a finite likelihood')
      if (use.raw) {                           # propagate(theta, u, v, y)$Y[instPeriod] + mu   (:281)
        s <- series[[jobs[[g]]$series]]
        yz <- s$y
        yz[jobs[[g]]$held] <- NA
        th <- .theta_list(res$theta[, res$best[g]], nrow(s$u), nrow(s$v))
        c(propagate(th, s$u, s$v, matrix(yz, nrow = 1))$Y[instPeriod]) + mu
      } else c(res$Y[[g]][instPeriod]) + mu    # fit$Y[instPeriod] + mu   (:283)
    })
    rowMeans(matrix(cols, ncol = nm))           # .final = rowMeans         (:379)
  })
}

# Host-side set-up of one station as LDS_reconstruction / cvLDS do it (R/LDS_reconstruction.R:128-183):
# the NULL sentinel, the transform, y centred and NA-padded to the station's horizon.
.station_setup <- function(st, transform) {
  u <- st$u; v <- st$v
  single <- !is.list(u) && !is.list(v)
  if (single) {
    if (is.null(u) && is.null(v)) stop('u and v cannot both be NULL')
    u <- list(u); v <- list(v)
  }
  if (is.null(u)) u <- vector('list', length(v))
  if (is.null(v)) v <- vector('list', length(u))
  for (i in seq_along(u)) {
    if (!is.null(u[[i]]) && !is.null(v[[i]]) && ncol(u[[i]]) != ncol(v[[i]]))
      stop('u and v must have the same number of time steps.')
  }
  N <- ncol(if (is.null(u[[1]])) v[[1]] else u[[1]])
  u <- lapply(u, function(m) if (is.null(m)) matrix(0) else m)
  v <- lapply(v, function(m) if (is.null(m)) matrix(0) else m)
  Qa <- st$Qa
  lambda <- NULL
  obs <- switch(transform,
    log = log(Qa$Qa),
    boxcox = {
      bc <- MASS::boxcox(Qa$Qa ~ 1, plotit = FALSE)
      lambda <- bc$x[which.max(bc$y)]
      if (abs(lambda) < 0.01) lambda <- 0
      if (lambda == 0) log(Qa$Qa) else (Qa$Qa^lambda - 1) / lambda
    },
    none = Qa$Qa,
    stop('Accepted transformations are "log", "boxcox" and "none" only.'))
  end.year <- st$start.year + N - 1
  if (end.year < max(Qa$year)) stop('The last year of u is earlier than the last year of the instrumental period.')
  mu <- mean(obs, na.rm = TRUE)
  y <- c(rep(NA, min(Qa$year) - st$start.year), obs - mu, rep(NA, end.year - max(Qa$year)))
  years <- st$start.year:end.year
  list(Qa = Qa, single = single, u = u, v = v, obs = obs, lambda = lambda, mu = mu, years = years,
       y = t(y), instPeriod = which(years %in% Qa$year))
}

.back_transform <- function(x, transform, lambda) {
  switch(transform, log = exp(x), boxcox = if (lambda == 0) exp(x) else (x * lambda + 1)^(1 / lambda), none = x)
}

#' cvLDS for many stations in one batched call: one .em_batch over all stations' folds x members x restarts
#' and one device call for all their metrics.  stations: list of list(Qa = data.frame(year, Qa), u, v,
#' start.year[, Z]); u / v a matrix, NULL or a list (ensemble) as in cvLDS; stations may differ in T, p, q,
#' instrumental period and start year.  Random numbers: station by station, make_Z (if Z is NULL) then make_init
#' fold-major / member-minor -- what the single-station calls draw one after another, so set.seed() gives the
#' same folds and restarts.  Returns one cvLDS-shaped list per station (mirrors api.cvLDS_stations).
cvLDS_stations <- function(stations, transform = 'log', num.restarts = 50, metric.space = 'original',
                           use.raw = FALSE, niter = 1000, tol = 1e-5, use.robust.mean = TRUE, n.devices = 0L) {
  prep <- lapply(stations, .station_setup, transform = transform)
  series <- list(); jobs <- list(); groups <- list()
  for (j in seq_along(prep)) {
    P <- prep[[j]]
    Z <- if (is.null(stations[[j]]$Z)) make_Z(P$Qa$Qa) else stations[[j]]$Z
    if (!is.list(Z)) stop('Please provide the cross-validation folds (Z) in a list.')
    prep[[j]]$Z <- Z
    s0 <- length(series)
    for (i in seq_along(P$u)) series[[s0 + i]] <- list(y = P$y, u = P$u[[i]], v = P$v[[i]])
    g0 <- length(jobs)
    for (z in Z) for (i in seq_along(P$u))
      jobs[[length(jobs) + 1L]] <- list(series = s0 + i, held = P$instPeriod[z],
                                        init = make_init(nrow(P$u[[i]]), nrow(P$v[[i]]), num.restarts))
    groups[[j]] <- (g0 + 1L):length(jobs)
  }
  res <- .em_batch(series, jobs, niter, tol, n.devices)
  if (any(res$status == 1L)) stop('inv(): matrix is singular')
  Ycv <- lapply(seq_along(prep), function(j) {
    P <- prep[[j]]
    y <- .fold_outputs(res, series, jobs, groups[[j]], length(P$u), P$instPeriod, P$mu, use.raw)
    if (metric.space == 'original') lapply(y, .back_transform, transform = transform, lambda = P$lambda) else y
  })
  targets <- lapply(prep, function(P) if (metric.space == 'original') P$Qa$Qa else P$obs)
  dist <- .Call('_ldsr_cv_metrics_stations', lapply(Ycv, function(y) do.call(cbind, y)), lapply(targets, as.numeric),
                lapply(prep, function(P) lapply(P$Z, as.integer)), FALSE, PACKAGE = 'ldsr')
  mean.func <- if (use.robust.mean) dplR::tbrm else mean
  lapply(seq_along(prep), function(j) {
    md <- data.table::as.data.table(t(dist[[j]]))
    data.table::setnames(md, c('R2', 'RE', 'CE', 'nRMSE', 'KGE'))
    list(metrics.dist = md, metrics = sapply(md, mean.func),
         target = data.table::data.table(year = prep[[j]]$Qa$year, y = targets[[j]]),
         Ycv = do.call(cbind, Ycv[[j]]), Z = prep[[j]]$Z)
  })
}

#' LDS_reconstruction for many stations in one batched call: one .em_batch over all stations' members x
#' restarts and one device call for all their reconstructions (construct_rec and the ensemble means).
#' stations: list of list(Qa, u, v, start.year[, init]), as cvLDS_stations.  Random numbers: station by station,
#' make_init per member unless `init` is given.  Returns one LDS_reconstruction-shaped list per station
#' (mirrors api.LDS_reconstruction_stations).
LDS_reconstruction_stations <- function(stations, transform = 'log', num.restarts = 50, return.init = FALSE,
                                        niter = 1000, tol = 1e-5, n.devices = 0L) {
  prep <- lapply(stations, .station_setup, transform = transform)
  series <- list(); jobs <- list()
  for (j in seq_along(prep)) {
    P <- prep[[j]]
    init <- stations[[j]]$init
    if (is.null(init)) init <- lapply(seq_along(P$u), function(i) make_init(nrow(P$u[[i]]), nrow(P$v[[i]]), num.restarts))
    else if (P$single) init <- list(init)
    for (i in seq_along(P$u)) {
      series[[length(series) + 1L]] <- list(y = P$y, u = P$u[[i]], v = P$v[[i]])
      jobs[[length(jobs) + 1L]] <- list(series = length(series), held = integer(0), init = init[[i]])
    }
  }
  res <- .em_batch(series, jobs, niter, tol, n.devices)
  if (any(res$status == 1L)) stop('inv(): matrix is singular')
  picks <- lapply(seq_along(jobs), function(g) .pick(res, g, series, jobs))
  first <- cumsum(c(0L, sapply(prep, function(P) length(P$u))))
  mine <- lapply(seq_along(prep), function(j) picks[(first[j] + 1L):first[j + 1L]])
  col <- function(key) lapply(mine, function(m) sapply(m, function(a) c(a$fit[[key]])))
  th <- function(key) lapply(mine, function(m) sapply(m, function(a) c(a$theta[[key]])))
  tr <- match(transform, c('none', 'log', 'boxcox')) - 1L
  rec <- .Call('_ldsr_construct_rec_stations', lapply(col('X'), as.matrix), lapply(col('V'), as.matrix),
               lapply(col('Y'), as.matrix), th('C'), th('R'), sapply(prep, `[[`, 'mu'),
               as.integer(tr), sapply(prep, function(P) if (is.null(P$lambda)) 0 else P$lambda), PACKAGE = 'ldsr')
  lapply(seq_along(prep), function(j) {
    P <- prep[[j]]; n <- length(P$u)
    a <- array(rec[[j]]$rec, dim = c(length(P$years), 6L, n))
    members <- lapply(seq_len(n), function(i) {
      dt <- data.table::as.data.table(a[, , i]); data.table::setnames(dt, c('X', 'Xl', 'Xu', 'Q', 'Ql', 'Qu'))
      out <- list(rec = cbind(data.table::data.table(year = P$years), dt), theta = mine[[j]][[i]]$theta,
                  lik = mine[[j]][[i]]$lik)
      if (return.init) out$init <- mine[[j]][[i]]$init
      if (transform == 'boxcox') out$lambda <- P$lambda
      out
    })
    if (P$single) members[[1]]
    else list(rec = data.table::data.table(year = P$years, X = rec[[j]]$mean[, 1], Q = rec[[j]]$mean[, 2]),
              ensemble = members)
  })
}

# The ensemble loop of LDS_reconstruction (R/LDS_reconstruction.R:236-246) as one batch: returns
# what `call_method(..., 'EM', ...)` returns for each member.
reconstruct_members_batched <- function(y, u, v, init, niter, tol, return.init, n.devices = 0L) {
  single <- is.matrix(u)
  if (single) { u <- list(u); v <- list(v); init <- list(init) }
  series <- lapply(seq_along(u), function(i) list(y = y, u = u[[i]], v = v[[i]]))
  jobs <- lapply(seq_along(u), function(i) list(series = i, held = integer(0), init = init[[i]]))
  res <- .em_batch(series, jobs, niter, tol, n.devices)
  if (any(res$status == 1L)) stop('inv(): matrix is singular')
  out <- lapply(seq_along(u), function(i) {
    a <- .pick(res, i, series, jobs)
    if (!return.init) a$init <- NULL
    a
  })
  if (single) out[[1]] else out
}

# R/stochastics.R:58-63.  exact.rng = TRUE (default): the noise comes from R's own RNG in exactly the
# order one_LDS_rep draws it -- per replicate rnorm(1) for x1, rnorm(n) for the state, rnorm(n) for the
# observations (R/stochastics.R:23-26); one rnorm() call of the total length yields the same stream as
# those calls in sequence, and rnorm(k, 0, s) is s * N(0,1) -- so set.seed() reproduces the
# reference's replicates.  r.seed = s: the same replicates as `set.seed(s); LDS_rep(...)` with R's
# default generators, but the stream (Mersenne-Twister + inversion) is generated on the device: no
# 1.3 GB of host noise for 100 000 replicates and no time in rnorm; R's own RNG state is left alone.
# exact.rng = FALSE uses the counter-based device generator keyed by `seed` (statistically, not
# bitwise, equal).
LDS_rep <- function(theta, u = NULL, v = NULL, years, num.reps = 100, mu = 0, exp.trans = TRUE,
                    exact.rng = TRUE, seed = 0, r.seed = NULL) {
  n <- length(years)
  z <- if (exact.rng && is.null(r.seed)) stats::rnorm(num.reps * (1 + 2 * n)) else NULL
  m <- .Call('_ldsr_rep_batch', theta, u, v, as.integer(n), as.integer(num.reps), as.numeric(seed),
             as.numeric(mu), as.logical(exp.trans), z, if (is.null(r.seed)) NULL else as.integer(r.seed),
             PACKAGE = 'ldsr')
  data.table::data.table(year = rep(years, num.reps), simX = m[, 1], simY = m[, 2], simQ = m[, 3],
                         rep = rep(seq_len(num.reps), each = n))
}


# Replicates conditioned on the observed record (beyond ldsr): whole trajectories drawn from the smoothing
# distribution p(x | y, theta) of the model LDS_reconstruction fitted, by forward filtering, backward sampling.
# They pass through the observed flows and their year-wise spread is the reconstruction's band.  theta: the
# fitted model, or a list of them for an ensemble (u / v lists).  y, mu and lambda are prepared as
# LDS_reconstruction prepares them (.station_setup); u = NULL drops B u and v = NULL drops D v (Kalman_smoother's
# convention, unlike LDS_rep).  exact.rng = TRUE: the noise is rnorm() in the documented order -- member by member,
# replicate by replicate, N state draws then N observation draws -- so set.seed() reproduces the replicates;
# exact.rng = FALSE uses the device's counter-based generator keyed by (seed, member, replicate).  Returns
# LDS_rep's data.table (year, simX, simY, simQ, rep), a list of them for an ensemble; simY is centred and
# transformed, simQ its back-transform.
LDS_rep_posterior <- function(theta, Qa, u, v, start.year, transform = 'log', num.reps = 100, exact.rng = TRUE,
                              seed = 0) {
  P <- .station_setup(list(Qa = Qa, u = u, v = v, start.year = start.year), transform)
  thetas <- if (P$single) list(theta) else theta
  if (length(thetas) != length(P$u)) stop('theta must be one model per ensemble member')
  series <- lapply(seq_along(P$u), function(k) list(y = P$y, u = P$u[[k]], v = P$v[[k]]))
  cols <- lapply(thetas, function(th) c(th$A, th$B, th$C, th$D, th$Q, th$R, th$mu1, th$V1))
  stride <- max(lengths(cols))
  th <- sapply(cols, function(x) c(x, rep(0, stride - length(x))))
  n <- length(P$years); nm <- length(series)
  z <- if (exact.rng) stats::rnorm(2 * num.reps * n * nm) else NULL
  code <- switch(transform, none = 0L, log = 1L, boxcox = 2L)
  m <- .Call('_ldsr_posterior_rep_batch', series, matrix(th, nrow = stride), as.integer(num.reps), z,
             as.numeric(seed), rep(P$mu, nm), code, if (transform == 'boxcox') rep(P$lambda, nm) else NULL,
             PACKAGE = 'ldsr')
  out <- lapply(seq_len(nm), function(k) {
    r <- (k - 1) * num.reps * n + seq_len(num.reps * n)
    data.table::data.table(year = rep(P$years, num.reps), simX = m[r, 1], simY = m[r, 2], simQ = m[r, 3],
                           rep = rep(seq_len(num.reps), each = n))
  })
  if (P$single) out[[1]] else out
}

# Drought statistics of LDS_rep_posterior's replicates (the same arguments and exact.rng / seed give the same draws),
# computed on the device in the sampler's walk: no trajectory is written, so 10^6 replicates and more fit.  windows:
# up to 4 moving-mean lengths of 1..64 years (lowest and highest mean and its first year, the earliest on a tie);
# threshold: flow below which a year is in drought (NULL: mean of the observed Qa); runs are maximal stretches below
# it (longest run and its first year, largest deficit sum(threshold - Q) and its first year, number of runs, the
# earliest on a tie); period = c(first.year, last.year) restricts every statistic (runs clipped), NULL the whole
# horizon.  Undefined values are NA / year NA; a replicate with a non-finite flow in the period has NA throughout.
# Returns a list with windows, threshold, period, data.tables `window` (rep, window, min, min.year, max, max.year)
# and `run` (rep, run.len, run.year, deficit, deficit.year, n.runs); a list of them for an ensemble.
LDS_rep_posterior_stats <- function(theta, Qa, u, v, start.year, transform = 'log', num.reps = 100, exact.rng = TRUE,
                                    seed = 0, windows = 10L, threshold = NULL, period = NULL) {
  P <- .station_setup(list(Qa = Qa, u = u, v = v, start.year = start.year), transform)
  thetas <- if (P$single) list(theta) else theta
  if (length(thetas) != length(P$u)) stop('theta must be one model per ensemble member')
  series <- lapply(seq_along(P$u), function(k) list(y = P$y, u = P$u[[k]], v = P$v[[k]]))
  cols <- lapply(thetas, function(th) c(th$A, th$B, th$C, th$D, th$Q, th$R, th$mu1, th$V1))
  stride <- max(lengths(cols))
  th <- sapply(cols, function(x) c(x, rep(0, stride - length(x))))
  n <- length(P$years); nm <- length(series); y0 <- P$years[1]
  if (is.null(period)) period <- range(P$years)
  rg <- c(period[1] - y0, period[2] - y0 + 1)
  if (rg[1] < 0 || rg[2] > n || rg[1] >= rg[2]) stop('period must lie inside the reconstruction horizon')
  if (is.null(threshold)) threshold <- mean(Qa$Qa)
  z <- if (exact.rng) stats::rnorm(2 * num.reps * n * nm) else NULL
  code <- switch(transform, none = 0L, log = 1L, boxcox = 2L)
  m <- .Call('_ldsr_posterior_stats_batch', series, matrix(th, nrow = stride), as.integer(num.reps), z,
             as.numeric(seed), rep(P$mu, nm), code, if (transform == 'boxcox') rep(P$lambda, nm) else NULL,
             as.integer(windows), rep(as.numeric(threshold), nm), as.integer(rep(rg, nm)), PACKAGE = 'ldsr')
  yr <- function(a) ifelse(a < 0, NA_integer_, a + y0)
  na <- function(a) ifelse(a < 0, NA_integer_, a)
  out <- lapply(seq_len(nm), function(k) {
    r <- (k - 1) * num.reps + seq_len(num.reps)
    win <- data.table::rbindlist(lapply(seq_along(windows), function(j) data.table::data.table(
      rep = seq_len(num.reps), window = windows[j], min = m[[1]][r, j], min.year = yr(m[[2]][r, j]),
      max = m[[3]][r, j], max.year = yr(m[[4]][r, j]))))
    run <- data.table::data.table(rep = seq_len(num.reps), run.len = na(m[[5]][r]), run.year = yr(m[[6]][r]),
                                  deficit = m[[7]][r], deficit.year = yr(m[[8]][r]), n.runs = na(m[[9]][r]))
    list(windows = windows, threshold = threshold, period = period, window = win, run = run)
  })
  if (P$single) out[[1]] else out
}

#' Kalman / RTS smoother for a state of dimension d > 1 (beyond ldsr, whose state is scalar).
#' theta: list(A d x d, B d x p, C 1 x d, D 1 x q, Q d x d, R, mu1 d x 1, V1 d x d); y 1 x T with NA.
#' method: 1 = associative scan over time (long series), 0 = sequential recursion.
#' Returns list(X d x T, Y 1 x T, V (d*d) x T with column t = vec(V_t), lik).
Kalman_smoother_d <- function(y, u, v, theta, stdlik = TRUE, method = 1L) {
  if (is.null(u)) u <- matrix(0)
  if (is.null(v)) v <- matrix(0)
  .Call(`_ldsr_smoother_d`, y, u, v, theta, stdlik, as.integer(method))
}


#' All folds' skill metrics in one device call; replaces
#' `mapply(calculate_metrics, sim = Ycv, z = Z, MoreArgs = list(obs = target))` in cvLDS
#' (R/LDS_reconstruction.R:395).  Ycv: list of per-fold vectors (or an n x n_folds matrix).
cv_metrics_batched <- function(Ycv, Z, target, exp_trans = FALSE) {
  if (is.list(Ycv)) Ycv <- do.call(cbind, Ycv)
  m <- .Call(`_ldsr_cv_metrics`, Ycv, as.numeric(target), lapply(Z, as.integer), exp_trans)
  rownames(m) <- c("R2", "RE", "CE", "nRMSE", "KGE")
  m
}


#' construct_rec for all ensemble members in one device call (R/LDS_reconstruction.R:190-212) and the
#' year-wise ensemble mean of X and Q (:247-248).  fits: list of fit lists (X, V, Y as 1 x T matrices),
#' thetas: the matching theta lists.  Returns list(members = list of data.tables, mean = data.table).
construct_rec_batched <- function(fits, thetas, mu, transform, years, lambda = 0) {
  X <- sapply(fits, function(f) c(f$X)); V <- sapply(fits, function(f) c(f$V)); Y <- sapply(fits, function(f) c(f$Y))
  C <- sapply(thetas, function(t) c(t$C)); R <- sapply(thetas, function(t) c(t$R))
  tr <- match(transform, c("none", "log", "boxcox")) - 1L
  r <- .Call(`_ldsr_construct_rec`, as.matrix(X), as.matrix(V), as.matrix(Y), as.numeric(C), as.numeric(R),
             as.numeric(mu), as.integer(tr), as.numeric(lambda))
  a <- array(r$rec, dim = c(length(years), 6L, length(fits)))
  members <- lapply(seq_along(fits), function(i) {
    dt <- data.table::as.data.table(a[, , i]); data.table::setnames(dt, c("X", "Xl", "Xu", "Q", "Ql", "Qu"))
    cbind(data.table::data.table(year = years), dt)
  })
  list(members = members, mean = data.table::data.table(year = years, X = r$mean[, 1], Q = r$mean[, 2]))
}


#' Objective of the experimental learners for a whole population (R/LDS_GA.R:28-44, 136-147):
#' `thetas` is a (2d+6) x n matrix of candidate vectors; kind is "penalized_likelihood", "negLogLik" or
#' "ssqTrain".  GA::gaisl / optim call the scalar versions once per candidate; with a vectorised fitness
#' (e.g. GA's `parallel` hook or a custom generation loop) one generation is one device call.
objective_batched <- function(y, u, v, thetas, kind = "penalized_likelihood", lambda = 1) {
  k <- match(kind, c("penalized_likelihood", "negLogLik", "ssqTrain")) - 1L
  .Call(`_ldsr_objective`, y, u, v, thetas, as.integer(k), as.numeric(lambda))
}


#' The shim keeps one device context per R session; its device and pinned buffers are cached between
#' calls.  This hands the cached device memory back to the driver (bytes released, invisibly); the next
#' call simply allocates again.  Unloading the package (R_unload_ldsr) releases everything.
ldsr_gpu_trim <- function() invisible(.Call(`_ldsr_trim`))
