# Final models of several responses of one design (the step after CrossValidateMulti): one `.Call` fits every column of
# Targets at its own (lambda, alpha) in one launch, and each response's compact record is turned into the list
# EBelasticNet.Gaussian / EBelasticNet.Binomial return for that response alone (the post-processing of
# EBEN_orig/R/EBelasticNet.Gaussian.R:56-98 and its binomial counterpart, as pareben_b200/cross_validate.py restates it):
# the same rows, in the same order, of the weight table built from the `.C` Beta matrix.
#   Gaussian main, binomial main: effects with beta != 0, in candidate order
#   Gaussian Epis: every used candidate, in candidate order      binomial Epis: Used order, beta != 0
#   Epis: main effects first, then pairs, each stably ordered by the first locus
# lambda, alpha: length ncol(Targets), or one value for every response.

.candidate_loci <- function(cand, k){            # 1-based candidate id -> 1-based loci (main effects, then pairs i < j)
  c0 <- cand - 1
  loci <- cbind(c0 + 1, c0 + 1)
  pc <- c0[c0 >= k] - k
  if (length(pc)) {
    i <- floor(((2 * k - 1) - sqrt((2 * k - 1)^2 - 8 * pc)) / 2)
    i <- ifelse(i * (2 * k - i - 1) / 2 > pc, i - 1, i)
    i <- ifelse((i + 1) * (2 * k - i - 2) / 2 <= pc, i + 1, i)
    j <- pc - i * (2 * k - i - 1) / 2 + i + 1
    loci[c0 >= k, ] <- cbind(i + 1, j + 1)
  }
  loci
}

.record_weight <- function(m, cand, beta, var, epis, gaussian, k, n){
  idx <- seq_len(m)
  cand <- cand[idx]; beta <- beta[idx]; var <- var[idx]
  if (gaussian || !epis) { o <- order(cand); cand <- cand[o]; beta <- beta[o]; var <- var[o] }
  keep <- if (gaussian && epis) idx else which(beta != 0)
  blup <- cbind(.candidate_loci(cand, k), beta, var)[keep, , drop = FALSE]
  if (nrow(blup) == 0) blup <- matrix(0, 1, 4)
  if (epis) {
    main <- blup[blup[, 1] == blup[, 2], , drop = FALSE]
    pair <- blup[blup[, 1] != blup[, 2], , drop = FALSE]
    blup <- rbind(main[order(main[, 1]), , drop = FALSE], pair[order(pair[, 1]), , drop = FALSE])
  }
  t <- abs(blup[, 3]) / (sqrt(blup[, 4]) + 1e-20)
  pv <- 2 * (1 - pt(t, df = n - 1))
  unname(cbind(blup, t, pv))
}

EBelasticNetMulti.gpu <- function(BASIS, Targets, lambda, alpha, Epis = "no", prior = "gaussian"){
  storage.mode(BASIS) <- "double"
  Targets <- as.matrix(Targets); storage.mode(Targets) <- "double"
  nT <- ncol(Targets)
  lambda <- rep_len(as.double(lambda), nT); alpha <- rep_len(as.double(alpha), nT)
  gaussian <- prior == "gaussian"; epis <- Epis == "yes"
  r <- .Call("pareben_fit_batch_call", BASIS, Targets, lambda, alpha, as.integer(epis), as.integer(!gaussian), 0L,
             PACKAGE = "parEBEN")
  lapply(seq_len(nT), function(t){
    w <- .record_weight(r$n_effects[t], r$cand[, t], r$beta[, t], r$var[, t], epis, gaussian, ncol(BASIS), nrow(BASIS))
    s <- r$scalars[, t]
    if (gaussian) list(weight = w, WaldScore = s[1], Intercept = s[2], residVar = s[4])
    else list(weight = w, logLikelihood = s[4], WaldScore = s[1], Intercept = s[2:3])
  })
}
