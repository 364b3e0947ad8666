# scde_b200.R -- R side of the drop-in.  With integration/scde_b200_shim.cpp in src/ (instead of jpmatLogBoot.cpp and
# matSlideMult.cpp) scde.posteriors / scde.expression.difference / scde.test.gene.expression.difference work UNCHANGED:
# their .Call sites resolve to the shim.  Two things to know:
#   * call them with n.cores = 1: papply forks (R/functions.R:6054), and a CUDA context does not survive fork(); the
#     shim's .Call entries draw as one call does, so results equal scde's at n.cores = 1;
#   * for large inputs use the fused entry below: the joint posteriors (genes x 401 doubles per group) then never cross
#     PCIe, `n.cores` reproduces scde's results at that n.cores (one draw set per gene chunk, computed in the same device
#     launches, nothing forks), and `n.devices` GPUs share the genes without changing results.
scde.expression.difference.b200 <- function(models, counts, prior, groups = NULL, batch = NULL, n.randomizations = 150,
                                            n.devices = 1, batch.models = models, expectation = 0, devices = seq_len(n.devices) - 1L,
                                            n.cores = 1) {
  if(!all(rownames(models) %in% colnames(counts))) stop("ERROR: provided count data does not cover all of the cells specified in the model matrix")
  counts <- as.matrix(counts[, match(rownames(models), colnames(counts))]); storage.mode(counts) <- "integer"
  if(is.null(groups)) { groups <- as.factor(attr(models, "groups")); names(groups) <- rownames(models) }
  if(length(levels(groups)) != 2) stop(paste("ERROR: wrong number of levels in the grouping factor (", paste(levels(groups), collapse = " "), "), but must be two.", sep = ""))
  mn <- c("conc.b", "conc.a", "fail.r", "corr.b", "corr.a", "corr.theta", "corr.ltheta.b", "corr.ltheta.t", "corr.ltheta.m",
          "corr.ltheta.s", "corr.ltheta.r", "conc.a2")
  pack <- function(m) {                                     # R/functions.R:579-583, 601-604
    mm <- matrix(NA_real_, nrow(m), 12); mc <- match(mn, colnames(m))
    mm[, !is.na(mc)] <- as.matrix(m[, mc[!is.na(mc)]]); mm[mm[, 5] < 1e-10, 5] <- 1e-10; mm
  }
  correct.batch <- !is.null(batch) && length(levels(as.factor(batch))) > 1
  if(correct.batch) {
    batch <- as.factor(batch)
    bgti.ft <- fisher.test(table(groups, batch))            # R/functions.R:336-349
    if(bgti.ft$p.value < 1e-3) { cat("WARNING: strong interaction between groups and batches! Correction may be ineffective:\n"); print(bgti.ft) }
  }
  x <- prior$x; K <- length(x)
  rv <- as.numeric(as.character(seq(x[1] - x[K], x[K] - x[1], length = 2 * K - 1)))              # R/functions.R:3506-3507
  arv <- as.numeric(as.character(seq(rv[1] - rv[2 * K - 1], rv[2 * K - 1] - rv[1], length = 4 * K - 3)))
  zidx <- function(g) sapply(expectation / log2(10), function(e) which.min(abs(g - e)))         # :3519,3524
  r <- .Call("scde_b200_diff", counts, pack(models), if(correct.batch) pack(batch.models) else matrix(0, 0, 0), x, prior$y,
             as.integer(groups) - 1L, if(correct.batch) as.integer(batch) - 1L else integer(0),
             if(correct.batch) length(levels(batch)) else 0L, as.integer(n.randomizations), 1L, as.integer(zidx(rv)),
             as.integer(zidx(arv)), as.integer("corr.ltheta.b" %in% colnames(models)), as.integer("conc.a2" %in% colnames(models)),
             as.integer(devices), as.integer(n.cores), PACKAGE = "scde")
  if(correct.batch) names(r) <- c("idx", "z", "cz", "batch.idx", "batch.z", "batch.cz", "adjusted.idx", "adjusted.z", "adjusted.cz")
  frame <- function(idx, z, cz, grid) {                      # quick.distribution.summary, R/functions.R:5045-5052
    dq <- cbind(lb = grid[idx[, 1] + 1], mle = grid[idx[, 2] + 1], ub = grid[idx[, 3] + 1]) / log10(2)
    cq <- rep(0, nrow(dq)); cq[dq[, 1] > 0] <- dq[dq[, 1] > 0, 1]; cq[dq[, 3] < 0] <- dq[dq[, 3] < 0, 3]
    # cZ comes from the library (BH over all genes of the call); in R: sign(z) * qnorm(p.adjust(pnorm(abs(z), lower.tail = F), "BH"), lower.tail = F)
    data.frame(dq, ce = cq, Z = as.numeric(z), cZ = as.numeric(cz), row.names = rownames(counts))
  }
  if(correct.batch)
    return(list(batch.adjusted = frame(r$adjusted.idx, r$adjusted.z, r$adjusted.cz, arv), results = frame(r$idx, r$z, r$cz, rv),
                batch.effect = frame(r$batch.idx, r$batch.z, r$batch.cz, rv)))
  frame(r$idx, r$z, r$cz, rv)
}

# Every contrast of a many-level grouping in one device session: the count matrix, its index and table are built once
# and each group's joint posterior is computed once, however many contrasts name it.  `contrasts`: NULL (all pairs of
# levels, a before b in level order), "rest" (each level against the union of the others), or a list of pairs
# list(A, B), each side a level name or a vector of level names (their union).  Returns a named list ("A vs B") of what
# scde.expression.difference.b200 returns for the two-level factor (A first; cells of neither side NA).
scde.expression.difference.contrasts.b200 <- function(models, counts, prior, groups, contrasts = NULL, batch = NULL,
                                                      n.randomizations = 150, n.devices = 1, batch.models = models,
                                                      expectation = 0, devices = seq_len(n.devices) - 1L, n.cores = 1) {
  if(!all(rownames(models) %in% colnames(counts))) stop("ERROR: provided count data does not cover all of the cells specified in the model matrix")
  counts <- as.matrix(counts[, match(rownames(models), colnames(counts))]); storage.mode(counts) <- "integer"
  groups <- as.factor(groups); lev <- levels(groups)
  if(length(lev) < 2) stop("ERROR: the grouping factor needs at least two levels to compare")
  rest <- identical(contrasts, "rest")
  if(is.null(contrasts)) {
    contrasts <- list(); for(i in seq_along(lev)) for(j in seq_along(lev)) if(i < j) contrasts[[length(contrasts) + 1]] <- list(lev[i], lev[j])
  } else if(rest) {
    contrasts <- lapply(lev, function(l) list(l, setdiff(lev, l)))
  }
  labels <- character(0); sides <- list(); pairs <- integer(0)
  for(cc in contrasts) {
    if(length(cc) != 2) stop("ERROR: each contrast must be a pair (A, B) of level names or vectors of level names")
    for(s in cc) if(!all(s %in% lev)) stop(paste("ERROR: unknown level", paste(setdiff(s, lev), collapse = " "), "in a contrast"))
    if(length(intersect(cc[[1]], cc[[2]]))) stop("ERROR: the two sides of a contrast share a level")
    a <- paste(cc[[1]], collapse = "+"); b <- if(rest) "rest" else paste(cc[[2]], collapse = "+")
    labels <- c(labels, paste(a, "vs", b))
    for(s in list(cc[[1]], cc[[2]])) {
      key <- paste(sort(match(s, lev)), collapse = ",")
      if(is.null(sides[[key]])) {
        cells <- which(groups %in% s) - 1L
        if(!length(cells)) stop(paste("ERROR: no cells in", paste(s, collapse = "+")))
        sides[[key]] <- list(id = length(sides), cells = cells)
      }
      pairs <- c(pairs, sides[[key]]$id)
    }
  }
  goff <- c(0L, cumsum(sapply(sides, function(s) length(s$cells))))
  gcells <- unlist(lapply(sides, function(s) s$cells))
  mn <- c("conc.b", "conc.a", "fail.r", "corr.b", "corr.a", "corr.theta", "corr.ltheta.b", "corr.ltheta.t", "corr.ltheta.m",
          "corr.ltheta.s", "corr.ltheta.r", "conc.a2")
  pack <- function(m) {                                     # R/functions.R:579-583, 601-604
    mm <- matrix(NA_real_, nrow(m), 12); mc <- match(mn, colnames(m))
    mm[, !is.na(mc)] <- as.matrix(m[, mc[!is.na(mc)]]); mm[mm[, 5] < 1e-10, 5] <- 1e-10; mm
  }
  correct.batch <- !is.null(batch) && length(levels(as.factor(batch))) > 1
  if(correct.batch) batch <- as.factor(batch)
  x <- prior$x; K <- length(x)
  rv <- as.numeric(as.character(seq(x[1] - x[K], x[K] - x[1], length = 2 * K - 1)))              # R/functions.R:3506-3507
  arv <- as.numeric(as.character(seq(rv[1] - rv[2 * K - 1], rv[2 * K - 1] - rv[1], length = 4 * K - 3)))
  zidx <- function(g) sapply(expectation / log2(10), function(e) which.min(abs(g - e)))         # :3519,3524
  r <- .Call("scde_b200_diff_contrasts", counts, pack(models), if(correct.batch) pack(batch.models) else matrix(0, 0, 0), x,
             prior$y, as.integer(goff), as.integer(gcells), as.integer(pairs),
             if(correct.batch) as.integer(batch) - 1L else integer(0), if(correct.batch) length(levels(batch)) else 0L,
             as.integer(n.randomizations), 1L, as.integer(zidx(rv)), as.integer(zidx(arv)),
             as.integer("corr.ltheta.b" %in% colnames(models)), as.integer("conc.a2" %in% colnames(models)),
             as.integer("corr.ltheta.b" %in% colnames(batch.models)), as.integer("conc.a2" %in% colnames(batch.models)),
             as.integer(devices), as.integer(n.cores), PACKAGE = "scde")
  frame <- function(idx, z, cz, grid) {                      # quick.distribution.summary, R/functions.R:5045-5052
    dq <- cbind(lb = grid[idx[, 1] + 1], mle = grid[idx[, 2] + 1], ub = grid[idx[, 3] + 1]) / log10(2)
    cq <- rep(0, nrow(dq)); cq[dq[, 1] > 0] <- dq[dq[, 1] > 0, 1]; cq[dq[, 3] < 0] <- dq[dq[, 3] < 0, 3]
    data.frame(dq, ce = cq, Z = as.numeric(z), cZ = as.numeric(cz), row.names = rownames(counts))
  }
  one <- function(s, c, grid) frame(r[[3 * s + 1]][, 3 * c + 1:3, drop = FALSE], r[[3 * s + 2]][, c + 1], r[[3 * s + 3]][, c + 1], grid)
  out <- lapply(seq_along(labels) - 1L, function(c) {
    if(correct.batch) list(batch.adjusted = one(2, c, arv), results = one(0, c, rv), batch.effect = one(1, c, rv)) else one(0, c, rv)
  })
  names(out) <- labels
  out
}
