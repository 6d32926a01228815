## fit_ffm.nim -- the field-aware twins.  `include` SGD's at the end of optimizer/sgd_ffm.nim in place of
## `proc fit*[L](self: SGD[L], X: RowFieldDataset, ...)` (sgd_ffm.nim:49-106) and AdaGrad's at the end of
## optimizer/adagrad_ffm.nim in place of adagrad_ffm.nim:11-66; the `maxThreads` overloads replace
## sgd_ffm_multi.nim:31-103 and adagrad_ffm_multi.nim:36-104 (synchronous minibatch of maxThreads samples).

proc fit*[L](self: SGD[L], X: RowFieldDataset, y: seq[float64],
             ffm: FieldAwareFactorizationMachine,
             callback: (SGD[L], FieldAwareFactorizationMachine)->void = nil) =
  ## Fits the factorization machine on X and y by stochastic gradient descent.
  ffm.init(X)
  var y = ffm.checkTarget(y)
  let nSamples = X.nSamples
  var
    indices = toSeq(0..<nSamples)
    isConverged = false
  if self.nCalls > 0 and not callback.isNil:
    raise newException(ValueError, "nCalls > 0 is not supported on the device path: one call runs a whole epoch.")
  if not ffm.warmstart:
    self.init()
  let ds = device(X)
  setTargets(ds, y)
  let h = toDevice(ffm, X.nFeatures, X.nFields)
  var cfg = SgdCfg(loss: lossKind(self.loss), huberThreshold: lossThreshold(self.loss), eta0: self.eta0,
                   alpha0: self.alpha0, alpha: self.alpha, beta: self.beta,
                   scheduling: schedCode(self.scheduling), power: self.power)
  try:
    check nimfm_ffm_sgd_begin(ctx(), h)
    for epoch in 0..<self.maxIter:
      var viol, lossSum: cdouble
      if X.nCached == X.nSamples and self.shuffle: shuffle(indices)
      var itc = int64(self.it)
      check nimfm_ffm_sgd_epoch(ctx(), h, ds, addr cfg, addr itc, cast[ptr int64](p(indices)), nSamples,
                                addr viol, addr lossSum)
      self.it = int(itc)
      let runningLoss = lossSum / float(nSamples)
      if not callback.isNil:
        check nimfm_ffm_sgd_end(ctx(), h)         # finalize (sgd_ffm.nim:88-92)
        fromDevice(ffm, h)
        callback(self, ffm)
      elif self.verbose > 0:
        fromDevice(ffm, h)
      let isContinue = stoppingCriterion(
        ffm.P, ffm.w, ffm.intercept, self.alpha0, self.alpha, self.beta, runningLoss,
        viol, self.tol, self.verbose, epoch, self.maxIter, isConverged)
      if not isContinue: break
    if not isConverged and self.verbose > 0:
      echo("Objective did not converge. Increase maxIter.")
    check nimfm_ffm_sgd_end(ctx(), h)
    fromDevice(ffm, h)
  finally:
    discard nimfm_ffm_free(ctx(), h)

proc runAdaGradFFM[L](self: AdaGrad[L], X: RowFieldDataset, y: seq[float64], ffm: FieldAwareFactorizationMachine,
                      miniBatch: int, callback: (AdaGrad[L], FieldAwareFactorizationMachine)->void) =
  ffm.init(X)
  var y = ffm.checkTarget(y)
  let nSamples = X.nSamples
  var
    indices = toSeq(0..<nSamples)
    isConverged = false
  if self.nCalls > 0 and not callback.isNil:
    raise newException(ValueError, "nCalls > 0 is not supported on the device path: one call runs a whole epoch.")
  let ds = device(X)
  setTargets(ds, y)
  let h = toDevice(ffm, X.nFeatures, X.nFields)
  var cfg = AdagradCfg(loss: lossKind(self.loss), huberThreshold: lossThreshold(self.loss), eta0: self.eta0,
                       alpha0: self.alpha0, alpha: self.alpha, beta: self.beta, eps: self.eps,
                       miniBatchSize: miniBatch)
  try:
    # init (adagrad.nim:47-62): g_sum <- 0, g_norm <- eps unless warm-started with a state of the right shape
    if not ffm.warmStart: self.it = 1
    check nimfm_ffm_adagrad_init(ctx(), h, self.eps, 1)
    if self.it != 1:
      var
        gsP = flat(self.g_sum.P)
        gnP = flat(self.g_norm.P)
      check nimfm_ffm_adagrad_set_state(ctx(), h, cast[ptr cdouble](p(gsP)), cast[ptr cdouble](p(gnP)),
                                        cast[ptr cdouble](p(self.g_sum.w)), cast[ptr cdouble](p(self.g_norm.w)),
                                        self.g_sum.intercept, self.g_norm.intercept)
    for epoch in 0..<self.maxIter:
      var viol, lossSum: cdouble
      if X.nCached == X.nSamples and self.shuffle: shuffle(indices)
      var itc = int64(self.it)
      check nimfm_ffm_adagrad_epoch(ctx(), h, ds, addr cfg, addr itc, cast[ptr int64](p(indices)), nSamples,
                                    addr viol, addr lossSum)
      self.it = int(itc)
      let runningLoss = lossSum / float(nSamples)
      if not callback.isNil:
        check nimfm_ffm_adagrad_finalize(ctx(), h, addr cfg, self.it)
        fromDevice(ffm, h)
        callback(self, ffm)
      elif self.verbose > 0:
        fromDevice(ffm, h)
      let isContinue = stoppingCriterion(
        ffm.P, ffm.w, ffm.intercept, self.alpha0, self.alpha, self.beta, runningLoss,
        viol, self.tol, self.verbose, epoch, self.maxIter, isConverged)
      if not isContinue: break
    if not isConverged and self.verbose > 0:
      echo("Objective did not converge. Increase maxIter.")
    # keep g_sum / g_norm for warm starts (adagrad.nim:15-16), shaped like ffm.P, then finalize (adagrad.nim:65-84)
    block:
      var
        gsP = newSeq[float64](ffm.P.shape[0] * ffm.P.shape[1] * ffm.P.shape[2])
        gnP = newSeq[float64](gsP.len)
        gsb, gnb: cdouble
      if self.g_sum.isNil:
        self.g_sum = newParams([ffm.P.shape[0], ffm.P.shape[1], ffm.P.shape[2]], ffm.w.len, ffm.fitLinear,
                               ffm.fitIntercept)
        self.g_norm = newParams([ffm.P.shape[0], ffm.P.shape[1], ffm.P.shape[2]], ffm.w.len, ffm.fitLinear,
                                ffm.fitIntercept)
      check nimfm_ffm_adagrad_get_state(ctx(), h, cast[ptr cdouble](p(gsP)), cast[ptr cdouble](p(gnP)),
                                        cast[ptr cdouble](p(self.g_sum.w)), cast[ptr cdouble](p(self.g_norm.w)),
                                        addr gsb, addr gnb)
      unflat(self.g_sum.P, gsP)
      unflat(self.g_norm.P, gnP)
      self.g_sum.intercept = gsb
      self.g_norm.intercept = gnb
    check nimfm_ffm_adagrad_finalize(ctx(), h, addr cfg, self.it)
    fromDevice(ffm, h)
  finally:
    discard nimfm_ffm_free(ctx(), h)

proc fit*[L](self: AdaGrad[L], X: RowFieldDataset, y: seq[float64],
             ffm: FieldAwareFactorizationMachine,
             callback: (AdaGrad[L], FieldAwareFactorizationMachine)->void = nil) =
  ## Fits the factorization machine on X and y by stochastic gradient descent.
  runAdaGradFFM(self, X, y, ffm, 1, callback)

proc fit*[L](self: AdaGrad[L], X: RowFieldDataset, y: seq[float64],
             ffm: FieldAwareFactorizationMachine, maxThreads: int,
             callback: (AdaGrad[L], FieldAwareFactorizationMachine)->void = nil) =
  ## Fits the factorization machine on X and y by stochastic gradient descent.
  runAdaGradFFM(self, X, y, ffm, (if maxThreads < 0: 4096 else: max(1, maxThreads)), callback)

proc fit*[L](self: SGD[L], X: RowFieldDataset, y: seq[float64],
             ffm: FieldAwareFactorizationMachine, maxThreads: int,
             callback: (SGD[L], FieldAwareFactorizationMachine)->void = nil) =
  ## Fits the factorization machine on X and y by stochastic gradient descent.
  ffm.init(X)
  var y = ffm.checkTarget(y)
  let
    nSamples = X.nSamples
    miniBatch = (if maxThreads < 0: 4096 else: max(1, maxThreads))
  var
    indices = toSeq(0..<nSamples)
    isConverged = false
  if not ffm.warmstart:
    self.init()
  let ds = device(X)
  setTargets(ds, y)
  let h = toDevice(ffm, X.nFeatures, X.nFields)
  var cfg = SgdCfg(loss: lossKind(self.loss), huberThreshold: lossThreshold(self.loss), eta0: self.eta0,
                   alpha0: self.alpha0, alpha: self.alpha, beta: self.beta,
                   scheduling: schedCode(self.scheduling), power: self.power)
  try:
    for epoch in 0..<self.maxIter:
      var viol, lossSum: cdouble
      if X.nCached == X.nSamples and self.shuffle: shuffle(indices)
      var itc = int64(self.it)
      check nimfm_ffm_sgd_minibatch_epoch(ctx(), h, ds, addr cfg, miniBatch, miniBatch, addr itc,
                                          cast[ptr int64](p(indices)), nSamples, addr viol, addr lossSum)
      self.it = int(itc)
      let runningLoss = lossSum / float(nSamples)
      if not callback.isNil or self.verbose > 0: fromDevice(ffm, h)
      if not callback.isNil: callback(self, ffm)
      let isContinue = stoppingCriterion(
        ffm.P, ffm.w, ffm.intercept, self.alpha0, self.alpha, self.beta, runningLoss,
        viol, self.tol, self.verbose, epoch, self.maxIter, isConverged)
      if not isContinue: break
    if not isConverged and self.verbose > 0:
      echo("Objective did not converge. Increase maxIter.")
    fromDevice(ffm, h)
  finally:
    discard nimfm_ffm_free(ctx(), h)
