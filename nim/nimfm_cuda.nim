## nimfm_cuda.nim -- the Nim side of the drop-in boundary: {.importc, dynlib.} declarations of every symbol of
## include/nimfm_cuda.h.  The procs that keep nimfm's own signatures are in the files beside this one.
##
## NOT COMPILED IN THIS REPOSITORY'S CI: the build image has no Nim toolchain (SURVEY.md, probe table).
## The same symbols are exercised through the ctypes mirror (nimfm_b200/_lib.py), whose prototype
## table is checked against the header by tests/test_abi_cpu.py.  See INTEGRATION.md for where each
## proc plugs into nimfm's modules.
##
## Type mapping: Nim int -> int64 (cint64), float64 -> cdouble, bool -> int32, seq[T] -> (ptr T, len)
## via `addr s[0]` (`nil` for empty seqs).

const libName = "libnimfm_cuda.so"

type
  CtxObj {.incompleteStruct.} = object
  DatasetObj {.incompleteStruct.} = object
  FmObj {.incompleteStruct.} = object
  FfmObj {.incompleteStruct.} = object
  Ctx* = ptr CtxObj
  DeviceDataset* = ptr DatasetObj
  DeviceFM* = ptr FmObj
  DeviceFFM* = ptr FfmObj

  MbpsgdCfg* {.bycopy.} = object
    loss*: int32
    huberThreshold*: cdouble
    eta0*, alpha0*, alpha*, beta*, gamma*: cdouble
    reg*: int32
    scheduling*: int32
    power*: cdouble
    miniBatchSize*, maxIterInner*: int64

  AdagradCfg* {.bycopy.} = object
    loss*: int32
    huberThreshold*: cdouble
    eta0*, alpha0*, alpha*, beta*, eps*: cdouble
    miniBatchSize*: int64

  SgdCfg* {.bycopy.} = object
    loss*: int32
    huberThreshold*: cdouble
    eta0*, alpha0*, alpha*, beta*: cdouble
    scheduling*: int32
    power*: cdouble

  CdCfg* {.bycopy.} = object
    loss*: int32
    huberThreshold*: cdouble
    alpha0*, alpha*, beta*: cdouble

type
  PcdCfg* {.bycopy.} = object     # nimfm_pcd_cfg
    loss*: int32
    huberThreshold*: cdouble
    alpha0*, alpha*, beta*, gamma*: cdouble
    reg*: int32                   # 1 = L1, 2 = SquaredL12(transpose=true), 3 = SquaredL12(transpose=false)

type
  PsgdCfg* {.bycopy.} = object    # nimfm_psgd_cfg
    loss*: int32
    huberThreshold*: cdouble
    eta0*, alpha0*, alpha*, beta*, gamma*: cdouble
    reg*: int32
    scheduling*: int32
    power*: cdouble

{.push importc, dynlib: libName, cdecl.}
proc nimfm_ctx_create*(device: int32, outCtx: ptr Ctx): int32
proc nimfm_ctx_destroy*(ctx: Ctx): int32
proc nimfm_last_error*(ctx: Ctx): cstring
proc nimfm_comm_unique_id*(uid: pointer): int32
proc nimfm_comm_init*(ctx: Ctx, rank, nranks: int32, uid: pointer): int32
proc nimfm_csr_upload*(ctx: Ctx, n, d: int64, data: ptr cdouble, indices, indptr, fields: ptr int64,
                      nFields, rowBegin, rowEnd: int64, outDs: ptr DeviceDataset): int32
proc nimfm_csc_upload*(ctx: Ctx, n, d: int64, data: ptr cdouble, indices, indptr: ptr int64,
                      outDs: ptr DeviceDataset): int32
proc nimfm_dataset_transpose*(ctx: Ctx, src: DeviceDataset, outDs: ptr DeviceDataset): int32
proc nimfm_dataset_take_rows*(ctx: Ctx, src: DeviceDataset, rowIdx: ptr int64, nIdx: int64,
                             outDs: ptr DeviceDataset): int32   # X[indicesRow], dataset.nim:319-367
proc nimfm_dataset_slice_rows*(ctx: Ctx, src: DeviceDataset, first, last: int64,
                              outDs: ptr DeviceDataset): int32  # X[a..b], dataset.nim:328-348
proc nimfm_dataset_vstack*(ctx: Ctx, parts: ptr DeviceDataset, nParts: int32,
                          outDs: ptr DeviceDataset): int32      # vstack, dataset.nim:452-483
proc nimfm_dataset_set_targets*(ctx: Ctx, ds: DeviceDataset, y: ptr cdouble): int32
proc nimfm_dataset_free*(ctx: Ctx, ds: DeviceDataset): int32
proc nimfm_load_svmlight*(ctx: Ctx, path: cstring, nFeatures: int64, asCsc: int32,
                         outDs: ptr DeviceDataset): int32        # loadSVMLightFile, dataset.nim:616-693
proc nimfm_load_ffm*(ctx: Ctx, path: cstring, nFeatures, nFields: int64,
                    outDs: ptr DeviceDataset): int32             # loadFFMFile, dataset.nim:768-790
proc nimfm_load_user_item_rating*(ctx: Ctx, path: cstring, asCsc: int32,
                                 outDs: ptr DeviceDataset): int32  # loadUserItemRatingFile, dataset.nim:840-990
proc nimfm_load_stream*(ctx: Ctx, pathX, pathY: cstring, outDs: ptr DeviceDataset): int32   # newStreamCSR/CSCDataset
proc nimfm_dataset_get_targets*(ctx: Ctx, ds: DeviceDataset, y: ptr cdouble): int32
proc nimfm_fm_create*(ctx: Ctx, degree, nComponents, nOrders, nAugments: int32, nFeatures: int64,
                     fitLinear, fitIntercept: int32, outFm: ptr DeviceFM): int32
proc nimfm_fm_set_params*(ctx: Ctx, fm: DeviceFM, P, w: ptr cdouble, intercept: cdouble, lams: ptr cdouble): int32
proc nimfm_fm_get_params*(ctx: Ctx, fm: DeviceFM, P, w: ptr cdouble, intercept: ptr cdouble): int32
proc nimfm_fm_free*(ctx: Ctx, fm: DeviceFM): int32
proc nimfm_fm_decision_function*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, outY: ptr cdouble): int32
proc nimfm_fm_loss_grad*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, loss: int32, huberThreshold: cdouble,
                        rowBegin, nRows: int64, rowIdx: ptr int64, miniBatchSize: int64,
                        zeroGrads, allreduce: int32, lossSum: ptr cdouble): int32
proc nimfm_fm_mbpsgd_epoch*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, cfg: ptr MbpsgdCfg, localBatch: int64,
                           it, ii: ptr int64, sampleIdx: ptr int64, runningLoss: ptr cdouble): int32
proc nimfm_fm_adagrad_init*(ctx: Ctx, fm: DeviceFM, eps: cdouble, reset: int32): int32
proc nimfm_fm_adagrad_epoch*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, cfg: ptr AdagradCfg, it: ptr int64,
                            perm: ptr int64, nRows: int64, viol, lossSum: ptr cdouble): int32
proc nimfm_fm_adagrad_finalize*(ctx: Ctx, fm: DeviceFM, cfg: ptr AdagradCfg, it: int64): int32
proc nimfm_fm_sgd_begin*(ctx: Ctx, fm: DeviceFM): int32
proc nimfm_fm_sgd_epoch*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, cfg: ptr SgdCfg, it: ptr int64,
                        perm: ptr int64, nRows: int64, viol, lossSum: ptr cdouble): int32
proc nimfm_fm_sgd_end*(ctx: Ctx, fm: DeviceFM): int32
proc nimfm_fm_cd_begin*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, cfg: ptr CdCfg): int32
proc nimfm_fm_cd_epoch*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, cfg: ptr CdCfg,
                       viol, lossMean, regOverN: ptr cdouble): int32
proc nimfm_fm_pcd_epoch*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, cfg: ptr PcdCfg,
                        viol, lossMean, regOverN: ptr cdouble): int32   # pcd.nim:156-172
proc nimfm_fm_cd_end*(ctx: Ctx, fm: DeviceFM): int32
proc nimfm_fm_psgd_begin*(ctx: Ctx, fm: DeviceFM): int32                      # psgd.nim:98-112
proc nimfm_fm_psgd_epoch*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, cfg: ptr PsgdCfg, it: ptr int64,
                         perm: ptr int64, nRows: int64, lossSum: ptr cdouble): int32   # psgd.nim:118-176
proc nimfm_fm_psgd_end*(ctx: Ctx, fm: DeviceFM, cfg: ptr PsgdCfg): int32      # finalize, psgd.nim:58-75
proc nimfm_ffm_create*(ctx: Ctx, nComponents: int32, nFields, nFeatures: int64, fitLinear, fitIntercept: int32,
                      outM: ptr DeviceFFM): int32
proc nimfm_ffm_set_params*(ctx: Ctx, m: DeviceFFM, P, w: ptr cdouble, intercept: cdouble): int32
proc nimfm_ffm_get_params*(ctx: Ctx, m: DeviceFFM, P, w: ptr cdouble, intercept: ptr cdouble): int32
proc nimfm_ffm_free*(ctx: Ctx, m: DeviceFFM): int32
proc nimfm_ffm_decision_function*(ctx: Ctx, m: DeviceFFM, X: DeviceDataset, outY: ptr cdouble): int32
proc nimfm_ffm_adagrad_init*(ctx: Ctx, m: DeviceFFM, eps: cdouble, reset: int32): int32
proc nimfm_ffm_adagrad_epoch*(ctx: Ctx, m: DeviceFFM, X: DeviceDataset, cfg: ptr AdagradCfg, it: ptr int64,
                             perm: ptr int64, nRows: int64, viol, lossSum: ptr cdouble): int32
proc nimfm_ffm_adagrad_finalize*(ctx: Ctx, m: DeviceFFM, cfg: ptr AdagradCfg, it: int64): int32
proc nimfm_ffm_adagrad_get_state*(ctx: Ctx, m: DeviceFFM, gsP, gnP, gsw, gnw, gsb, gnb: ptr cdouble): int32
proc nimfm_ffm_adagrad_set_state*(ctx: Ctx, m: DeviceFFM, gsP, gnP, gsw, gnw: ptr cdouble, gsb, gnb: cdouble): int32
proc nimfm_ffm_sgd_begin*(ctx: Ctx, m: DeviceFFM): int32
proc nimfm_fm_sgd_minibatch_epoch*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, cfg: ptr SgdCfg, miniBatchSize, localBatch: int64,
                                  it: ptr int64, perm: ptr int64, nRows: int64, viol, lossSum: ptr cdouble): int32
proc nimfm_ffm_sgd_minibatch_epoch*(ctx: Ctx, m: DeviceFFM, X: DeviceDataset, cfg: ptr SgdCfg, miniBatchSize, localBatch: int64,
                                   it: ptr int64, perm: ptr int64, nRows: int64, viol, lossSum: ptr cdouble): int32
proc nimfm_ffm_sgd_epoch*(ctx: Ctx, m: DeviceFFM, X: DeviceDataset, cfg: ptr SgdCfg, it: ptr int64,
                         perm: ptr int64, nRows: int64, viol, lossSum: ptr cdouble): int32
proc nimfm_ffm_sgd_end*(ctx: Ctx, m: DeviceFFM): int32
# ---- the remaining entry points of include/nimfm_cuda.h (diagnostics, state transfer, measurement hooks)
proc nimfm_version*(): int32
proc nimfm_launch_count*(ctx: Ctx): int64
proc nimfm_stream_open*(ctx: Ctx, pathX, pathY: cstring, sh: ptr pointer): int32
proc nimfm_stream_info*(sh: pointer, kind: ptr int32, nRows, nCols, nnz, maxSegNnz, payloadBytes: ptr int64): int32
proc nimfm_stream_window_end*(sh: pointer, segBegin, maxBytes: int64): int64
proc nimfm_stream_load_window*(ctx: Ctx, sh: pointer, segBegin, segEnd: int64, ds: ptr DeviceDataset): int32
proc nimfm_stream_close*(sh: pointer): int32
proc nimfm_mem_info*(ctx: Ctx, freeBytes, totalBytes: ptr int64): int32
proc nimfm_stream_stats*(ctx: Ctx, h2dBytes, d2hBytes: ptr int64, hostThreads: ptr int32): int32
proc nimfm_comm_size*(ctx: Ctx): int32
proc nimfm_comm_allgather_i64*(ctx: Ctx, mine: ptr int64, count: int32, all: ptr int64): int32
proc nimfm_host_register*(ctx: Ctx, p: pointer, bytes: int64): int32      # page-lock a dataset's seqs once
proc nimfm_host_unregister*(ctx: Ctx, p: pointer): int32
proc nimfm_dataset_info*(ds: DeviceDataset, n, d, nnz: ptr int64, kind: ptr int32, nFields, maxRowNnz: ptr int64): int32
proc nimfm_dataset_download*(ctx: Ctx, ds: DeviceDataset, data: ptr cdouble, indices, indptr, fields: ptr int64): int32
proc nimfm_fm_loss_grad_host*(ctx: Ctx, fm: DeviceFM, nRows, d: int64, data: ptr cdouble, indices, indptr: ptr int64,
                             y: ptr cdouble, loss: int32, huberThreshold: cdouble, miniBatchSize, chunkRows: int64,
                             zeroGrads, allreduce: int32, lossSum: ptr cdouble): int32
proc nimfm_fm_decision_function_host*(ctx: Ctx, fm: DeviceFM, nRows, d: int64, data: ptr cdouble,
                                     indices, indptr: ptr int64, chunkRows: int64, outY: ptr cdouble): int32
proc nimfm_fm_get_grads*(ctx: Ctx, fm: DeviceFM, gP, gw, gb: ptr cdouble): int32
proc nimfm_fm_adagrad_get_state*(ctx: Ctx, fm: DeviceFM, gsP, gnP, gsw, gnw, gsb, gnb: ptr cdouble): int32
proc nimfm_fm_adagrad_set_state*(ctx: Ctx, fm: DeviceFM, gsP, gnP, gsw, gnw: ptr cdouble, gsb, gnb: cdouble): int32
proc nimfm_fm_cd_get_ypred*(ctx: Ctx, fm: DeviceFM, yPred: ptr cdouble): int32
proc nimfm_ffm_loss_grad*(ctx: Ctx, m: DeviceFFM, X: DeviceDataset, loss: int32, huberThreshold: cdouble,
                         rowBegin, nRows: int64, rowIdx: ptr int64, miniBatchSize: int64,
                         zeroGrads, allreduce: int32, lossSum: ptr cdouble): int32
proc nimfm_ffm_get_grads*(ctx: Ctx, m: DeviceFFM, gP, gw, gb: ptr cdouble): int32
proc nimfm_fm_time_loss_grad*(ctx: Ctx, fm: DeviceFM, X: DeviceDataset, loss: int32, nRows, miniBatchSize: int64,
                             reps, gradToo: int32, msPerLaunch: ptr cfloat): int32
proc nimfm_ffm_time_loss_grad*(ctx: Ctx, m: DeviceFFM, X: DeviceDataset, loss: int32, nRows, miniBatchSize: int64,
                              reps, gradToo: int32, msPerLaunch: ptr cfloat): int32
proc nimfm_timer_start*(ctx: Ctx): int32
proc nimfm_timer_stop*(ctx: Ctx, ms: ptr cfloat): int32
proc nimfm_fm_grad_device_ptr*(fm: DeviceFM, p: ptr pointer, nDoubles: ptr int64): int32
{.pop.}

# The Nim host layer over these symbols lives beside this file: device.nim (context, dataset / model twins),
# fit_cd.nim, fit_mbpsgd.nim, fit_adagrad.nim, fit_sgd.nim, fit_ffm.nim (the replaced `fit` bodies) and
# decision_function.nim -- see INTEGRATION.md for where each one plugs into nimfm's modules.
