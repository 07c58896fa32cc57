"""oem_b200 -- B200-native (sm_100a) implementation of the hot path of the R package `oem`:
row-sharded FP64 Gram / X'y build + persistent OEM lambda-path kernel + logistic GEMV passes,
behind the reference's own entry points.  See DESIGN.md, INTEGRATION.md, include/oem_b200.h."""
from .api import (DeviceMatrix, OemB200Error, load, lib_path, make_opts, oem_fit_dense, oem_fit_big, oem_fit_sparse, oem_fit_logistic_sparse, oem_fit_logistic_dense,
                  oem_xval_dense, oem_xval_big, oem_xval_logistic_dense, logit_fold_pass, oem_xtx, predict_matrix, EXPORTS)

__all__ = ["DeviceMatrix", "OemB200Error", "load", "lib_path", "make_opts", "oem_fit_dense", "oem_fit_big", "oem_fit_sparse", "oem_fit_logistic_sparse",
           "oem_fit_logistic_dense", "oem_xval_dense", "oem_xval_big", "oem_xval_logistic_dense", "logit_fold_pass", "oem_xtx", "predict_matrix", "EXPORTS"]
