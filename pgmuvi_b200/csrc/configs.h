// Every compiled (KIND, QT, D) instantiation of the model kernels, one PGM_CONFIG line each (the
// KIND numbers are the PGM_KIND_* of include/pgmuvi_b200.h).  build.py compiles inst.cu once per
// line; cabi.cu sends a (kind, Q) model to the line of its kind with the smallest QT >= max(Q, 1).

// 1-D SM, 2-D ARD product-of-sums, 2-D ARD sum-of-products: QT = padded mixture count
PGM_CONFIG(0, 1, 1)
PGM_CONFIG(0, 2, 1)
PGM_CONFIG(0, 4, 1)
PGM_CONFIG(0, 8, 1)
PGM_CONFIG(1, 1, 2)
PGM_CONFIG(1, 2, 2)
PGM_CONFIG(1, 4, 2)
PGM_CONFIG(1, 8, 2)
PGM_CONFIG(2, 1, 2)
PGM_CONFIG(2, 2, 2)
PGM_CONFIG(2, 4, 2)
PGM_CONFIG(2, 8, 2)
// separable SM(time) x {RBF, Matern-1.5, RQ, Constant}(wavelength): QT in {4, 8}
PGM_CONFIG(3, 4, 2)
PGM_CONFIG(3, 8, 2)
PGM_CONFIG(4, 4, 2)
PGM_CONFIG(4, 8, 2)
PGM_CONFIG(5, 4, 2)
PGM_CONFIG(5, 8, 2)
PGM_CONFIG(6, 4, 2)
PGM_CONFIG(6, 8, 2)
// stationary time kernels, kind = 8 + 5 * TK + WK, no mixtures (QT = 4): TK in {RBF, Matern-1.5,
// quasi-periodic}, WK = 0 (1-D) or a wavelength kernel (2-D)
PGM_CONFIG(8, 4, 1)
PGM_CONFIG(9, 4, 2)
PGM_CONFIG(10, 4, 2)
PGM_CONFIG(11, 4, 2)
PGM_CONFIG(12, 4, 2)
PGM_CONFIG(13, 4, 1)
PGM_CONFIG(14, 4, 2)
PGM_CONFIG(15, 4, 2)
PGM_CONFIG(16, 4, 2)
PGM_CONFIG(17, 4, 2)
PGM_CONFIG(18, 4, 1)
PGM_CONFIG(19, 4, 2)
PGM_CONFIG(20, 4, 2)
PGM_CONFIG(21, 4, 2)
PGM_CONFIG(22, 4, 2)
// quasi-periodic + RBF (PeriodicPlusStochasticGPModel), Matern-0.5 / Matern-2.5 (MaternGPModel
// nu): 1-D only
PGM_CONFIG(23, 4, 1)
PGM_CONFIG(28, 4, 1)
PGM_CONFIG(33, 4, 1)
