// SE3::exp of the Sophus stand-in (oracle/ref_shim/sophus/geometry.hpp), the same call the reference build exports
// as se3_exp (oracle/ref_lm_tu.cpp), built without the reference's sources: a = (upsilon, omega) -> 4x4 row-major.
// tests/test_oracle_ref.py compiles it together with oracle/ref_shim/standin_impl.cpp.
#include <Eigen/Dense>
#include <sophus/geometry.hpp>

extern "C" void standin_se3_exp(const double* a, double* T) {
    Eigen::MatrixXd v(6, 1);
    for (int i = 0; i < 6; ++i) v(i, 0) = a[i];
    const Eigen::MatrixXd m = Sophus::SE3<double>::exp(v).matrix();
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) T[i * 4 + j] = m(i, j);
}
