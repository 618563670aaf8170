// localization_b200.hpp -- host C++ facade over the C ABI of include/slb.h.
//
// Re-creates the public member surface of the reference's filter class templates for BATCHES of
// independent instances (a batch of one behaves like the reference object):
//   localization::Usckf<AugmentedState,State>   (src/filters/Usckf.hpp)   -> slb200::Usckf
//   localization::Msckf<MultiState,State>       (src/filters/Msckf.hpp)   -> slb200::Msckf
//   ukfom::ukf<state>                           (test/UKFoMUnitTest.cpp)  -> slb200::Ukf
//   localization::DataModel<double,D>           (src/core/DataModel.hpp)  -> slb200::DataModel<D>
// Same method names, argument meaning and error behaviour, with two differences forced by the GPU:
// (1) the process / measurement functors are ids of the device model catalogue (the reference's
//     boost::bind functors are host code and cannot be called from a kernel); (2) matrices are plain
//     row-major std::vector<double> (Eigen is not a dependency), instance-major for batches.
// Header-only; link with libslb.so.  No CUDA headers are needed by the includer.
#pragma once
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/slb.h"

namespace slb200 {

typedef std::vector<double> Vec;

enum CloningMode { STATEK = SLB_STATEK, STATEK_L = SLB_STATEK_L, STATEK_I = SLB_STATEK_I };  // Usckf.hpp:37-42

struct Error : std::runtime_error {
    int code;
    Error(int c, const char *what) : std::runtime_error(std::string(what) + ": " + slb_last_error()), code(c) {}
};
inline void check(int rc, const char *what) {
    if (rc != SLB_OK) throw Error(rc, what);
}

// RAII device buffer filled from host memory
class DevBuf {
    void *p_ = nullptr;
  public:
    DevBuf() {}
    DevBuf(const double *host, size_t n) { assign(host, n); }
    explicit DevBuf(const Vec &v) { assign(v.data(), v.size()); }
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { slb_dev_free(p_); }
    void assign(const double *host, size_t n) {
        slb_dev_free(p_);
        p_ = nullptr;
        check(slb_dev_alloc(n * sizeof(double), &p_), "slb_dev_alloc");
        check(slb_dev_copy(p_, host, n * sizeof(double), 1, nullptr), "slb_dev_copy");
    }
    const double *get() const { return static_cast<const double *>(p_); }
};

// RAII device buffer that is written by a kernel and read back
class DevOut {
    void *p_ = nullptr;
    size_t n_ = 0;
  public:
    explicit DevOut(size_t n) : n_(n) { check(slb_dev_alloc(n * sizeof(double), &p_), "slb_dev_alloc"); }
    DevOut(const Vec &init) : n_(init.size()) {
        check(slb_dev_alloc(n_ * sizeof(double), &p_), "slb_dev_alloc");
        check(slb_dev_copy(p_, init.data(), n_ * sizeof(double), 1, nullptr), "slb_dev_copy");
    }
    DevOut(const DevOut &) = delete;
    DevOut &operator=(const DevOut &) = delete;
    ~DevOut() { slb_dev_free(p_); }
    double *get() { return static_cast<double *>(p_); }
    void download(Vec &v) {
        v.resize(n_);
        check(slb_dev_copy(v.data(), p_, n_ * sizeof(double), 2, nullptr), "slb_dev_copy");
    }
};

// Common part: the device-resident batch (mu_state / Pk of every instance, Usckf.hpp:77-78)
class Batch {
  protected:
    slb_handle h_ = nullptr;
    int B_ = 0, N_ = 0, QD_ = 0;
    int noise_ = 0;   // slb_set_noise_layout flags of the handle
    // Noise matrices are n x n row-major: n*n doubles are shared by the batch, batch*n*n doubles are one matrix per
    // instance (with batch == 1 the two are the same thing, as in the reference).  Sets the handle's layout bit `bit`
    // from the length of `v`; any other length throws.
    void useNoise(const Vec &v, size_t n, int bit, const char *what) {
        int flag;
        if (v.size() == n * n) flag = 0;
        else if (v.size() == (size_t)B_ * n * n) flag = bit;
        else throw Error(SLB_ERR_INVALID, (std::string(what) + ": noise must hold n*n or batch*n*n doubles").c_str());
        const int flags = (noise_ & ~bit) | flag;
        if (flags != noise_) {
            check(slb_set_noise_layout(h_, flags), "slb_set_noise_layout");
            noise_ = flags;
        }
    }
    void create(int kind, int batch, int layout, int nk, int nl, int nclones, int device) {
        slb_config cfg = {};
        cfg.kind = kind; cfg.layout = layout; cfg.batch = batch; cfg.nk = nk; cfg.nl = nl; cfg.nclones = nclones;
        cfg.device = device;
        check(slb_create(&cfg, &h_), "slb_create");
        B_ = batch; N_ = slb_dof(h_); QD_ = slb_qdim(h_);
    }
  public:
    Batch() {}
    Batch(const Batch &) = delete;
    Batch &operator=(const Batch &) = delete;
    ~Batch() { slb_destroy(h_); }
    int batch() const { return B_; }
    unsigned getDOF() const { return (unsigned)N_; }   // State.hpp:373-376,590-593
    int qdim() const { return QD_; }
    slb_handle handle() const { return h_; }
    // muState() (Usckf.hpp:518, Msckf.hpp:376) / mu(): batch x qdim q-vectors
    Vec muState() const {
        Vec v((size_t)B_ * QD_);
        check(slb_download(h_, SLB_FIELD_MU, v.data(), v.size(), nullptr), "slb_download(mu)");
        return v;
    }
    // PkAugmentedState() (Usckf.hpp:523) / getPk() (Msckf.hpp:386) / sigma(): batch x N x N
    Vec Pk() const {
        Vec v((size_t)B_ * N_ * N_);
        check(slb_download(h_, SLB_FIELD_P, v.data(), v.size(), nullptr), "slb_download(P)");
        return v;
    }
    void setMu(const Vec &mu) { check(slb_upload(h_, SLB_FIELD_MU, mu.data(), mu.size(), nullptr), "slb_upload(mu)"); }
    void setPk(const Vec &P) { check(slb_upload(h_, SLB_FIELD_P, P.data(), P.size(), nullptr), "slb_upload(P)"); }  // Msckf.hpp:391
    std::vector<int32_t> status() const {
        std::vector<int32_t> s(B_);
        check(slb_download(h_, SLB_FIELD_STATUS, s.data(), s.size(), nullptr), "slb_download(status)");
        return s;
    }
    // Ensemble statistics (count, sum x, sum x x^T) of this batch's means, merged over an NCCL communicator when one
    // is given (ncclComm_t as void*, see slb_gather_stats): the path's only collective, end of run.
    Vec gatherStats(void *nccl_comm = nullptr) const {
        DevOut out((size_t)1 + N_ + (size_t)N_ * N_);
        check(slb_gather_stats(h_, nccl_comm, out.get(), nullptr), "slb_gather_stats");
        Vec v;
        out.download(v);
        return v;
    }
    // NIS capture (slb_set_nis_capture, Ukf / Usckf only): while on, every update stores the distance its gate was given
    void setNisCapture(bool on) { check(slb_set_nis_capture(h_, on ? 1 : 0), "slb_set_nis_capture"); }
    // The m2 = nu^T S^-1 nu of every instance's last update: what the reference passes to update()'s `mt` functor
    // (Usckf.hpp:262,290-294).  NaN where the update failed before forming it.  Needs setNisCapture(true).
    Vec mahalanobis() const {
        Vec v((size_t)B_);
        check(slb_download(h_, SLB_FIELD_NIS, v.data(), v.size(), nullptr), "slb_download(nis)");
        return v;
    }
    // {NEES count, sum, sum of squares, NIS count, sum, sum of squares} (slb_gather_consistency): NEES of `truth`
    // (batch x qdim q-vectors; empty = NIS only, with t0 = n = 0) over the tangent coordinates [t0, t0 + n), merged over
    // an NCCL communicator when one is given.
    Vec consistencyStats(const Vec &truth, int t0, int n, void *nccl_comm = nullptr) const {
        if (!truth.empty() && truth.size() != (size_t)B_ * QD_)
            throw Error(SLB_ERR_INVALID, "consistencyStats: truth must hold batch * qdim doubles");
        DevBuf dt;
        if (!truth.empty()) dt.assign(truth.data(), truth.size());
        DevOut out((size_t)6);
        check(slb_gather_consistency(h_, nccl_comm, truth.empty() ? nullptr : dt.get(), t0, n, nullptr, out.get(), nullptr),
              "slb_gather_consistency");
        Vec v;
        out.download(v);
        return v;
    }
  protected:
    // checkSigmaPoints() (Usckf.hpp:769-789, Msckf.hpp:818-838).  The reference assert()s; a batch returns per-instance
    // flags: bit 0 max|Pktest - Pk| > 1e-6, bit 1 the sigma-point mean moved away from mu_state, bit 2 LLT failed.
    std::vector<int32_t> checkSigmaPointsImpl() const {
        void *fl = nullptr;
        check(slb_dev_alloc((size_t)B_ * sizeof(int32_t), &fl), "slb_dev_alloc");
        const int rc = slb_check_sigma_points(h_, static_cast<int32_t *>(fl), nullptr, nullptr);
        std::vector<int32_t> out(B_);
        if (rc == SLB_OK) slb_dev_copy(out.data(), fl, (size_t)B_ * sizeof(int32_t), 2, nullptr);
        slb_dev_free(fl);
        check(rc, "slb_check_sigma_points");
        return out;
    }
};

// ---- ukfom::ukf<state>: ukf(mu, sigma), predict(g, R), update(z, h, Q[, mt]), mu(), sigma() ---------
class Ukf : public Batch {
  public:
    Ukf(int batch, int layout, const Vec &mu0, const Vec &sigma0, int device = 0) {
        create(SLB_KIND_UKF, batch, layout, 0, 0, 0, device);
        setMu(mu0);
        setPk(sigma0);
    }
    // u: batch x nu control inputs of process model `g`; Q: n x n, or batch x n x n (one per instance)
    void predict(int g, const Vec &u, double dt, const Vec &Q) {
        useNoise(Q, N_, SLB_NOISE_Q_PER_INSTANCE, "Ukf::predict");
        DevBuf du(u), dQ(Q);
        check(slb_ukf_predict(h_, g, du.get(), dt, dQ.get(), nullptr), "slb_ukf_predict");
    }
    // gate_dof = 0 is ukfom::accept_any_mahalanobis_distance; R: 3 x 3, or batch x 3 x 3
    void update(const Vec &z, int h, const Vec &R, int gate_dof = 0) {
        useNoise(R, 3, SLB_NOISE_R_PER_INSTANCE, "Ukf::update");
        DevBuf dz(z), dR(R);
        check(slb_ukf_update(h_, h, dz.get(), dR.get(), gate_dof, nullptr), "slb_ukf_update");
    }
    Vec mu() const { return muState(); }
    Vec sigma() const { return Pk(); }
};

// ---- localization::Usckf ----------------------------------------------------------------------------
class Usckf : public Batch {
    int nk_, nl_;
  public:
    // ctor #1 (Usckf.hpp:83): full augmented state and covariance
    Usckf(int batch, int nk, int nl, const Vec &state, const Vec &P0, int device = 0) : nk_(nk), nl_(nl) {
        create(SLB_KIND_USCKF, batch, 0, nk, nl, 0, device);
        setMu(state);
        setPk(P0);
    }
    // ctor #2 (Usckf.hpp:90-103): statek_i = single state, P_ii = P0_single, then cloning(STATEK_I),
    // cloning(STATEK_L) -- including the clone order that leaves Pk indefinite (SURVEY quirk Q13).
    Usckf(int batch, int nk, int nl, const Vec &single_state, const Vec &P0_single, bool /*ctor2*/, int device = 0)
        : nk_(nk), nl_(nl) {
        create(SLB_KIND_USCKF, batch, 0, nk, nl, 0, device);
        const int N = N_, QD = QD_;
        Vec mu((size_t)batch * QD, 0.0), P((size_t)batch * N * N, 0.0);
        for (int b = 0; b < batch; ++b) {
            double *m = &mu[(size_t)b * QD];
            m[3] = m[16] = 1.0;  // identity orientations of statek, statek_l
            for (int c = 0; c < 13; ++c) m[26 + c] = single_state[(size_t)b * 13 + c];
            for (int r = 0; r < 12; ++r)
                for (int c = 0; c < 12; ++c) P[(size_t)b * N * N + (24 + r) * N + 24 + c] = P0_single[(size_t)b * 144 + r * 12 + c];
        }
        setMu(mu);
        setPk(P);
        cloning(STATEK_I);
        cloning(STATEK_L);
    }
    // Q: 12 x 12, or batch x 12 x 12 (one per instance); R: nk x nk, or batch x nk x nk
    void predict(int f, const Vec &u, double dt, const Vec &Q) {                       // Usckf.hpp:107-244
        useNoise(Q, 12, SLB_NOISE_Q_PER_INSTANCE, "Usckf::predict");
        DevBuf du(u), dQ(Q);
        check(slb_usckf_predict(h_, f, du.get(), dt, dQ.get(), nullptr), "slb_usckf_predict");
    }
    void update(const Vec &z, int h, const Vec &R, int gate_dof = 0) {                // Usckf.hpp:246-308
        useNoise(R, (size_t)nk_, SLB_NOISE_R_PER_INSTANCE, "Usckf::update");
        DevBuf dz(z), dR(R);
        check(slb_usckf_update(h_, h, dz.get(), dR.get(), gate_dof, nullptr), "slb_usckf_update");
    }
    void setMeasurement(CloningMode mode, const Vec &z, const Vec &R) {               // Usckf.hpp:322-389
        const size_t len = mode == STATEK ? nk_ : nl_;
        if (z.size() != len * B_ || (R.size() != len * len && R.size() != B_ * len * len))   // the asserts at :325-327
            throw Error(SLB_ERR_INVALID, "setMeasurement: z.size() must equal R.rows() == R.cols()");
        useNoise(R, len, SLB_NOISE_R_PER_INSTANCE, "Usckf::setMeasurement");   // R: len x len, or batch x len x len
        DevBuf dz(z), dR(R);
        check(slb_usckf_set_measurement(h_, mode, dz.get(), dR.get(), nullptr), "slb_usckf_set_measurement");
    }
    void cloning(int mode) { check(slb_usckf_clone(h_, mode, nullptr), "slb_usckf_clone"); }  // Usckf.hpp:391-433
    // muSingleState(state = STATEK_I) (Usckf.hpp:457-478): batch x 13
    Vec muSingleState(int state = STATEK_I) const {
        const int off = state == STATEK_L ? 13 : state == STATEK ? 0 : 26;
        const Vec mu = muState();
        Vec out((size_t)B_ * 13);
        for (int b = 0; b < B_; ++b)
            for (int c = 0; c < 13; ++c) out[(size_t)b * 13 + c] = mu[(size_t)b * QD_ + off + c];
        return out;
    }
    // setSingleState(state, order) (Usckf.hpp:435-455) -- including order == STATEK writing statek_l (Q12)
    void setSingleState(const Vec &state, int order = STATEK_I) {
        const int off = order == STATEK_I ? 26 : (order == STATEK_L || order == STATEK) ? 13 : -1;
        if (off < 0) return;
        Vec mu = muState();
        for (int b = 0; b < B_; ++b)
            for (int c = 0; c < 13; ++c) mu[(size_t)b * QD_ + off + c] = state[(size_t)b * 13 + c];
        setMu(mu);
    }
    // PkSingleState(state) (Usckf.hpp:493-516): batch x 12 x 12
    Vec PkSingleState(int state = STATEK_I) const {
        const int off = state == STATEK_L ? 12 : state == STATEK ? 0 : 24;
        const Vec P = Pk();
        Vec out((size_t)B_ * 144);
        for (int b = 0; b < B_; ++b)
            for (int r = 0; r < 12; ++r)
                for (int c = 0; c < 12; ++c) out[(size_t)b * 144 + r * 12 + c] = P[(size_t)b * N_ * N_ + (off + r) * N_ + off + c];
        return out;
    }
    // setPkSingleState(Pk_i, order) (Usckf.hpp:480-491): only STATEK_I is honoured by the reference
    void setPkSingleState(const Vec &Pk_i, int order = STATEK_I) {
        if (order != STATEK_I) return;
        Vec P = Pk();
        for (int b = 0; b < B_; ++b)
            for (int r = 0; r < 12; ++r)
                for (int c = 0; c < 12; ++c) P[(size_t)b * N_ * N_ + (24 + r) * N_ + 24 + c] = Pk_i[(size_t)b * 144 + r * 12 + c];
        setPk(P);
    }
    Vec PkAugmentedState() const { return Pk(); }
    std::vector<int32_t> checkSigmaPoints() const { return checkSigmaPointsImpl(); }               // Usckf.hpp:769-789
};

// ---- localization::Msckf ----------------------------------------------------------------------------
class Msckf : public Batch {
  public:
    Msckf(int batch, int nclones, const Vec &state, const Vec &P0, int device = 0) {   // Msckf.hpp:80
        create(SLB_KIND_MSCKF, batch, 0, 0, 0, nclones, device);
        setMu(state);
        setPk(P0);
    }
    // Q: 12 x 12, or batch x 12 x 12 (one per instance)
    void predict(int f, const Vec &u, double dt, const Vec &Q) {                        // Msckf.hpp:89-189
        useNoise(Q, 12, SLB_NOISE_Q_PER_INSTANCE, "Msckf::predict");
        DevBuf du(u), dQ(Q);
        check(slb_msckf_predict(h_, f, du.get(), dt, dQ.get(), nullptr), "slb_msckf_predict");
    }
    // unsigned update(z, h, R[, mt]) (Msckf.hpp:196-277): returns the per-instance outlier counts (:276)
    std::vector<int32_t> update(const Vec &z, int h, const Vec &params, const Vec &R, bool gate = true) {
        const int m = (int)(z.size() / B_);
        DevBuf dz(z), dp(params), dR(R);
        check(slb_msckf_update(h_, h, dp.get(), m, dz.get(), dR.get(), gate ? 1 : 0, nullptr), "slb_msckf_update");
        std::vector<int32_t> out(B_);
        check(slb_download(h_, SLB_FIELD_OUTLIERS, out.data(), out.size(), nullptr), "slb_download(outliers)");
        return out;
    }
    // unsigned update(z, h, H, R[, mt]) (Msckf.hpp:285-349): the EKF flavour -- h also supplies its Jacobian H, outliers
    // are removed on the information matrix (:756-792), (H, innovation, R) are QR-compressed (:794-816)
    std::vector<int32_t> updateEKF(const Vec &z, int h, const Vec &params, const Vec &R, bool gate = true) {
        const int m = (int)(z.size() / B_);
        DevBuf dz(z), dp(params), dR(R);
        check(slb_msckf_update_ekf(h_, h, dp.get(), m, dz.get(), dR.get(), gate ? 1 : 0, nullptr), "slb_msckf_update_ekf");
        std::vector<int32_t> out(B_);
        check(slb_download(h_, SLB_FIELD_OUTLIERS, out.data(), out.size(), nullptr), "slb_download(outliers)");
        return out;
    }
    Vec getPk() const { return Pk(); }                                                    // Msckf.hpp:386
    std::vector<int32_t> checkSigmaPoints() const { return checkSigmaPointsImpl(); }      // Msckf.hpp:818-838
    // muSingleState(state) (Msckf.hpp:351-354): mu_state.statek = state; batch x 13
    void muSingleState(const Vec &state) {
        Vec mu = muState();
        for (int b = 0; b < B_; ++b)
            for (int c = 0; c < 13; ++c) mu[(size_t)b * QD_ + c] = state[(size_t)b * 13 + c];
        setMu(mu);
    }
    // setPkSingleState(Pk_i) (Msckf.hpp:363-366): Pk.block(0, 0, 12, 12) = Pk_i; batch x 12 x 12
    void setPkSingleState(const Vec &Pk_i) {
        Vec P = Pk();
        for (int b = 0; b < B_; ++b)
            for (int r = 0; r < 12; ++r)
                for (int c = 0; c < 12; ++c) P[(size_t)b * N_ * N_ + r * N_ + c] = Pk_i[(size_t)b * 144 + r * 12 + c];
        setPk(P);
    }
    Vec muSingleState() const {                                                           // Msckf.hpp:356
        const Vec mu = muState();
        Vec out((size_t)B_ * 13);
        for (int b = 0; b < B_; ++b)
            for (int c = 0; c < 13; ++c) out[(size_t)b * 13 + c] = mu[(size_t)b * QD_ + c];
        return out;
    }
    Vec getPkSingleState() const {                                                        // Msckf.hpp:368
        const Vec P = Pk();
        Vec out((size_t)B_ * 144);
        for (int b = 0; b < B_; ++b)
            for (int r = 0; r < 12; ++r)
                for (int c = 0; c < 12; ++c) out[(size_t)b * 144 + r * 12 + c] = P[(size_t)b * N_ * N_ + r * N_ + c];
        return out;
    }
};

// ---- localization::DataModel<double, D> over n estimates (DataModel.hpp) --------------------------------
template <int D>
struct DataModel {
    size_t n;
    Vec data;  // n x D          (DataModel.hpp:25)
    Vec Cov;   // n x D x D      (DataModel.hpp:26)
    explicit DataModel(size_t n_ = 1) : n(n_), data(n_ * D, 0.0), Cov(n_ * D * D, 0.0) {   // :32-36
        for (size_t i = 0; i < n; ++i)
            for (int d = 0; d < D; ++d) Cov[i * D * D + d * D + d] = 1.0e-10;               // ZERO_UNCERTAINTY
    }
    DataModel(const Vec &x, const Vec &C) : n(x.size() / D), data(x), Cov(C) {}              // :38-41
    int size() const { return D; }                                                           // :43-46
    void fusion(const DataModel &o) {                                                        // :48-60
        Vec xo(data.size()), Co(Cov.size());
        check(slb_datamodel_fuse_host(D, (int64_t)n, data.data(), Cov.data(), o.data.data(), o.Cov.data(), xo.data(),
                                      Co.data()),
              "slb_datamodel_fuse_host");
        data.swap(xo);
        Cov.swap(Co);
    }
    void safeFusion(const DataModel &o) {                                                    // :62-130 (D = 3, :104)
        if (D != 3) throw Error(SLB_ERR_INVALID, "safeFusion is only defined for D = 3 (DataModel.hpp:104)");
        DevBuf a(data), b(Cov), c(o.data), d(o.Cov);
        DevOut xo(data.size()), Co(Cov.size());
        check(slb_datamodel_safe_fuse((int64_t)n, a.get(), b.get(), c.get(), d.get(), xo.get(), Co.get(), nullptr),
              "slb_datamodel_safe_fuse");
        xo.download(data);
        Co.download(Cov);
    }
    DataModel operator+(const DataModel &o) const { return addsub(o, +1); }                  // :132-141
    DataModel operator-(const DataModel &o) const { return addsub(o, -1); }                  // :143-152 (Cov adds)
  private:
    DataModel addsub(const DataModel &o, int sign) const {
        DevBuf a(data), b(Cov), c(o.data), d(o.Cov);
        void *xo = nullptr, *Co = nullptr;
        check(slb_dev_alloc(data.size() * 8, &xo), "slb_dev_alloc");
        check(slb_dev_alloc(Cov.size() * 8, &Co), "slb_dev_alloc");
        DataModel r(n);
        int rc = slb_datamodel_addsub(D, (int64_t)n, sign, a.get(), b.get(), c.get(), d.get(), (double *)xo, (double *)Co, nullptr);
        if (rc == SLB_OK) rc = slb_dev_copy(r.data.data(), xo, data.size() * 8, 2, nullptr);
        if (rc == SLB_OK) rc = slb_dev_copy(r.Cov.data(), Co, Cov.size() * 8, 2, nullptr);
        slb_dev_free(xo);
        slb_dev_free(Co);
        check(rc, "slb_datamodel_addsub");
        return r;
    }
};

// ---- the error-state `Usckf` of src/filters/UsckfError.hpp (SURVEY 8f row f2) over n instances -------------------
// 3 x 15-DOF augmented state; mu_state as q-vectors (n x 48: per single state pos vel quat(w,x,y,z) gbias abias),
// mu_error vectorised (n x 45), Pk_error dense (n x 45 x 45), all device-resident between calls.
class UsckfError {
    size_t n_;
    DevOut mu_, err_, P_;
  public:
    UsckfError(const Vec &state, const Vec &error, const Vec &P0)                        // UsckfError.hpp:72-75
        : n_(state.size() / 48), mu_(state), err_(error), P_(P0) {}
    void ekfPredict(const Vec &F, const Vec &Q) {                                         // :87-137, F: n x 15 x 15
        DevBuf dF(F), dQ(Q);
        check(slb_ekf_predict((int64_t)n_, err_.get(), P_.get(), dF.get(), dQ.get(), nullptr), "slb_ekf_predict");
    }
    // ekfUpdate(z, H, R[, mt]) :322-384: returns the reference's return value per instance (zeros when accepted)
    Vec ekfUpdate(const Vec &z, const Vec &H, const Vec &R, bool gate = true) {
        const int m = (int)(z.size() / n_);
        DevBuf dz(z), dH(H), dR(R);
        DevOut ret(z.size());
        void *acc = nullptr;
        check(slb_dev_alloc(n_ * sizeof(int32_t), &acc), "slb_dev_alloc");
        const int rc = slb_ekf_update((int64_t)n_, m, mu_.get(), P_.get(), dz.get(), dH.get(), dR.get(), gate ? 1 : 0, ret.get(),
                                      (int32_t *)acc, nullptr);
        slb_dev_free(acc);
        check(rc, "slb_ekf_update");
        Vec out;
        ret.download(out);
        return out;
    }
    void ekfSingleUpdate(const Vec &z, const Vec &H, const Vec &R, bool gate = true) {   // :489-571, H: m x 15
        const int m = (int)(z.size() / n_);
        DevBuf dz(z), dH(H), dR(R);
        void *acc = nullptr;
        check(slb_dev_alloc(n_ * sizeof(int32_t), &acc), "slb_dev_alloc");
        const int rc = slb_ekf_single_update((int64_t)n_, m, mu_.get(), err_.get(), P_.get(), dz.get(), dH.get(), dR.get(),
                                             gate ? 1 : 0, (int32_t *)acc, nullptr);
        slb_dev_free(acc);
        check(rc, "slb_ekf_single_update");
    }
    void cloning() { check(slb_ekf_clone((int64_t)n_, mu_.get(), err_.get(), P_.get(), nullptr), "slb_ekf_clone"); }  // :573-603
    Vec muState() { Vec v; mu_.download(v); return v; }                                   // :606
    Vec muError() { Vec v; err_.download(v); return v; }                                  // :611
    Vec PkAugmentedState() { Vec v; P_.download(v); return v; }                           // :616
};

// ---- DeadReckon::updatePose with uncertainty over n poses (DeadReckon.hpp:30-79; SURVEY 8f row f4) ----------------
// pose = pos(3) quat(w,x,y,z); covariance 6 x 6 over [r t]
struct PoseWithUncertainty {
    Vec pose, cov;  // n x 7, n x 6 x 6
};
struct DeadReckon {
    // returns deltaPose; postPose = prevPose * deltaPose (TransformWithUncertainty::operator*, Transform.cpp:215-254)
    static PoseWithUncertainty updatePose(double delta_t, const Vec &vel0, const Vec &vel1, const Vec &velCov,
                                          const PoseWithUncertainty &prev, PoseWithUncertainty &post) {
        const size_t n = vel0.size() / 6;
        DevBuf v0(vel0), v1(vel1), vc(velCov), pp(prev.pose), pc(prev.cov);
        DevOut op(n * 7), oc(n * 36), dp(n * 7), dc(n * 36);
        check(slb_deadreckon_update_pose((int64_t)n, delta_t, v0.get(), v1.get(), vc.get(), pp.get(), pc.get(), op.get(), oc.get(),
                                         dp.get(), dc.get(), nullptr),
              "slb_deadreckon_update_pose");
        op.download(post.pose);
        oc.download(post.cov);
        PoseWithUncertainty delta;
        dp.download(delta.pose);
        dc.download(delta.cov);
        return delta;
    }
    static PoseWithUncertainty compose(const PoseWithUncertainty &t2, const PoseWithUncertainty &t1) {   // t2 * t1
        const size_t n = t2.pose.size() / 7;
        DevBuf a(t2.pose), b(t2.cov), c(t1.pose), d(t1.cov);
        DevOut op(n * 7), oc(n * 36);
        check(slb_transform_compose((int64_t)n, a.get(), b.get(), c.get(), d.get(), op.get(), oc.get(), nullptr),
              "slb_transform_compose");
        PoseWithUncertainty r;
        op.download(r.pose);
        oc.download(r.cov);
        return r;
    }
};

}  // namespace slb200
