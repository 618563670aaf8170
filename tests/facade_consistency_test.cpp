// facade_consistency_test.cpp -- one USCKF predict + update through the host C++ facade with NIS capture on, then
// mahalanobis() and consistencyStats(), for tests/test_consistency_facade.py to compare with the Python engine.
// Usage: facade_consistency_test IN OUT.  IN holds doubles: B, nk, nl, dt, then mu (B x QD), P (B x N x N), u (B x 6),
// Q (12 x 12), z (B x nk), R (nk x nk), truth (B x QD).  OUT receives the NIS (B), the full-state consistency stats (6)
// and the statek_i [24, 36) ones (6).  Prints "OK" on success, "MSCKF_REFUSED" when an MSCKF batch refused NIS capture
// as it must, and exits 3 with "NO_DEVICE" when there is no GPU (no CPU fallback).
#include <cstdio>
#include <vector>

#include "../slam-localization_b200/facade/localization_b200.hpp"

using namespace slb200;

static Vec take(const Vec &in, size_t &pos, size_t n) {
    Vec v(in.begin() + pos, in.begin() + pos + n);
    pos += n;
    return v;
}

int main(int argc, char **argv) {
    if (argc != 3) return 2;
    Vec in;
    {
        FILE *f = std::fopen(argv[1], "rb");
        if (!f) return 2;
        double x;
        while (std::fread(&x, sizeof(double), 1, f) == 1) in.push_back(x);
        std::fclose(f);
    }
    size_t pos = 0;
    const int B = (int)in[pos++], nk = (int)in[pos++], nl = (int)in[pos++];
    const double dt = in[pos++];
    const size_t N = 36 + nk + nl, QD = 39 + nk + nl;
    const Vec mu = take(in, pos, B * QD), P = take(in, pos, B * N * N), u = take(in, pos, (size_t)B * 6),
              Q = take(in, pos, 144), z = take(in, pos, (size_t)B * nk), R = take(in, pos, (size_t)nk * nk),
              truth = take(in, pos, B * QD);
    try {
        {
            Msckf m(4, 1, Vec(4 * 20, 0.0), Vec(4 * 18 * 18, 0.0));
            try {
                m.setNisCapture(true);
                std::printf("MSCKF_ACCEPTED\n");
                return 1;
            } catch (const Error &e) {
                if (e.code != SLB_ERR_INVALID) throw;
                std::printf("MSCKF_REFUSED\n");
            }
        }
        Usckf f(B, nk, nl, mu, P);
        f.setNisCapture(true);
        f.predict(SLB_PM_USCKF_TEST, u, dt, Q);
        f.update(z, SLB_MM_USCKF_VO, R);
        Vec out = f.mahalanobis();
        const Vec full = f.consistencyStats(truth, 0, (int)N), si = f.consistencyStats(truth, 24, 12);
        out.insert(out.end(), full.begin(), full.end());
        out.insert(out.end(), si.begin(), si.end());
        FILE *o = std::fopen(argv[2], "wb");
        if (!o) return 2;
        std::fwrite(out.data(), sizeof(double), out.size(), o);
        std::fclose(o);
        std::printf("OK\n");
    } catch (const Error &e) {
        if (e.code == SLB_ERR_NO_DEVICE) {
            std::printf("NO_DEVICE %s\n", e.what());
            return 3;
        }
        std::printf("ERROR %d %s\n", e.code, e.what());
        return 1;
    }
    return 0;
}
