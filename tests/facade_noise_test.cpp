// facade_noise_test.cpp -- one USCKF predict + update through the host C++ facade with a process noise Q and a
// measurement noise R per instance (slb_set_noise_layout), for tests/test_noise_facade.py to compare with the Python
// engine.  Usage: facade_noise_test IN OUT.  IN holds doubles: B, nk, nl, dt, then mu (B x QD), P (B x N x N), u (B x 6),
// Q (B x 12 x 12), z (B x nk), R (B x nk x nk).  OUT receives mu, P and the status words (as doubles).
// Prints "OK" on success, "BADLEN" when a noise vector of the wrong length was refused as it must be, and exits 3 with
// "NO_DEVICE" when there is no GPU (no CPU fallback).
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
              Q = take(in, pos, (size_t)B * 144), z = take(in, pos, (size_t)B * nk), R = take(in, pos, (size_t)B * nk * nk);
    try {
        Usckf f(B, nk, nl, mu, P);
        try {   // neither 12*12 nor batch*12*12 doubles
            f.predict(SLB_PM_USCKF_TEST, u, dt, Vec(145, 0.0));
            std::printf("BADLEN_ACCEPTED\n");
            return 1;
        } catch (const Error &e) {
            if (e.code != SLB_ERR_INVALID) throw;
            std::printf("BADLEN\n");
        }
        f.predict(SLB_PM_USCKF_TEST, u, dt, Q);
        f.update(z, SLB_MM_USCKF_VO, R);
        Vec out = f.muState();
        const Vec Pk = f.PkAugmentedState();
        out.insert(out.end(), Pk.begin(), Pk.end());
        for (int32_t s : f.status()) out.push_back((double)s);
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
