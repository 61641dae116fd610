// met2_epg.cuh — the arithmetic of one EPG echo train (epg/epg.py:64-153), for a scalar type S.
//
// S = double is the dictionary (epg_decay, met2_epg.cu); S = met2::Dual (met2_param.cu) carries the derivatives with
// respect to T2 and the flip angle next to each value.  Both instantiations run the same operations in the same order,
// so the value part of a Dual evaluation is bit for bit the dictionary entry at the same (alpha, T2).  The caller owns
// the state layout and the shift; here are the coefficients, the initial state and the per-block operators.
#pragma once
// Include after met2_host.h (which supplies __device__ under the SIMT emulator).

namespace met2 {

template <class S>
struct EpgCoef {
    S e2;        // T2 decay over tau/2
    double e1;   // T1 recovery over tau/2
    S c2, s2, sa, ca;   // RF mixing of a (F+k, F-k, Zk) block
    S f0, fm1;   // initial state after the alpha/2 excitation: F0 and F-1
};

template <class S>
__device__ __forceinline__ EpgCoef<S> epg_coef(S alpha_deg, S T2, double T1, double tau) {
    const double rad = 3.14159265358979323846 / 180.0;
    const S a = alpha_deg * rad;
    const S a_exc = (alpha_deg / 2.0) * rad;   // epg.py:57: excitation = alpha/2
    const double half = tau / 2.0;
    EpgCoef<S> c;
    c.e2 = exp(-half * (1.0 / T2));
    c.e1 = exp(-half * (1.0 / T1));
    const S ch = cos(a / 2.0), sh = sin(a / 2.0);
    c.c2 = ch * ch;
    c.s2 = sh * sh;
    c.sa = sin(a);
    c.ca = cos(a);
    c.f0 = sin(a_exc);    // epg.py:145
    c.fm1 = cos(a_exc);   // epg.py:147 (index 2 of the state vector is the F-1 slot)
    return c;
}

// relaxation over tau/2 of one block (epg.py:82-85,133-141)
template <class S>
__device__ __forceinline__ void epg_relax(S& fp, S& fm, S& z, const EpgCoef<S>& c) {
    fp = fp * c.e2;
    fm = fm * c.e2;
    z = z * c.e1;
}

// RF mixing of one (F+k, F-k, Zk) block; F0 is not mixed (epg.py:118-131)
template <class S>
__device__ __forceinline__ void epg_rf(S& fp, S& fm, S& z, const EpgCoef<S>& c) {
    const S p = fp, m = fm, q = z;
    fp = c.c2 * p + c.s2 * m + c.sa * q;
    fm = c.s2 * p + c.c2 * m - c.sa * q;
    z = -0.5 * c.sa * p + 0.5 * c.sa * m + c.ca * q;
}

}  // namespace met2
