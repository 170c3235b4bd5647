// Number formatting of json.dumps, as __host__ __device__ functions: the score-file writer
// (blp_json.cu) runs them on the device, tests/test_json_format.py compiles them for the host and
// compares them with Python's int.__repr__ / float.__repr__.
//
// Doubles: Ryu (Ulf Adams, "Ryu: fast float-to-string conversion", PLDI 2018) gives the shortest
// digit string that reads back as the same double, the closest one when there are several -- the
// digits of float.__repr__ (David Gay's dtoa, mode 0).  The layout is Python's 'r' format:
// exponent notation exactly when the decimal exponent is < -4 or >= 16, exponent signed and at
// least two digits long, ".0" after whole numbers in fixed notation; NaN / Infinity / -Infinity
// as json.dumps spells them.
//
// The power-of-5 tables (blp_json_pow5.h, 10.7 KB) are passed in as pointers: the device copy
// lives in global memory and is read through the read-only data cache, since the lanes of a warp
// index it at different places (constant memory would serialise those reads).
#ifndef BLP_JSON_FORMAT_CUH_
#define BLP_JSON_FORMAT_CUH_

#include <stdint.h>

#include "blp_json_pow5.h"

#ifndef __CUDACC__
#define __host__
#define __device__
#define __forceinline__ inline
#endif

namespace blp_json {

constexpr int kMaxDoubleChars = 24;   // -1.7976931348623157e+308
constexpr int kMaxIntChars = 20;      // -9223372036854775808

struct Pow5Tables {
    const unsigned long long* inv_split;   // [342][2] {low, high}
    const unsigned long long* split;       // [326][2]
};

__host__ __device__ __forceinline__ unsigned long long ld_table(const unsigned long long* p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

// Decimal digits of v (v < 10^17 for the Ryu output, any value for ints).
__host__ __device__ __forceinline__ int decimal_length(unsigned long long v) {
    int n = 1;
    while (v >= 10ull) {
        v /= 10ull;
        ++n;
    }
    return n;
}

// Writes the decimal digits of v to out[0..len) (len = decimal_length(v)).
__host__ __device__ __forceinline__ void write_digits(char* out, unsigned long long v, int len) {
    for (int i = len - 1; i >= 0; --i) {
        out[i] = (char)('0' + (int)(v % 10ull));
        v /= 10ull;
    }
}

// int.__repr__ of a signed 64-bit value; returns the number of bytes written.
__host__ __device__ __forceinline__ int format_int64(long long v, char* out) {
    int n = 0;
    unsigned long long u = (unsigned long long)v;
    if (v < 0) {
        out[n++] = '-';
        u = 0ull - u;
    }
    const int len = decimal_length(u);
    write_digits(out + n, u, len);
    return n + len;
}

// ------------------------------------------------------------------------------------ Ryu core
__host__ __device__ __forceinline__ int pow5bits(int e) { return (int)(((unsigned)e * 1217359u) >> 19) + 1; }
__host__ __device__ __forceinline__ int log10_pow2(int e) { return (int)(((unsigned)e * 78913u) >> 18); }
__host__ __device__ __forceinline__ int log10_pow5(int e) { return (int)(((unsigned)e * 732923u) >> 20); }

__host__ __device__ __forceinline__ int pow5_factor(unsigned long long v) {
    int count = 0;
    while (v % 5ull == 0ull) {
        v /= 5ull;
        ++count;
    }
    return count;
}
__host__ __device__ __forceinline__ bool multiple_of_pow5(unsigned long long v, int p) { return pow5_factor(v) >= p; }
__host__ __device__ __forceinline__ bool multiple_of_pow2(unsigned long long v, int p) {
    return (v & ((1ull << p) - 1ull)) == 0ull;
}

// (m * mul) >> j for a 125-bit mul = {lo, hi}, 64 < j < 192
__host__ __device__ __forceinline__ unsigned long long mul_shift64(unsigned long long m, unsigned long long lo,
                                                                   unsigned long long hi, int j) {
    const unsigned __int128 b0 = (unsigned __int128)m * lo;
    const unsigned __int128 b2 = (unsigned __int128)m * hi;
    return (unsigned long long)(((b0 >> 64) + b2) >> (j - 64));
}

// Shortest decimal of a finite positive double with ieee fields (mantissa, exponent):
// value = *digits * 10^*exp10.
__host__ __device__ inline void ryu_shortest(unsigned long long ieee_m, int ieee_e, const Pow5Tables& t,
                                             unsigned long long* digits, int* exp10) {
    int e2;
    unsigned long long m2;
    if (ieee_e == 0) {
        e2 = 1 - 1023 - 52 - 2;
        m2 = ieee_m;
    } else {
        e2 = ieee_e - 1023 - 52 - 2;
        m2 = (1ull << 52) | ieee_m;
    }
    const bool accept_bounds = (m2 & 1ull) == 0ull;
    const unsigned long long mv = 4ull * m2;
    const unsigned mm_shift = (ieee_m != 0ull || ieee_e <= 1) ? 1u : 0u;
    unsigned long long vr, vp, vm;
    int e10;
    bool vm_trailing_zeros = false, vr_trailing_zeros = false;
    if (e2 >= 0) {
        const int q = log10_pow2(e2) - (e2 > 3 ? 1 : 0);
        e10 = q;
        const int k = BLP_POW5_INV_BITCOUNT + pow5bits(q) - 1;
        const int i = -e2 + q + k;
        const unsigned long long lo = ld_table(t.inv_split + 2 * q), hi = ld_table(t.inv_split + 2 * q + 1);
        vr = mul_shift64(4ull * m2, lo, hi, i);
        vp = mul_shift64(4ull * m2 + 2ull, lo, hi, i);
        vm = mul_shift64(4ull * m2 - 1ull - mm_shift, lo, hi, i);
        if (q <= 21) {
            if (mv % 5ull == 0ull) vr_trailing_zeros = multiple_of_pow5(mv, q);
            else if (accept_bounds) vm_trailing_zeros = multiple_of_pow5(mv - 1ull - mm_shift, q);
            else vp -= multiple_of_pow5(mv + 2ull, q) ? 1ull : 0ull;
        }
    } else {
        const int q = log10_pow5(-e2) - (-e2 > 1 ? 1 : 0);
        e10 = q + e2;
        const int i = -e2 - q;
        const int k = pow5bits(i) - BLP_POW5_BITCOUNT;
        const int j = q - k;
        const unsigned long long lo = ld_table(t.split + 2 * i), hi = ld_table(t.split + 2 * i + 1);
        vr = mul_shift64(4ull * m2, lo, hi, j);
        vp = mul_shift64(4ull * m2 + 2ull, lo, hi, j);
        vm = mul_shift64(4ull * m2 - 1ull - mm_shift, lo, hi, j);
        if (q <= 1) {
            vr_trailing_zeros = true;
            if (accept_bounds) vm_trailing_zeros = mm_shift == 1u;
            else --vp;
        } else if (q < 63) {
            vr_trailing_zeros = multiple_of_pow2(mv, q);
        }
    }
    int removed = 0;
    unsigned last_removed = 0;
    unsigned long long output;
    if (vm_trailing_zeros || vr_trailing_zeros) {
        while (vp / 10ull > vm / 10ull) {
            vm_trailing_zeros &= vm % 10ull == 0ull;
            vr_trailing_zeros &= last_removed == 0u;
            last_removed = (unsigned)(vr % 10ull);
            vr /= 10ull;
            vp /= 10ull;
            vm /= 10ull;
            ++removed;
        }
        if (vm_trailing_zeros) {
            while (vm % 10ull == 0ull) {
                vr_trailing_zeros &= last_removed == 0u;
                last_removed = (unsigned)(vr % 10ull);
                vr /= 10ull;
                vp /= 10ull;
                vm /= 10ull;
                ++removed;
            }
        }
        if (vr_trailing_zeros && last_removed == 5u && vr % 2ull == 0ull) last_removed = 4u;   // round half to even
        output = vr + (((vr == vm && (!accept_bounds || !vm_trailing_zeros)) || last_removed >= 5u) ? 1ull : 0ull);
    } else {
        bool round_up = false;
        if (vp / 100ull > vm / 100ull) {
            round_up = vr % 100ull >= 50ull;
            vr /= 100ull;
            vp /= 100ull;
            vm /= 100ull;
            removed += 2;
        }
        while (vp / 10ull > vm / 10ull) {
            round_up = vr % 10ull >= 5ull;
            vr /= 10ull;
            vp /= 10ull;
            vm /= 10ull;
            ++removed;
        }
        output = vr + ((vr == vm || round_up) ? 1ull : 0ull);
    }
    *digits = output;
    *exp10 = e10 + removed;
}

__host__ __device__ __forceinline__ int copy_str(char* out, const char* s) {
    int n = 0;
    while (s[n]) {
        out[n] = s[n];
        ++n;
    }
    return n;
}

// json.dumps of a double (float.__repr__ for finite values); returns the bytes written
// (at most kMaxDoubleChars).
__host__ __device__ inline int format_double(double v, char* out, const Pow5Tables& t) {
    union {
        double d;
        unsigned long long u;
    } bits;
    bits.d = v;
    const bool neg = (bits.u >> 63) != 0ull;
    const int ieee_e = (int)((bits.u >> 52) & 0x7ffull);
    const unsigned long long ieee_m = bits.u & ((1ull << 52) - 1ull);
    if (ieee_e == 0x7ff) {
        if (ieee_m != 0ull) return copy_str(out, "NaN");
        return copy_str(out, neg ? "-Infinity" : "Infinity");
    }
    int n = 0;
    if (neg) out[n++] = '-';
    if (ieee_e == 0 && ieee_m == 0ull) return n + copy_str(out + n, "0.0");
    unsigned long long digits;
    int exp10;
    ryu_shortest(ieee_m, ieee_e, t, &digits, &exp10);
    const int len = decimal_length(digits);
    const int decpt = exp10 + len;          // value = 0.d1d2... * 10^decpt
    if (decpt <= -4 || decpt > 16) {         // d1.d2...e(+|-)XX
        char d[17];
        write_digits(d, digits, len);
        out[n++] = d[0];
        if (len > 1) {
            out[n++] = '.';
            for (int i = 1; i < len; ++i) out[n++] = d[i];
        }
        out[n++] = 'e';
        int x = decpt - 1;
        out[n++] = x < 0 ? '-' : '+';
        if (x < 0) x = -x;
        if (x >= 100) out[n++] = (char)('0' + x / 100);
        out[n++] = (char)('0' + (x / 10) % 10);
        out[n++] = (char)('0' + x % 10);
    } else if (decpt <= 0) {                 // 0.000ddd
        out[n++] = '0';
        out[n++] = '.';
        for (int i = 0; i < -decpt; ++i) out[n++] = '0';
        write_digits(out + n, digits, len);
        n += len;
    } else if (decpt >= len) {               // ddd000.0
        write_digits(out + n, digits, len);
        n += len;
        for (int i = len; i < decpt; ++i) out[n++] = '0';
        out[n++] = '.';
        out[n++] = '0';
    } else {                                 // dd.ddd
        char d[17];
        write_digits(d, digits, len);
        for (int i = 0; i < decpt; ++i) out[n++] = d[i];
        out[n++] = '.';
        for (int i = decpt; i < len; ++i) out[n++] = d[i];
    }
    return n;
}

}  // namespace blp_json

#endif  // BLP_JSON_FORMAT_CUH_
