// Shortest round-trip decimal text of an fp32 value widened to float64, byte for byte Python's `float.__repr__`
// (David Gay's dtoa, mode 0: the shortest digit string that reads back to the same double, the nearest of those to the
// exact value) in the spelling `json.dump` writes: NaN, Infinity, -Infinity; -0.0 keeps its sign; integral values get
// ".0"; fixed notation unless the decimal exponent is < -4 or >= 16, where it is d[.ddd]e(+|-)XX with at least two
// exponent digits.
//
// The digits come from Ryu (Ulf Adams, "Ryu: fast float-to-string conversion", PLDI 2018) for doubles, with 64x64->128
// products (__umul64hi on the device). Everything is integer arithmetic and the functions are __host__ __device__, so
// the CPU tests and the exhaustive 2^32 sweep (scripts/json_float_sweep.py) check the very code the kernels in
// results.cu run. A widened fp32 value has a binary exponent e2 = exponent - 1077 in [-203, 73], so only the table
// rows for that band are kept: POW5_INV[q] for q in [0, 20] (e2 >= 0) and POW5[i] for i in [0, 63] (e2 < 0):
//   POW5_INV[q] = floor(2^(pow5bits(q) - 1 + 125) / 5^q) + 1,  POW5[i] = 5^i scaled to 125 bits,
//   pow5bits(e) = ((e * 1217359) >> 19) + 1
// as {low, high} 64-bit words (tests/test_json_format.py recomputes them). The device reads them with __ldg.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define AVDF_HD __host__ __device__ __forceinline__
#else
#define AVDF_HD static inline
#endif

namespace avdf_json {

// longest text of a finite value ("-1.2345678901234567e-40"); the non-finite spellings are shorter
#define AVDF_JSON_NUM_MAX 23

#define AVDF_RYU_POW5_INV \
  {0x0000000000000001ull, 0x2000000000000000ull}, \
  {0x999999999999999aull, 0x1999999999999999ull}, \
  {0x47ae147ae147ae15ull, 0x147ae147ae147ae1ull}, \
  {0x6c8b4395810624deull, 0x10624dd2f1a9fbe7ull}, \
  {0x7a786c226809d496ull, 0x1a36e2eb1c432ca5ull}, \
  {0x61f9f01b866e43abull, 0x14f8b588e368f084ull}, \
  {0xb4c7f34938583622ull, 0x10c6f7a0b5ed8d36ull}, \
  {0x87a6520ec08d236aull, 0x1ad7f29abcaf4857ull}, \
  {0x9fb841a566d74f88ull, 0x15798ee2308c39dfull}, \
  {0xe62d01511f12a607ull, 0x112e0be826d694b2ull}, \
  {0xd6ae6881cb5109a4ull, 0x1b7cdfd9d7bdbab7ull}, \
  {0xdef1ed34a2a73aeaull, 0x15fd7fe17964955full}, \
  {0x7f27f0f6e885c8bbull, 0x119799812dea1119ull}, \
  {0x650cb4be40d60df8ull, 0x1c25c268497681c2ull}, \
  {0xea70909833de7193ull, 0x16849b86a12b9b01ull}, \
  {0x21f3a6e0297ec143ull, 0x1203af9ee756159bull}, \
  {0x6985d7cd0f313537ull, 0x1cd2b297d889bc2bull}, \
  {0x2137dfd73f5a90f9ull, 0x170ef54646d49689ull}, \
  {0xe75fe645cc4873faull, 0x12725dd1d243aba0ull}, \
  {0xa5663d3c7a0d865dull, 0x1d83c94fb6d2ac34ull}, \
  {0x511e976394d79eb1ull, 0x179ca10c9242235dull}

#define AVDF_RYU_POW5 \
  {0x0000000000000000ull, 0x1000000000000000ull}, \
  {0x0000000000000000ull, 0x1400000000000000ull}, \
  {0x0000000000000000ull, 0x1900000000000000ull}, \
  {0x0000000000000000ull, 0x1f40000000000000ull}, \
  {0x0000000000000000ull, 0x1388000000000000ull}, \
  {0x0000000000000000ull, 0x186a000000000000ull}, \
  {0x0000000000000000ull, 0x1e84800000000000ull}, \
  {0x0000000000000000ull, 0x1312d00000000000ull}, \
  {0x0000000000000000ull, 0x17d7840000000000ull}, \
  {0x0000000000000000ull, 0x1dcd650000000000ull}, \
  {0x0000000000000000ull, 0x12a05f2000000000ull}, \
  {0x0000000000000000ull, 0x174876e800000000ull}, \
  {0x0000000000000000ull, 0x1d1a94a200000000ull}, \
  {0x0000000000000000ull, 0x12309ce540000000ull}, \
  {0x0000000000000000ull, 0x16bcc41e90000000ull}, \
  {0x0000000000000000ull, 0x1c6bf52634000000ull}, \
  {0x0000000000000000ull, 0x11c37937e0800000ull}, \
  {0x0000000000000000ull, 0x16345785d8a00000ull}, \
  {0x0000000000000000ull, 0x1bc16d674ec80000ull}, \
  {0x0000000000000000ull, 0x1158e460913d0000ull}, \
  {0x0000000000000000ull, 0x15af1d78b58c4000ull}, \
  {0x0000000000000000ull, 0x1b1ae4d6e2ef5000ull}, \
  {0x0000000000000000ull, 0x10f0cf064dd59200ull}, \
  {0x0000000000000000ull, 0x152d02c7e14af680ull}, \
  {0x0000000000000000ull, 0x1a784379d99db420ull}, \
  {0x0000000000000000ull, 0x108b2a2c28029094ull}, \
  {0x0000000000000000ull, 0x14adf4b7320334b9ull}, \
  {0x4000000000000000ull, 0x19d971e4fe8401e7ull}, \
  {0x8800000000000000ull, 0x1027e72f1f128130ull}, \
  {0xaa00000000000000ull, 0x1431e0fae6d7217cull}, \
  {0xd480000000000000ull, 0x193e5939a08ce9dbull}, \
  {0xc9a0000000000000ull, 0x1f8def8808b02452ull}, \
  {0xbe04000000000000ull, 0x13b8b5b5056e16b3ull}, \
  {0xad85000000000000ull, 0x18a6e32246c99c60ull}, \
  {0xd8e6400000000000ull, 0x1ed09bead87c0378ull}, \
  {0x878fe80000000000ull, 0x13426172c74d822bull}, \
  {0x6973e20000000000ull, 0x1812f9cf7920e2b6ull}, \
  {0x03d0da8000000000ull, 0x1e17b84357691b64ull}, \
  {0x8262889000000000ull, 0x12ced32a16a1b11eull}, \
  {0x22fb2ab400000000ull, 0x178287f49c4a1d66ull}, \
  {0xabb9f56100000000ull, 0x1d6329f1c35ca4bfull}, \
  {0xcb54395ca0000000ull, 0x125dfa371a19e6f7ull}, \
  {0xbe2947b3c8000000ull, 0x16f578c4e0a060b5ull}, \
  {0x2db399a0ba000000ull, 0x1cb2d6f618c878e3ull}, \
  {0xfc90400474400000ull, 0x11efc659cf7d4b8dull}, \
  {0x7bb4500591500000ull, 0x166bb7f0435c9e71ull}, \
  {0xdaa16406f5a40000ull, 0x1c06a5ec5433c60dull}, \
  {0xa8a4de8459868000ull, 0x118427b3b4a05bc8ull}, \
  {0xd2ce16256fe82000ull, 0x15e531a0a1c872baull}, \
  {0x87819baecbe22800ull, 0x1b5e7e08ca3a8f69ull}, \
  {0xf4b1014d3f6d5900ull, 0x111b0ec57e6499a1ull}, \
  {0x71dd41a08f48af40ull, 0x1561d276ddfdc00aull}, \
  {0x0e549208b31adb10ull, 0x1aba4714957d300dull}, \
  {0x28f4db456ff0c8eaull, 0x10b46c6cdd6e3e08ull}, \
  {0x33321216cbecfb24ull, 0x14e1878814c9cd8aull}, \
  {0xbffe969c7ee839edull, 0x1a19e96a19fc40ecull}, \
  {0xf7ff1e21cf512434ull, 0x105031e2503da893ull}, \
  {0xf5fee5aa43256d41ull, 0x14643e5ae44d12b8ull}, \
  {0x337e9f14d3eec892ull, 0x197d4df19d605767ull}, \
  {0x005e46da08ea7ab6ull, 0x1fdca16e04b86d41ull}, \
  {0xa03aec4845928cb2ull, 0x13e9e4e4c2f34448ull}, \
  {0xc849a75a56f72fdeull, 0x18e45e1df3b0155aull}, \
  {0x7a5c1130ecb4fbd6ull, 0x1f1d75a5709c1ab1ull}, \
  {0xec798abe93f11d65ull, 0x13726987666190aeull}

#ifdef __CUDACC__
__device__ const uint64_t kPow5InvDev[21][2] = {AVDF_RYU_POW5_INV};
__device__ const uint64_t kPow5Dev[64][2] = {AVDF_RYU_POW5};
#endif
static const uint64_t kPow5InvHost[21][2] = {AVDF_RYU_POW5_INV};
static const uint64_t kPow5Host[64][2] = {AVDF_RYU_POW5};

AVDF_HD void table_row(bool inv, int idx, uint64_t& lo, uint64_t& hi) {
#ifdef __CUDA_ARCH__
  const uint64_t* p = inv ? kPow5InvDev[idx] : kPow5Dev[idx];
  lo = __ldg(p); hi = __ldg(p + 1);
#else
  const uint64_t* p = inv ? kPow5InvHost[idx] : kPow5Host[idx];
  lo = p[0]; hi = p[1];
#endif
}

AVDF_HD uint64_t umulhi(uint64_t a, uint64_t b) {
#ifdef __CUDA_ARCH__
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

AVDF_HD int pow5bits(int e) { return (int)(((uint32_t)e * 1217359u) >> 19) + 1; }
AVDF_HD int log10pow2(int e) { return (int)(((uint32_t)e * 78913u) >> 18); }
AVDF_HD int log10pow5(int e) { return (int)(((uint32_t)e * 732923u) >> 20); }

// (m * mul) >> j for m < 2^55, 64 <= j < 128
AVDF_HD uint64_t mul_shift(uint64_t m, uint64_t lo, uint64_t hi, int j) {
  const uint64_t low1 = m * hi, high1 = umulhi(m, hi);
  const uint64_t high0 = umulhi(m, lo);
  const uint64_t sum = high0 + low1;
  const uint64_t h = high1 + (sum < high0 ? 1 : 0);
  const int d = j - 64;
  return d == 0 ? sum : (h << (64 - d)) | (sum >> d);
}

AVDF_HD bool multiple_of_pow5(uint64_t v, int p) {
  int c = 0;
  while (v != 0 && v % 5 == 0) { v /= 5; ++c; if (c >= p) return true; }
  return c >= p;
}

AVDF_HD int decimal_length(uint64_t v) {
  int n = 1;
  while (v >= 10) { v /= 10; ++n; }
  return n;
}

// Shortest digits of the double equal to the fp32 value with bits `bits` (finite, non-zero): value = digits * 10^exp10.
AVDF_HD void shortest(uint32_t bits, uint64_t& digits, int& exp10) {
  const uint32_t e8 = (bits >> 23) & 0xff, m23 = bits & 0x7fffff;
  uint64_t m2;
  int e2;
  if (e8 != 0) {
    m2 = (uint64_t)(m23 | 0x800000u) << 29;
    e2 = (int)e8 - 181;
  } else {                                  // fp32 subnormal: a normal double
    int s = 52;
    for (uint32_t t = m23; t > 1; t >>= 1) --s;
    m2 = (uint64_t)m23 << s;
    e2 = -151 - s;
  }
  const bool even = (m2 & 1) == 0, accept = even;
  const uint64_t mv = 4 * m2;
  const uint32_t mm_shift = (m2 & ((1ull << 52) - 1)) != 0 ? 1 : 0;   // the double's exponent is never <= 1 here
  uint64_t vr, vp, vm;
  int e10;
  bool vm_tz = false, vr_tz = false;
  if (e2 >= 0) {
    const int q = log10pow2(e2) - (e2 > 3 ? 1 : 0);
    e10 = q;
    const int k = 125 + pow5bits(q) - 1;
    const int i = -e2 + q + k;
    uint64_t lo, hi;
    table_row(true, q, lo, hi);
    vr = mul_shift(4 * m2, lo, hi, i);
    vp = mul_shift(4 * m2 + 2, lo, hi, i);
    vm = mul_shift(4 * m2 - 1 - mm_shift, lo, hi, i);
    if (q <= 21) {
      if (mv % 5 == 0) vr_tz = multiple_of_pow5(mv, q);
      else if (accept) vm_tz = multiple_of_pow5(mv - 1 - mm_shift, q);
      else vp -= multiple_of_pow5(mv + 2, q) ? 1 : 0;
    }
  } else {
    const int q = log10pow5(-e2) - (-e2 > 1 ? 1 : 0);
    e10 = q + e2;
    const int i = -e2 - q;
    const int k = pow5bits(i) - 125;
    const int j = q - k;
    uint64_t lo, hi;
    table_row(false, i, lo, hi);
    vr = mul_shift(4 * m2, lo, hi, j);
    vp = mul_shift(4 * m2 + 2, lo, hi, j);
    vm = mul_shift(4 * m2 - 1 - mm_shift, lo, hi, j);
    if (q <= 1) {
      vr_tz = true;
      if (accept) vm_tz = mm_shift == 1;
      else --vp;
    } else if (q < 63) {
      vr_tz = (mv & ((1ull << q) - 1)) == 0;
    }
  }
  int removed = 0;
  uint32_t last = 0;
  uint64_t out;
  if (vm_tz || vr_tz) {
    while (vp / 10 > vm / 10) {
      vm_tz &= vm % 10 == 0;
      vr_tz &= last == 0;
      last = (uint32_t)(vr % 10);
      vr /= 10; vp /= 10; vm /= 10; ++removed;
    }
    if (vm_tz) {
      while (vm % 10 == 0) {
        vr_tz &= last == 0;
        last = (uint32_t)(vr % 10);
        vr /= 10; vp /= 10; vm /= 10; ++removed;
      }
    }
    if (vr_tz && last == 5 && vr % 2 == 0) last = 4;      // exactly half-way: round to even
    out = vr + (((vr == vm && (!accept || !vm_tz)) || last >= 5) ? 1 : 0);
  } else {
    bool up = false;
    while (vp / 10 > vm / 10) {
      up = vr % 10 >= 5;
      vr /= 10; vp /= 10; vm /= 10; ++removed;
    }
    out = vr + ((vr == vm || up) ? 1 : 0);
  }
  digits = out;
  exp10 = e10 + removed;
}

// Writes the JSON text of the fp32 value `bits` to `out` (when not NULL) and returns its length (<= AVDF_JSON_NUM_MAX).
AVDF_HD int format_f32(uint32_t bits, char* out) {
  const bool neg = (bits >> 31) != 0;
  const uint32_t mag = bits & 0x7fffffffu;
  if (mag >= 0x7f800000u) {
    if (mag > 0x7f800000u) {
      if (out) { out[0] = 'N'; out[1] = 'a'; out[2] = 'N'; }
      return 3;
    }
    const char* s = "-Infinity";
    const int o = neg ? 0 : 1;
    if (out) for (int c = o; c < 9; ++c) out[c - o] = s[c];
    return 9 - o;
  }
  int p = 0;
  if (neg) { if (out) out[0] = '-'; p = 1; }
  if (mag == 0) {
    if (out) { out[p] = '0'; out[p + 1] = '.'; out[p + 2] = '0'; }
    return p + 3;
  }
  uint64_t v;
  int e10;
  shortest(bits, v, e10);
  const int n = decimal_length(v);
  const int x = e10 + n - 1;                 // scientific exponent: value = d.ddd * 10^x
  if (x < -4 || x >= 16) {
    const int exp_digits = (x <= -100 || x >= 100) ? 3 : 2;
    const int len = p + n + (n > 1 ? 1 : 0) + 2 + exp_digits;
    if (out) {
      for (int k = n - 1; k >= 0; --k) { out[p + (k == 0 ? 0 : k + 1)] = (char)('0' + v % 10); v /= 10; }
      if (n > 1) out[p + 1] = '.';
      int q = p + n + (n > 1 ? 1 : 0);
      out[q++] = 'e';
      out[q++] = x < 0 ? '-' : '+';
      int a = x < 0 ? -x : x;
      for (int c = exp_digits - 1; c >= 0; --c) { out[q + c] = (char)('0' + a % 10); a /= 10; }
    }
    return len;
  }
  if (x >= 0) {
    // integer part x + 1 digits; digits beyond it go after the point, or ".0" when there are none
    const int int_digits = x + 1;
    if (n <= int_digits) {
      const int len = p + int_digits + 2;
      if (out) {
        for (int c = n; c < int_digits; ++c) out[p + c] = '0';
        for (int k = n - 1; k >= 0; --k) { out[p + k] = (char)('0' + v % 10); v /= 10; }
        out[p + int_digits] = '.'; out[p + int_digits + 1] = '0';
      }
      return len;
    }
    const int len = p + n + 1;
    if (out) {
      for (int k = n - 1; k >= 0; --k) { out[p + (k < int_digits ? k : k + 1)] = (char)('0' + v % 10); v /= 10; }
      out[p + int_digits] = '.';
    }
    return len;
  }
  const int zeros = -x - 1;                  // "0." then -x - 1 zeros then the digits
  const int len = p + 2 + zeros + n;
  if (out) {
    out[p] = '0'; out[p + 1] = '.';
    for (int c = 0; c < zeros; ++c) out[p + 2 + c] = '0';
    for (int k = n - 1; k >= 0; --k) { out[p + 2 + zeros + k] = (char)('0' + v % 10); v /= 10; }
  }
  return len;
}

}  // namespace avdf_json
