// xmapper_b200 — text output on the device, shared by the SAM and the VCF / mutations formatters.  A writer with p == nullptr
// only counts bytes (the measure pass); with p set it writes them (the write pass).
#pragma once

struct SamOut {
  char* p; long long n;
  __device__ __forceinline__ void ch(char c) { if (p) p[n] = c; n++; }
  __device__ void str(const char* s, long long len) { for (long long i = 0; i < len; i++) ch(s[i]); }
  __device__ void lit(const char* s) { while (*s) ch(*s++); }
  __device__ void num(long long v) {  // "" + int
    if (v < 0) { ch('-'); v = -v; }
    char d[20]; int k = 0;
    do { d[k++] = (char)('0' + (int)(v % 10)); v /= 10; } while (v);
    while (k) ch(d[--k]);
  }
  // Java Float.toString of a finite float: shortest digits that identify it; decimal form for 1e-3 <= |v| < 1e7, else d.dddE<n>
  __device__ void jfloat(float v) {
    if (v == 0.0f) { if (signbit(v)) ch('-'); lit("0.0"); return; }
    if (v < 0) { ch('-'); v = -v; }
    const double s = (double)v;
    // powers of ten are exact doubles up to 1e22; negative exponents divide by the exact power instead of multiplying by an inexact one
    auto p10 = [](int k) { double r = 1.0; for (int i = 0; i < k; i++) r *= 10.0; return r; };
    auto scale = [&](double x, int ex) { return ex >= 0 ? x * p10(ex) : x / p10(-ex); };  // x * 10^ex
    int e10 = (int)floor(log10(s));
    if (scale(1.0, e10) > s) e10--;
    if (scale(1.0, e10 + 1) <= s) e10++;
    unsigned long long D = 0; int p = 1;
    for (p = 1; p <= 9; p++) {
      const int ex = e10 - p + 1;               // candidate = D * 10^ex with p digits
      D = (unsigned long long)rint(scale(s, -ex));
      if ((float)scale((double)D, ex) == v) break;
    }
    if (p > 9) p = 9;
    { unsigned long long lim = 1; for (int i = 0; i < p; i++) lim *= 10; if (D >= lim) { D /= 10; e10++; } }  // rounding carried into a new digit
    while (p > 1 && D % 10 == 0) { D /= 10; p--; }
    char dg[12];
    { unsigned long long t = D; for (int i = p - 1; i >= 0; i--) { dg[i] = (char)('0' + (int)(t % 10)); t /= 10; } }
    if (s >= 1e-3 && s < 1e7) {
      if (e10 >= 0) {
        for (int i = 0; i <= e10; i++) ch(i < p ? dg[i] : '0');
        ch('.');
        if (p > e10 + 1) { for (int i = e10 + 1; i < p; i++) ch(dg[i]); } else ch('0');
      } else {
        lit("0.");
        for (int i = 0; i < -e10 - 1; i++) ch('0');
        for (int i = 0; i < p; i++) ch(dg[i]);
      }
    } else {
      ch(dg[0]); ch('.');
      if (p > 1) { for (int i = 1; i < p; i++) ch(dg[i]); } else ch('0');
      ch('E'); num(e10);
    }
  }
  __device__ void score(const char* tag, double penalty) {  // formatSequencePenalty / formatQueryPenalty / formatNumber :263-277
    const float sc = (float)(-1 * penalty);
    const double scaled = (double)sc * (double)10000.0f;
    const long long r = (long long)floor(scaled + 0.5);        // Math.round(double)
    const float rounded = (float)r / 10000.0f;                 // long / float -> float
    lit(tag); lit("f:"); jfloat(rounded);
  }
};
