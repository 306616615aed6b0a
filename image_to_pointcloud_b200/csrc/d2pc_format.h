// d2pc_format.h -- byte layouts of the reference's point-cloud writers (row f3), written once for
// host and device like d2pc_math.h (tests/hostmath compiles it with g++ and checks it against
// Python's own formatting).
//
//   save_xyz  (backend/app.py:379-389):  f"{x:.6f} {y:.6f} {z:.6f} {int(r)} {int(g)} {int(b)}\n"
//             x, y, z are numpy.float32 scalars: __format__ goes through the exact double value,
//             fixed notation, 6 decimals, round-half-even on the exact binary value.
//   save_las  (app.py:343-377): LAS 1.2 point format 2, 26-byte records,
//             X = int32(np.round((float64(x) - offset) / 0.01)), colours clip(c,0,255).astype(uint16)*256.
//   save_ply  (app.py:329-341, Open3D binary_little_endian): double x, y, z; uchar red, green, blue
//             = round(clamp(float32(c / 255.0), 0, 1) * 255); with normals (51 bytes): double x, y, z,
//             nx, ny, nz; uchar red, green, blue.
#ifndef D2PC_FORMAT_H_
#define D2PC_FORMAT_H_

#include "d2pc_math.h"

namespace d2pc {

constexpr int kXyzMaxNumber = 1 + 20 + 1 + 6;            // sign, <= 20 integer digits, '.', 6 decimals
constexpr int kXyzMaxLine = 3 * kXyzMaxNumber + 3 * 11 + 6;  // three coordinates, three ints, 5 spaces + '\n'
constexpr int kLasRecordBytes = 26;
constexpr int kPlyRecordBytes = 27;
constexpr int kPlyNormalRecordBytes = 51;
constexpr int kPlyFaceRecordBytes = 13;

// Writes the decimal digits of n (at least one) to out, returns the count.
D2PC_HD int put_u64(unsigned long long n, char *out) {
  int k = 1;  // number of digits
  if (n <= 0xFFFFFFFFull) {
    uint32_t m = (uint32_t)n;
    for (uint32_t t = m; t >= 10u; t /= 10u) ++k;
    for (int i = k - 1; i >= 0; --i) { out[i] = (char)('0' + (int)(m % 10u)); m /= 10u; }
  } else {
    for (unsigned long long t = n; t >= 10ull; t /= 10ull) ++k;
    for (int i = k - 1; i >= 0; --i) { out[i] = (char)('0' + (int)(n % 10ull)); n /= 10ull; }
  }
  return k;
}

// format(float(v), ".6f") for a float32 v.  Returns the length, or -1 when |v| >= 2^44 (the scaled
// integer would not fit 64 bits; the caller reports an error instead of printing something else).
D2PC_HD int format_fixed6(float v, char *out) {
  const uint32_t bits = f32_bits(v);
  const bool neg = (bits >> 31) != 0u;
  const uint32_t ex = (bits >> 23) & 0xFFu;
  uint32_t man = bits & 0x7FFFFFu;
  int n = 0;
  if (ex == 0xFFu) {
    if (man != 0u) { out[0] = 'n'; out[1] = 'a'; out[2] = 'n'; return 3; }  // Python prints "nan" for either sign
    if (neg) out[n++] = '-';
    out[n++] = 'i'; out[n++] = 'n'; out[n++] = 'f';
    return n;
  }
  int e;  // v = man * 2^e
  if (ex == 0u) {
    e = -149;
  } else {
    man |= 0x800000u;
    e = (int)ex - 150;
  }
  const unsigned long long a = (unsigned long long)man * 1000000ull;  // < 2^44
  unsigned long long scaled;                                           // round_half_even(|v| * 10^6)
  if (e >= 0) {
    if (e > 20) return -1;
    scaled = a << e;
  } else {
    const int sh = -e;
    if (sh >= 64) {
      scaled = 0ull;  // a / 2^sh < 2^-20
    } else {
      unsigned long long q = a >> sh;
      const unsigned long long rem = a & ((1ull << sh) - 1ull), half = 1ull << (sh - 1);
      if (rem > half || (rem == half && (q & 1ull))) ++q;
      scaled = q;
    }
  }
  if (neg) out[n++] = '-';
  n += put_u64(scaled / 1000000ull, out + n);
  out[n++] = '.';
  uint32_t frac = (uint32_t)(scaled % 1000000ull);
  for (int i = 5; i >= 0; --i) {
    out[n + i] = (char)('0' + (int)(frac % 10u));
    frac /= 10u;
  }
  return n + 6;
}

// str(int(c)) for a float32 c (truncation toward zero).  -1 for NaN / inf / |c| >= 2^31
// (Python raises there; so does the caller).
D2PC_HD int format_int(float c, char *out) {
  if (!is_finite_f32(c) || !(fabsf(c) < 2147483648.0f)) return -1;
  const int32_t i = (int32_t)c;
  int n = 0;
  unsigned long long mag = (unsigned long long)(i < 0 ? -(long long)i : (long long)i);
  if (i < 0) out[n++] = '-';
  return n + put_u64(mag, out + n);
}

// One line of save_xyz; returns its length or -1.
D2PC_HD int format_xyz_line(const float *p, const float *c, char *out) {
  int n = 0;
  for (int k = 0; k < 3; ++k) {
    const int m = format_fixed6(p[k], out + n);
    if (m < 0) return -1;
    n += m;
    out[n++] = ' ';
  }
  for (int k = 0; k < 3; ++k) {
    const int m = format_int(c[k], out + n);
    if (m < 0) return -1;
    n += m;
    out[n++] = (k == 2) ? '\n' : ' ';
  }
  return n;
}

D2PC_HD void put_le16(uint8_t *o, uint32_t v) { o[0] = (uint8_t)(v & 255u); o[1] = (uint8_t)((v >> 8) & 255u); }
D2PC_HD void put_le32(uint8_t *o, uint32_t v) { put_le16(o, v & 0xFFFFu); put_le16(o + 2, v >> 16); }
D2PC_HD void put_le64(uint8_t *o, unsigned long long v) { put_le32(o, (uint32_t)v); put_le32(o + 4, (uint32_t)(v >> 32)); }

// LAS 1.2 point format 2 record.  Returns false when a scaled coordinate leaves the int32 range.
//   X = np.round((float64(x) - offset) / scale)   (rint: half to even)
//   red = uint16(clip(c, 0, 255)) * 256            (uint16 arithmetic)
D2PC_HD bool las_record(const float *p, const float *c, const double off[3], double scale, uint8_t *o,
                        int32_t xyz_i[3]) {
  bool ok = true;
  for (int k = 0; k < 3; ++k) {
    const double q = rint(((double)p[k] - off[k]) / scale);
    if (!(q >= -2147483648.0 && q <= 2147483647.0)) { ok = false; xyz_i[k] = 0; }
    else xyz_i[k] = (int32_t)q;
    put_le32(o + 4 * k, (uint32_t)xyz_i[k]);
  }
  put_le16(o + 12, 0u);  // intensity
  o[14] = 0;             // return number / number of returns / scan direction / edge of flight line
  o[15] = 0;             // classification
  o[16] = 0;             // scan angle rank
  o[17] = 0;             // user data
  put_le16(o + 18, 0u);  // point source id
  for (int k = 0; k < 3; ++k) {
    float cc = c[k];
    cc = cc < 0.0f ? 0.0f : cc;   // np.clip (NaN propagates; astype(uint16) of NaN is 0 on x86)
    cc = cc > 255.0f ? 255.0f : cc;
    const uint32_t u = (cc == cc) ? (uint32_t)cc : 0u;
    put_le16(o + 20 + 2 * k, (u * 256u) & 0xFFFFu);
  }
  return ok;
}

D2PC_HD void put_f64(uint8_t *o, double d) {
  unsigned long long u;
#if defined(__CUDA_ARCH__)
  u = (unsigned long long)__double_as_longlong(d);
#else
  memcpy(&u, &d, 8);
#endif
  put_le64(o, u);
}

// Open3D's PLY colour byte: round(clamp(float32(c / 255), 0, 1) * 255)
D2PC_HD uint8_t ply_colour(float c) {
  const float c32 = c / 255.0f;  // colors / 255.0 stays float32 (weak Python scalar)
  double t = (double)c32;
  t = t < 0.0 ? 0.0 : t;
  t = t > 1.0 ? 1.0 : t;
  return (t == t) ? (uint8_t)(int)floor(t * 255.0 + 0.5) : (uint8_t)0;  // std::round of a value >= 0
}

// Open3D binary PLY vertex: three float64 coordinates, three uchar colours.
D2PC_HD void ply_record(const float *p, const float *c, uint8_t *o) {
  for (int k = 0; k < 3; ++k) put_f64(o + 8 * k, (double)p[k]);
  for (int k = 0; k < 3; ++k) o[24 + k] = ply_colour(c[k]);
}

// Open3D binary PLY vertex of a cloud with normals, in its writer's property order: float64 x, y, z, nx, ny, nz,
// then uchar red, green, blue.
D2PC_HD void ply_normal_record(const float *p, const double *nrm, const float *c, uint8_t *o) {
  for (int k = 0; k < 3; ++k) put_f64(o + 8 * k, (double)p[k]);
  for (int k = 0; k < 3; ++k) put_f64(o + 24 + 8 * k, nrm[k]);
  for (int k = 0; k < 3; ++k) o[48 + k] = ply_colour(c[k]);
}

// Open3D binary PLY face: uchar 3 (property list uchar uint vertex_indices), then three uint32 vertex ids.
D2PC_HD void ply_face_record(const int32_t *t, uint8_t *o) {
  o[0] = 3;
  for (int k = 0; k < 3; ++k) put_le32(o + 1 + 4 * k, (uint32_t)t[k]);
}

// preview stride of app.py:495-500: points[::stride] with stride = max(1, n // max_preview) when
// n > max_preview, else every row.
D2PC_HD uint32_t preview_stride(uint32_t n, uint32_t max_preview) {
  if (n <= max_preview || max_preview == 0u) return 1u;
  const uint32_t s = n / max_preview;
  return s < 1u ? 1u : s;
}

}  // namespace d2pc
#endif  // D2PC_FORMAT_H_
