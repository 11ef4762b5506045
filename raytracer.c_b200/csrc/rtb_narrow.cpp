/* Host side of the narrowed mesh upload (rtb_scene.cu: upload_narrowed).
 *
 * The reference's Vertex is five doubles (pos.xyz, tex.uv: raytracer.h:104-108), 120 B per triangle, but every
 * coordinate of an OBJ-loaded mesh is a float widened to double (tinyobj_loader.h:470-481).  The staging threads
 * that copy a caller's pageable vertex array into page-locked buffers therefore convert while they copy:
 * 15 doubles -> 15 floats per triangle, half the bytes written by the host and half the bytes over PCIe.  The
 * conversion reports whether every one of the five lanes -- positions and texture coordinates -- survived it
 * exactly; if one did not (a mesh transformed in double, main.c:140-147, or texture coordinates computed in double)
 * the caller uploads that piece as raw doubles instead, so the exact triangle test and the checker pattern always
 * see the numbers the reference would see. */
#include <cstddef>
#include <immintrin.h>

namespace
{
bool narrow_scalar(const double *src, float *dst, size_t n_vertices)
{
  bool exact = true;
  for (size_t v = 0; v < n_vertices; v++)
    for (int a = 0; a < 5; a++)
    {
      const double x = src[5 * v + a];
      const float f = (float)x;
      dst[5 * v + a] = f;
      if (!((double)f == x)) /* NaN, overflow to infinity and lost bits all count as inexact */
        exact = false;
    }
  return exact;
}

/* four vertices = 20 doubles = five vectors, every lane checked */
__attribute__((target("avx2"))) bool narrow_avx2(const double *src, float *dst, size_t n_vertices)
{
  __m256d bad = _mm256_setzero_pd();
  const size_t groups = n_vertices / 4;
  for (size_t g = 0; g < groups; g++)
  {
    const double *s = src + 20 * g;
    float *d = dst + 20 * g;
#define RTB_NARROW4(K)                                                             \
  {                                                                                \
    const __m256d x = _mm256_loadu_pd(s + 4 * (K));                                \
    const __m128 f = _mm256_cvtpd_ps(x);                                           \
    _mm_storeu_ps(d + 4 * (K), f);                                                 \
    bad = _mm256_or_pd(bad, _mm256_cmp_pd(_mm256_cvtps_pd(f), x, _CMP_NEQ_UQ));    \
  }
    RTB_NARROW4(0)
    RTB_NARROW4(1)
    RTB_NARROW4(2)
    RTB_NARROW4(3)
    RTB_NARROW4(4)
#undef RTB_NARROW4
  }
  bool exact = _mm256_movemask_pd(bad) == 0;
  const size_t done = 4 * groups;
  if (done < n_vertices)
    exact = narrow_scalar(src + 5 * done, dst + 5 * done, n_vertices - done) && exact;
  return exact;
}
} // namespace

/* n_vertices records of five doubles -> five floats each; returns true when every double is float-representable.
 * C linkage so that the CPU test can reach it (internal: declared in rtb_internal.h, not in include/rtb200.h). */
extern "C" bool rtb_narrow_vertices(const double *src, float *dst, size_t n_vertices)
{
  static const bool have_avx2 = __builtin_cpu_supports("avx2");
  return have_avx2 ? narrow_avx2(src, dst, n_vertices) : narrow_scalar(src, dst, n_vertices);
}

/* the scalar form, for the test that compares the two */
extern "C" bool rtb_narrow_vertices_scalar(const double *src, float *dst, size_t n_vertices)
{
  return narrow_scalar(src, dst, n_vertices);
}
