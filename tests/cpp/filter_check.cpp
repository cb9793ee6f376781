// tests/cpp/filter_check.cpp -- the shim's ApplyGauss / ApplyDog / ApplyLog (visfd_cuda_shim.hpp), which run through
// visfd_cuda_filter_stream, called with the reference's and filter_mrc's overloads on float*** tables: contiguous
// (Alloc3D layout), non-contiguous, and with aaafDest == aaafSource.  Every result and peak height must equal the
// one-shot C call (visfd_cuda_apply_gauss / _dog2 / _log) bit for bit.
// Exit code 0 = all checks passed.  Built and run by tests/test_gpu_filter_shim.py.
#include <cstdio>
#include <cstring>
#include <functional>
#include <random>
#include <string>
#include <vector>
#include "../../visfd_b200/csrc/visfd_cuda_shim.hpp"

// pointer tables over a flat buffer; `gap` > 0 makes rows non-contiguous
struct Image3 {
  int nx, ny, nz;
  size_t pitch;
  std::vector<float> data;
  std::vector<float *> rows;
  std::vector<float **> planes;
  Image3(int nx_, int ny_, int nz_, int gap) : nx(nx_), ny(ny_), nz(nz_), pitch(nx_ + gap) {
    data.assign(pitch * ny * nz, 0.0f);
    rows.resize((size_t)ny * nz);
    planes.resize(nz);
    for (int z = 0; z < nz; z++) {
      for (int y = 0; y < ny; y++) rows[(size_t)z * ny + y] = data.data() + ((size_t)z * ny + y) * pitch;
      planes[z] = rows.data() + (size_t)z * ny;
    }
  }
  float ***p() { return planes.data(); }
  void load(const std::vector<float> &f) {
    for (size_t r = 0; r < rows.size(); r++) std::copy(&f[r * nx], &f[r * nx] + nx, rows[r]);
  }
  std::vector<float> flat() const {
    std::vector<float> f((size_t)nx * ny * nz);
    for (size_t r = 0; r < rows.size(); r++) std::copy(rows[r], rows[r] + nx, f.begin() + r * nx);
    return f;
  }
};

static int failures = 0;
static void check(bool ok, const std::string &what) {
  std::printf("%s  %s\n", ok ? "PASS" : "FAIL", what.c_str());
  if (!ok) failures++;
}
static bool same_bits(const std::vector<float> &a, const std::vector<float> &b) {
  return a.size() == b.size() && std::memcmp(a.data(), b.data(), a.size() * sizeof(float)) == 0;
}
static bool same_bits(float a, float b) { return std::memcmp(&a, &b, sizeof(float)) == 0; }

int main() {
  const int nx = 42, ny = 36, nz = 51;   // nx % 4 != 0: the fall-back X sweeps
  const int size[3] = {nx, ny, nz};
  const size_t N = (size_t)nx * ny * nz;
  std::mt19937 rng(11);
  std::normal_distribution<float> noise(0.f, 1.f);
  std::vector<float> vol(N), cell(N);
  for (auto &v : vol) v = noise(rng);
  for (int z = 0; z < nz; z++)
    for (int y = 0; y < ny; y++)
      for (int x = 0; x < nx; x++) {
        const float u = (x - nx / 2.f) / (0.45f * nx), v = (y - ny / 2.f) / (0.48f * ny), w = (z - nz / 2.f) / (0.45f * nz);
        cell[((size_t)z * ny + y) * nx + x] = u * u + v * v + w * w <= 1.f ? 1.f : 0.f;
      }
  visfd_ctx *ctx = visfd_cuda::Context();
  const float ratio = 2.5f, thresh = 0.03f;

  // (shim call on (src, dst, mask) tables -> A, B) and the one-shot C call on flat arrays
  struct Case {
    std::string name;
    std::function<void(float ***, float ***, float ***, float *, float *)> shim;
    std::function<int(const float *, float *, const float *, float *, float *)> one_shot;
  };
  const float s1[3] = {1.5f, 1.5f, 1.5f}, s2[3] = {2.4f, 2.4f, 2.4f}, saniso[3] = {1.0f, 2.0f, 3.0f};
  const int hw1[3] = {4, 4, 4}, hwaniso[3] = {3, 5, 7};
  auto hw_of = [&](const float *s, int *hw) {
    for (int d = 0; d < 3; d++) hw[d] = visfd_cuda_gauss_halfwidth(s[d], ratio, thresh);
  };
  std::vector<Case> cases = {
      {"ApplyGauss(sigma[3], hw[3], normalize)",
       [&](float ***s, float ***d, float ***m, float *A, float *) {
         *A = visfd_cuda::ApplyGauss(size, s, d, m, saniso, hwaniso, true);
       },
       [&](const float *s, float *d, const float *m, float *A, float *) {
         return visfd_cuda_apply_gauss(ctx, nx, ny, nz, s, d, m, saniso, hwaniso, 1, A);
       }},
      {"ApplyGauss(sigma, hw, normalize = false)",
       [&](float ***s, float ***d, float ***m, float *A, float *) {
         *A = visfd_cuda::ApplyGauss(size, s, d, m, 2.0f, 5, false);
       },
       [&](const float *s, float *d, const float *m, float *A, float *) {
         const float sg[3] = {2.0f, 2.0f, 2.0f};
         const int hw[3] = {5, 5, 5};
         return visfd_cuda_apply_gauss(ctx, nx, ny, nz, s, d, m, sg, hw, 0, A);
       }},
      {"filter_mrc ApplyGauss(sigma[3], ratio, threshold, normalize, &cerr)",
       [&](float ***s, float ***d, float ***m, float *A, float *) {
         *A = visfd_cuda::ApplyGauss(size, s, d, m, s2, ratio, thresh, true, nullptr);
       },
       [&](const float *s, float *d, const float *m, float *A, float *) {
         int hw[3];
         hw_of(s2, hw);
         return visfd_cuda_apply_gauss(ctx, nx, ny, nz, s, d, m, s2, hw, 1, A);
       }},
      {"ApplyDog(sigma_a, sigma_b, hw[3], &A, &B)",
       [&](float ***s, float ***d, float ***m, float *A, float *B) {
         visfd_cuda::ApplyDog(size, s, d, m, s1, s2, hw1, A, B);
       },
       [&](const float *s, float *d, const float *m, float *A, float *B) {
         return visfd_cuda_apply_dog(ctx, nx, ny, nz, s, d, m, s1, s2, hw1, A, B);
       }},
      {"filter_mrc ApplyDog(sigma_a, sigma_b, ratio, threshold, &A, &B, &cerr)",
       [&](float ***s, float ***d, float ***m, float *A, float *B) {
         visfd_cuda::ApplyDog(size, s, d, m, s1, s2, ratio, thresh, A, B, nullptr);
       },
       [&](const float *s, float *d, const float *m, float *A, float *B) {
         int hwa[3], hwb[3];
         hw_of(s1, hwa);
         hw_of(s2, hwb);
         return visfd_cuda_apply_dog2(ctx, nx, ny, nz, s, d, m, s1, s2, hwa, hwb, A, B);
       }},
      {"ApplyLog(sigma, delta, ratio, &A, &B)",
       [&](float ***s, float ***d, float ***m, float *A, float *B) {
         visfd_cuda::ApplyLog(size, s, d, m, s2, 0.02f, ratio, A, B);
       },
       [&](const float *s, float *d, const float *m, float *A, float *B) {
         return visfd_cuda_apply_log(ctx, nx, ny, nz, s, d, m, s2, 0.02f, ratio, A, B);
       }},
      {"filter_mrc ApplyLog(sigma, delta, ratio = -1, threshold, &A, &B, &cerr)",
       [&](float ***s, float ***d, float ***m, float *A, float *B) {
         visfd_cuda::ApplyLog(size, s, d, m, s1, 0.02f, -1.0f, thresh, A, B, nullptr);
       },
       [&](const float *s, float *d, const float *m, float *A, float *B) {
         return visfd_cuda_apply_log(ctx, nx, ny, nz, s, d, m, s1, 0.02f, std::sqrt(-2 * std::log(thresh)), A, B);
       }},
  };

  for (const Case &c : cases)
    for (bool masked : {false, true}) {
      std::vector<float> want(N);
      float wA = 0, wB = 0;
      if (c.one_shot(vol.data(), want.data(), masked ? cell.data() : nullptr, &wA, &wB) != 0) {
        check(false, c.name + ": one-shot call: " + visfd_cuda_last_error());
        continue;
      }
      for (int gap : {0, 3}) {
        for (bool in_place : {false, true}) {
          Image3 src(nx, ny, nz, gap), dst(nx, ny, nz, gap), mask(nx, ny, nz, gap);
          src.load(vol);
          mask.load(cell);
          float A = 0, B = 0;
          const std::string what = c.name + (masked ? ", masked" : "") + (gap ? ", non-contiguous" : "") +
                                   (in_place ? ", aaafDest == aaafSource" : "");
          try {
            c.shim(src.p(), in_place ? src.p() : dst.p(), masked ? mask.p() : nullptr, &A, &B);
            check(same_bits((in_place ? src : dst).flat(), want) && same_bits(A, wA) && same_bits(B, wB), what);
          } catch (const std::exception &e) {
            check(false, what + ": " + e.what());
          }
        }
      }
    }
  std::printf("%s (%d failures)\n", failures ? "FAILED" : "OK", failures);
  return failures ? 1 : 0;
}
