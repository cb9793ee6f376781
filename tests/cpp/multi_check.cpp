// tests/cpp/multi_check.cpp -- drives visfd_cuda_membrane_multi the way a C++ host (filter_mrc) would: plain host
// arrays, a list of CUDA devices, one call.  The result must equal visfd_cuda_membrane on one GPU BIT FOR BIT
// (thresholds included) for every split.  Usage: multi_check [ndev]   (default: all visible devices; with one
// visible device the same device is listed several times, which exercises the slab logic all the same).  Two calls
// made at once must both give that result, and a call that fails must return its error instead of blocking.
// Exit code 0 = all checks passed.  Run by tests/test_gpu_multi.py.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <random>
#include <string>
#include <thread>
#include <vector>
#include "../../include/visfd_cuda.h"

static std::vector<float> volume(int nx, int ny, int nz, unsigned seed) {
  std::mt19937 g(seed);
  std::normal_distribution<float> noise(0.0f, 1.0f);
  std::vector<float> v((size_t)nx * ny * nz);
  const float cx = 0.5f * nx, cy = 0.5f * ny, cz = 0.5f * nz, R = 0.3f * std::min(nx, std::min(ny, nz));
  for (int z = 0; z < nz; z++)
    for (int y = 0; y < ny; y++)
      for (int x = 0; x < nx; x++) {
        const float r = std::sqrt((x - cx) * (x - cx) + (y - cy) * (y - cy) + (z - cz) * (z - cz));
        v[((size_t)z * ny + y) * nx + x] = noise(g) - 3.0f * std::exp(-0.5f * (r - R) * (r - R) / 4.0f);
      }
  return v;
}

static size_t count_differing(const std::vector<float> &a, const std::vector<float> &b) {
  size_t diff = 0;
  for (size_t i = 0; i < a.size(); i++) diff += std::memcmp(&a[i], &b[i], sizeof(float)) != 0;
  return diff;
}

// rc: the return code of a call that must fail with an error containing `cause`
static int expect_error(const char *what, int rc, const char *cause) {
  const bool ok = rc != 0 && std::strstr(visfd_cuda_last_error(), cause) != nullptr;
  std::printf("%s %s: %s\n", ok ? "ok  " : "FAIL", what, rc ? visfd_cuda_last_error() : "no error");
  return ok ? 0 : 1;
}

int main(int argc, char **argv) {
  const int visible = visfd_cuda_device_count();
  if (visible < 1) { std::printf("no CUDA device\n"); return 2; }
  const int want = argc > 1 ? std::atoi(argv[1]) : 0;
  int failures = 0;
  visfd_ctx *ctx = nullptr;
  if (visfd_cuda_init(0, &ctx) != 0) { std::printf("init: %s\n", visfd_cuda_last_error()); return 2; }
  struct Case { int nx, ny, nz; float sigma, tv_sigma, cut; int fraction; bool mask; };
  const Case cases[] = {{48, 40, 72, 1.5f, 4.3f, 0.08f, 1, false},    // 9 units of 8 planes
                        {40, 36, 61, 1.2f, 3.1f, 0.10f, 1, true},     // ragged tail, mask
                        {64, 48, 96, 2.0f, 6.0f, 0.05f, 1, false},    // halo wider than a slab at 8 workers
                        {32, 32, 40, 1.0f, 0.0f, 0.20f, 1, false},    // no voting: saliency after the cut
                        {40, 40, 48, 1.5f, 4.0f, 0.002f, 0, false},   // absolute threshold
                        {40, 36, 61, 1.2f, 3.1f, 1.0f, 1, true}};     // rank clamped to the last un-masked voxel
  for (const Case &c : cases) {
    const size_t N = (size_t)c.nx * c.ny * c.nz;
    std::vector<float> src = volume(c.nx, c.ny, c.nz, 11u + (unsigned)c.nz), mask, one(N), multi(N);
    if (c.mask) {
      mask.assign(N, 1.0f);
      for (int z = 0; z < c.nz; z++)
        for (int y = 0; y < c.ny; y++)
          for (int x = 0; x < c.nx; x++)
            if (x < 3 || y > c.ny - 5 || (z % 17) == 0) mask[((size_t)z * c.ny + y) * c.nx + x] = 0.0f;
    }
    visfd_membrane_params p;
    p.sigma = c.sigma; p.truncate_ratio = 2.6482f; p.eival_order = VISFD_DECREASING_EIVALS;
    p.cut = c.cut; p.cut_is_fraction = c.fraction;
    p.tv_sigma = c.tv_sigma; p.tv_exponent = 4; p.tv_cutoff_ratio = 1.41421354f;
    float thr1 = 0;
    if (visfd_cuda_membrane(ctx, c.nx, c.ny, c.nz, src.data(), c.mask ? mask.data() : nullptr, &p, one.data(), nullptr,
                            nullptr, nullptr, &thr1) != 0) {
      std::printf("one GPU: %s\n", visfd_cuda_last_error());
      return 2;
    }
    for (int ndev : {1, 2, 3, 4, 8}) {
      if (want && ndev != want && ndev != 1) continue;
      std::vector<int> devs((size_t)ndev);
      for (int r = 0; r < ndev; r++) devs[(size_t)r] = r % visible;
      std::fill(multi.begin(), multi.end(), -7.0f);
      float thrn = 0;
      std::vector<double> ms((size_t)ndev);
      if (visfd_cuda_membrane_multi(ndev, devs.data(), c.nx, c.ny, c.nz, src.data(), c.mask ? mask.data() : nullptr, &p,
                                    multi.data(), &thrn, ms.data()) != 0) {
        std::printf("FAIL %dx%dx%d ndev %d: %s\n", c.nx, c.ny, c.nz, ndev, visfd_cuda_last_error());
        failures++;
        continue;
      }
      const size_t diff = count_differing(one, multi);
      const bool ok = diff == 0 && std::memcmp(&thr1, &thrn, sizeof(float)) == 0;
      std::printf("%s %dx%dx%d%s tv %.1f: %d worker(s) on %d device(s): %zu voxels differ, threshold %.9g vs %.9g\n",
                  ok ? "ok  " : "FAIL", c.nx, c.ny, c.nz, c.mask ? " masked" : "", c.tv_sigma, ndev, std::min(ndev, visible), diff,
                  thrn, thr1);
      failures += !ok;
    }
    // two calls at once, every device listed twice: both results equal the one-GPU result
    {
      std::vector<int> devs((size_t)(2 * visible));
      for (int r = 0; r < 2 * visible; r++) devs[(size_t)r] = r % visible;
      std::vector<float> a(N, -7.0f), b(N, -7.0f);
      float thra = 0, thrb = 0;
      int rca = 1, rcb = 1;
      std::string erra, errb;
      auto call = [&](std::vector<float> &out, float &thr, int &rc, std::string &err) {
        rc = visfd_cuda_membrane_multi(2 * visible, devs.data(), c.nx, c.ny, c.nz, src.data(),
                                       c.mask ? mask.data() : nullptr, &p, out.data(), &thr, nullptr);
        if (rc != 0) err = visfd_cuda_last_error();
      };
      std::thread other(call, std::ref(a), std::ref(thra), std::ref(rca), std::ref(erra));
      call(b, thrb, rcb, errb);
      other.join();
      const size_t da = count_differing(one, a), db = count_differing(one, b);
      const bool ok = rca == 0 && rcb == 0 && da == 0 && db == 0 && std::memcmp(&thr1, &thra, sizeof(float)) == 0 &&
                      std::memcmp(&thr1, &thrb, sizeof(float)) == 0;
      std::printf("%s %dx%dx%d%s tv %.1f: two calls at once on %d slot(s): %zu and %zu voxels differ%s%s%s%s\n",
                  ok ? "ok  " : "FAIL", c.nx, c.ny, c.nz, c.mask ? " masked" : "", c.tv_sigma, 2 * visible, da, db,
                  erra.empty() ? "" : "; ", erra.c_str(), errb.empty() ? "" : "; ", errb.c_str());
      failures += !ok;
    }
  }
  // error paths: the call returns with the cause
  {
    const int nx = 16, ny = 16, nz = 32;
    std::vector<float> src = volume(nx, ny, nz, 3), zero((size_t)nx * ny * nz, 0.0f), out((size_t)nx * ny * nz);
    visfd_membrane_params p = {1.0f, 2.6482f, 1, 0.1f, 1, 2.0f, 4, 1.41421354f};
    const int bad[2] = {0, 1000}, two[2] = {0, 1 % visible};
    failures += expect_error("device 1000 refused",
                             visfd_cuda_membrane_multi(2, bad, nx, ny, nz, src.data(), nullptr, &p, out.data(), nullptr,
                                                       nullptr),
                             "device index out of range");
    // the cut fails on the calling thread, between two phases
    failures += expect_error("all-zero mask",
                             visfd_cuda_membrane_multi(2, two, nx, ny, nz, src.data(), zero.data(), &p, out.data(),
                                                       nullptr, nullptr),
                             "no un-masked voxels");
    // half-width floor(50 * sqrt(2)) = 70 > 56: the vote fails on the thread of every slab
    p.tv_sigma = 50.0f;
    failures += expect_error("voting radius 70",
                             visfd_cuda_membrane_multi(2, two, nx, ny, nz, src.data(), nullptr, &p, out.data(), nullptr,
                                                       nullptr),
                             "slab 0 on device 0: visfd_cuda: tensor-voting radius too large");
  }
  visfd_cuda_destroy(ctx);
  std::printf("%s (%d failures)\n", failures ? "FAILED" : "OK", failures);
  return failures ? 1 : 0;
}
