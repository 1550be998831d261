// See lfbm5d_host.h. Error behaviour follows the reference's drivers: message on cout, EXIT_FAILURE (1).
#include "lfbm5d_host.h"
#include "lfbm5d_cuda.h"
#include "lfbm5d_host_c.h"
#include "lf_io.h"
#include <cstdlib>
#include <iostream>

namespace {
lfbm5d_ctx *context()
{
    static lfbm5d_ctx *ctx = nullptr;
    if (!ctx) {
        const char *dev = getenv("LFBM5D_DEVICE");
        if (lfbm5d_create(&ctx, dev ? atoi(dev) : 0) != 0) {
            std::cout << "lfbm5d: " << lfbm5d_last_error() << std::endl;
            ctx = nullptr;
        }
    }
    return ctx;
}
std::vector<float *> pointers(std::vector<std::vector<float> > &LF, const std::vector<unsigned> &mask, size_t each, bool resize)
{
    std::vector<float *> p(LF.size(), nullptr);
    for (size_t st = 0; st < LF.size(); st++) {
        if (st < mask.size() && mask[st]) {
            if (resize && LF[st].size() != each) LF[st].resize(each);
            p[st] = LF[st].data();
        }
    }
    return p;
}
int check_sizes(const std::vector<std::vector<float> > &LF, const std::vector<unsigned> &mask, unsigned asize, size_t each, const char *what)
{
    if (LF.size() != asize || mask.size() != asize) {
        std::cout << what << " should have awidth*aheight sub-aperture images." << std::endl;
        return 1;
    }
    for (unsigned st = 0; st < asize; st++)
        if (mask[st] && LF[st].size() != each) {
            std::cout << what << ": SAI " << st << " does not have width*height*chnls samples." << std::endl;
            return 1;
        }
    return 0;
}
} // namespace

int run_bm5d_1st_step(const float sigma, const float lambdaHard5D, std::vector<std::vector<float> > &LF_noisy,
                      std::vector<unsigned> &LF_SAI_mask, std::vector<std::vector<float> > &LF_basic, const unsigned ang_major,
                      const unsigned awidth, const unsigned aheight, const unsigned anHard, const unsigned width,
                      const unsigned height, const unsigned chnls, const unsigned NHard, const unsigned nSim, const unsigned nDisp,
                      const unsigned kHard, const unsigned pHard, const bool useSD, const unsigned tau_2D, unsigned tau_4D,
                      const unsigned tau_5D, const unsigned color_space, const unsigned nb_threads)
{
    lfbm5d_ctx *ctx = context();
    if (!ctx) return EXIT_FAILURE;
    const unsigned asize = awidth * aheight;
    const size_t each = (size_t) width * height * chnls;
    if (LF_basic.size() != asize) LF_basic.resize(asize);      // bm5d.cpp:129-130
    if (check_sizes(LF_noisy, LF_SAI_mask, asize, each, "LF_noisy")) return EXIT_FAILURE;
    lfbm5d_params p = { sigma, lambdaHard5D, ang_major, awidth, aheight, anHard, width, height, chnls, NHard, nSim, nDisp, kHard, pHard,
                        useSD ? 1u : 0u, tau_2D, tau_4D, tau_5D, color_space, nb_threads };
    std::vector<float *> n = pointers(LF_noisy, LF_SAI_mask, each, false), b = pointers(LF_basic, LF_SAI_mask, each, true);
    if (lfbm5d_step1(ctx, &p, n.data(), LF_SAI_mask.data(), b.data()) != 0) {
        std::cout << lfbm5d_last_error() << std::endl;
        return EXIT_FAILURE;
    }
    return EXIT_SUCCESS;
}

int run_bm5d_2nd_step(const float sigma, std::vector<std::vector<float> > &LF_noisy, std::vector<unsigned> &LF_SAI_mask,
                      std::vector<std::vector<float> > &LF_basic, std::vector<std::vector<float> > &LF_denoised,
                      const unsigned ang_major, const unsigned awidth, const unsigned aheight, const unsigned anWien,
                      const unsigned width, const unsigned height, const unsigned chnls, const unsigned NWien, const unsigned nSim,
                      const unsigned nDisp, const unsigned kWien, const unsigned pWien, const bool useSD, const unsigned tau_2D,
                      unsigned tau_4D, const unsigned tau_5D, const unsigned color_space, const unsigned nb_threads)
{
    lfbm5d_ctx *ctx = context();
    if (!ctx) return EXIT_FAILURE;
    const unsigned asize = awidth * aheight;
    const size_t each = (size_t) width * height * chnls;
    if (LF_denoised.size() != asize) LF_denoised.resize(asize);   // bm5d.cpp:823-824
    if (check_sizes(LF_noisy, LF_SAI_mask, asize, each, "LF_noisy") || check_sizes(LF_basic, LF_SAI_mask, asize, each, "LF_basic"))
        return EXIT_FAILURE;
    lfbm5d_params p = { sigma, 0.0f, ang_major, awidth, aheight, anWien, width, height, chnls, NWien, nSim, nDisp, kWien, pWien,
                        useSD ? 1u : 0u, tau_2D, tau_4D, tau_5D, color_space, nb_threads };
    std::vector<float *> n = pointers(LF_noisy, LF_SAI_mask, each, false), b = pointers(LF_basic, LF_SAI_mask, each, false),
                         d = pointers(LF_denoised, LF_SAI_mask, each, true);
    if (lfbm5d_step2(ctx, &p, n.data(), b.data(), LF_SAI_mask.data(), d.data()) != 0) {
        std::cout << lfbm5d_last_error() << std::endl;
        return EXIT_FAILURE;
    }
    return EXIT_SUCCESS;
}

int run_bm3d_LF(const float sigma, std::vector<std::vector<float> > &LF_noisy, std::vector<unsigned> &LF_SAI_mask,
                std::vector<std::vector<float> > &LF_basic, std::vector<std::vector<float> > &LF_denoised, const unsigned width,
                const unsigned height, const unsigned chnls, const unsigned nHard, const unsigned nWien, const unsigned kHard,
                const unsigned kWien, const unsigned NHard, const unsigned NWien, const unsigned pHard, const unsigned pWien,
                const bool useSD_h, const bool useSD_w, const unsigned tau_2D_hard, const unsigned tau_2D_wien,
                const float lambdaHard3D, const unsigned color_space, const unsigned nb_threads, char *sub_img_name)
{
    (void) sub_img_name;
    lfbm5d_ctx *ctx = context();
    if (!ctx) return EXIT_FAILURE;
    const unsigned asize = (unsigned) LF_noisy.size();
    const size_t each = (size_t) width * height * chnls;
    if (LF_basic.size() != asize) LF_basic.resize(asize);         // bm3d_LF.cpp:98-101
    if (LF_denoised.size() != asize) LF_denoised.resize(asize);
    if (check_sizes(LF_noisy, LF_SAI_mask, asize, each, "LF_noisy")) return EXIT_FAILURE;
    lfbm3d_params p = { sigma, asize, width, height, chnls, nHard, nWien, kHard, kWien, NHard, NWien, pHard, pWien,
                        useSD_h ? 1u : 0u, useSD_w ? 1u : 0u, tau_2D_hard, tau_2D_wien, lambdaHard3D, color_space, nb_threads };
    std::vector<float *> n = pointers(LF_noisy, LF_SAI_mask, each, false), b = pointers(LF_basic, LF_SAI_mask, each, true),
                         d = pointers(LF_denoised, LF_SAI_mask, each, true);
    if (lfbm3d_run(ctx, &p, n.data(), LF_SAI_mask.data(), b.data(), d.data()) != 0) {
        std::cout << lfbm5d_last_error() << std::endl;
        return EXIT_FAILURE;
    }
    return EXIT_SUCCESS;
}

int estimate_sigma_LF(const std::vector<std::vector<float> > &LF, const std::vector<unsigned> &mask, unsigned width, unsigned height,
                      unsigned chnls, float *sigma, std::vector<float> *sigma_chnl, std::vector<float> *sigma_sai)
{
    lfbm5d_ctx *ctx = context();
    if (!ctx) return EXIT_FAILURE;
    const unsigned asize = (unsigned) LF.size();
    const size_t each = (size_t) width * height * chnls;
    if (check_sizes(LF, mask, asize, each, "LF")) return EXIT_FAILURE;
    std::vector<float *> p(asize, nullptr);      // read only: the C ABI takes the pointer type of the step entry points
    for (unsigned st = 0; st < asize; st++) if (mask[st]) p[st] = const_cast<float *>(LF[st].data());
    std::vector<float> sc(chnls), ss(asize);
    if (lfbm5d_estimate_sigma(ctx, p.data(), mask.data(), asize, chnls, width, height, sigma, sc.data(), ss.data()) != 0) {
        std::cout << lfbm5d_last_error() << std::endl;
        return EXIT_FAILURE;
    }
    if (sigma_chnl) *sigma_chnl = sc;
    if (sigma_sai) *sigma_sai = ss;
    return EXIT_SUCCESS;
}

// ---- C exports of the host-side noise / metric helpers of the command lines (include/lfbm5d_host_c.h) ----
extern "C" {

void lfio_add_noise(const float *img, float *out, size_t n, float sigma, unsigned long seed)
{
    lfio::MT g;
    g.seed(seed);
    for (size_t k = 0; k < n; k++) {      // utilities.cpp:177-184
        const double a = g.res53(), b = g.res53();
        const double z = (double) sigma * sqrt(-2.0 * log(a)) * cos(2.0 * M_PI * b);
        out[k] = img[k] + (float) z;
    }
}

void lfio_psnr(const float *a, const float *b, size_t n, float *psnr, float *rmse)
{
    float tmp = 0.0f;      // utilities.cpp:427-432: float accumulator
    for (size_t k = 0; k < n; k++) tmp += (a[k] - b[k]) * (a[k] - b[k]);
    *rmse = sqrtf(tmp / (float) n);
    *psnr = 20.0f * log10f(255.0f / (*rmse));
}

// ---- the file formats and the report of the command lines, for callers / tests without a C++ toolchain ----
int lfio_png_read(const char *name, float *out, size_t capacity, size_t *w, size_t *h, size_t *c)
{
    std::vector<float> v;
    size_t ww = 0, hh = 0, cc = 0;
    if (!name || !w || !h || !c || !lfio::read_png_f32(name, v, ww, hh, cc)) return 1;
    *w = ww; *h = hh; *c = cc;
    if (out) { if (capacity < v.size()) return 1; memcpy(out, v.data(), v.size() * sizeof(float)); }
    return 0;
}

int lfio_png_write(const char *name, const float *data, size_t w, size_t h, size_t c)
{
    return name && data && lfio::write_png_f32(name, data, w, h, c) ? 0 : 1;
}

// load_LF / save_LF (utilities_LF.cpp:72-231) on a light field stored as [asize][c*W*H] floats (st ordered per ang_major). With
// out == NULL lfio_load_LF only reports the size of the first image and the mask.
int lfio_load_LF(const char *dir, const char *sub, const char *sep, unsigned ang_major, unsigned awidth, unsigned aheight, unsigned s_start,
                 unsigned t_start, float *out, size_t capacity, unsigned *mask, unsigned *width, unsigned *height, unsigned *chnls)
{
    std::vector<std::vector<float> > LF;
    std::vector<unsigned> m;
    if (lfio::load_LF(dir, sub, sep, LF, m, ang_major, awidth, aheight, s_start, t_start, width, height, chnls, LFBM5D_ROWMAJOR) != EXIT_SUCCESS) return 1;
    const size_t each = (size_t) *width * *height * *chnls;
    if (mask) memcpy(mask, m.data(), m.size() * sizeof(unsigned));
    if (out) {
        if (capacity < each * LF.size()) return 1;
        for (size_t st = 0; st < LF.size(); st++) {
            if (LF[st].size() != each) return 1;       // every image must have the size of the first one
            memcpy(out + st * each, LF[st].data(), each * sizeof(float));
        }
    }
    return 0;
}

static std::vector<std::vector<float> > lf_of(const float *a, unsigned asize, size_t each);

int lfio_save_LF(const char *dir, const char *sub, const char *sep, const float *lf, const unsigned *mask, unsigned ang_major, unsigned awidth,
                 unsigned aheight, unsigned s_start, unsigned t_start, unsigned width, unsigned height, unsigned chnls)
{
    const unsigned asize = awidth * aheight;
    return lfio::save_LF(dir, sub, sep, lf_of(lf, asize, (size_t) width * height * chnls), std::vector<unsigned>(mask, mask + asize), ang_major, awidth, aheight,
                         s_start, t_start, width, height, chnls, LFBM5D_ROWMAJOR) == EXIT_SUCCESS ? 0 : 1;
}

static std::vector<std::vector<float> > lf_of(const float *a, unsigned asize, size_t each)
{
    std::vector<std::vector<float> > v(asize);
    for (unsigned st = 0; st < asize; st++) v[st].assign(a + (size_t) st * each, a + (size_t) (st + 1) * each);
    return v;
}

int lfio_psnr_LF(const float *lf1, const float *lf2, const unsigned *mask, unsigned asize, size_t each, float *psnr, float *rmse, float *stats4)
{
    const std::vector<unsigned> m(mask, mask + asize);
    std::vector<float> ps, rm;
    if (lfio::compute_psnr_LF(lf_of(lf1, asize, each), lf_of(lf2, asize, each), m, ps, &stats4[0], &stats4[1], rm, &stats4[2], &stats4[3]) != EXIT_SUCCESS) return 1;
    memcpy(psnr, ps.data(), asize * sizeof(float));
    memcpy(rmse, rm.data(), asize * sizeof(float));
    return 0;
}

int lfio_diff_LF(const float *lf1, const float *lf2, const unsigned *mask, unsigned asize, size_t each, float sigma, float *diff)
{
    const std::vector<unsigned> m(mask, mask + asize);
    std::vector<std::vector<float> > d;
    lfio::compute_diff_LF(lf_of(lf1, asize, each), lf_of(lf2, asize, each), m, d, sigma);
    for (unsigned st = 0; st < asize; st++) if (m[st]) memcpy(diff + (size_t) st * each, d[st].data(), each * sizeof(float));
    return 0;
}

int lfio_write_psnr_LF(const char *file_name, const char *LF_name, const unsigned *mask, unsigned ang_major, unsigned awidth, unsigned aheight,
                       const float *psnr, float avg_psnr, float std_psnr, const float *rmse, float avg_rmse, float std_rmse)
{
    const unsigned asize = awidth * aheight;
    return lfio::write_psnr_LF(file_name, LF_name, std::vector<unsigned>(mask, mask + asize), ang_major, awidth, aheight, std::vector<float>(psnr, psnr + asize),
                               avg_psnr, std_psnr, std::vector<float>(rmse, rmse + asize), avg_rmse, std_rmse, LFBM5D_ROWMAJOR) == EXIT_SUCCESS ? 0 : 1;
}

} // extern "C"
