// C++ adapters with the reference's own signatures (bm5d.h:11-62, bm3d_LF.h:10-35) over the C ABI of
// include/lfbm5d_cuda.h. A program written against the reference's headers links against liblfbm5d_host.so instead
// of bm5d.cpp / bm5d_core_processing.cpp / bm3d*.cpp and keeps calling the same functions.
#pragma once
#include <vector>

// the reference's #defines (main.cpp:20-32)
#ifndef YUV
#define YUV 0
#define YCBCR 1
#define OPP 2
#define RGB 3
#define ID 4
#define DCT 5
#define SADCT 6
#define BIOR 7
#define HADAMARD 8
#define HAAR 9
#define NONE 10
#define ROWMAJOR 11
#define COLMAJOR 12
#endif

//! Hard thresholding step (bm5d.h:11-35)
int run_bm5d_1st_step(const float sigma, const float lambdaHard5D, std::vector<std::vector<float> > &LF_noisy,
                      std::vector<unsigned> &LF_SAI_mask, std::vector<std::vector<float> > &LF_basic, const unsigned ang_major,
                      const unsigned awidth, const unsigned aheight, const unsigned anHard, const unsigned width,
                      const unsigned height, const unsigned chnls, const unsigned NHard, const unsigned nSim, const unsigned nDisp,
                      const unsigned kHard, const unsigned pHard, const bool useSD, const unsigned tau_2D, unsigned tau_4D,
                      const unsigned tau_5D, const unsigned color_space, const unsigned nb_threads);

//! Wiener filtering step (bm5d.h:38-62)
int run_bm5d_2nd_step(const float sigma, std::vector<std::vector<float> > &LF_noisy, std::vector<unsigned> &LF_SAI_mask,
                      std::vector<std::vector<float> > &LF_basic, std::vector<std::vector<float> > &LF_denoised,
                      const unsigned ang_major, const unsigned awidth, const unsigned aheight, const unsigned anWien,
                      const unsigned width, const unsigned height, const unsigned chnls, const unsigned NWien, const unsigned nSim,
                      const unsigned nDisp, const unsigned kWien, const unsigned pWien, const bool useSD, const unsigned tau_2D,
                      unsigned tau_4D, const unsigned tau_5D, const unsigned color_space, const unsigned nb_threads);

//! BM3D on every SAI (bm3d_LF.h:10-35)
int run_bm3d_LF(const float sigma, std::vector<std::vector<float> > &LF_noisy, std::vector<unsigned> &LF_SAI_mask,
                std::vector<std::vector<float> > &LF_basic, std::vector<std::vector<float> > &LF_denoised, const unsigned width,
                const unsigned height, const unsigned chnls, const unsigned nHard, const unsigned nWien, const unsigned kHard,
                const unsigned kWien, const unsigned NHard, const unsigned NWien, const unsigned pHard, const unsigned pWien,
                const bool useSD_h, const bool useSD_w, const unsigned tau_2D_hard, const unsigned tau_2D_wien,
                const float lambdaHard3D, const unsigned color_space, const unsigned nb_threads, char *sub_img_name);

//! Noise level of a light field without ground truth (lfbm5d_estimate_sigma, include/lfbm5d_cuda.h; not in the reference): LF[st] of
//! width*height*chnls floats (planar, as given: RGB or grey), SAIs with mask[st] == 0 ignored. *sigma pools every SAI and channel;
//! sigma_chnl / sigma_sai, when given, receive the value per channel and per SAI (0 for masked SAIs). The input is not modified.
int estimate_sigma_LF(const std::vector<std::vector<float> > &LF, const std::vector<unsigned> &mask, unsigned width, unsigned height,
                      unsigned chnls, float *sigma, std::vector<float> *sigma_chnl = nullptr, std::vector<float> *sigma_sai = nullptr);
