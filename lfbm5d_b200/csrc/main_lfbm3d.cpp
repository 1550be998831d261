// LFBM3Ddenoising — BM3D on every sub-aperture image; same 31 positional arguments, messages and report as the
// reference's main_bm3d_LF.cpp:56-272 (argument grammar: utilities_LF.cpp:1342-1470, README.md:82).
#include "lfbm5d_host.h"
#include "lf_io.h"

using namespace std;

static unsigned pick(const char *a, std::initializer_list<std::pair<const char *, unsigned> > opts)
{
    for (auto &o : opts) if (strcmp(a, o.first) == 0) return o.second;
    return NONE;
}

int main(int argc, char **argv)
{
    cout << "*********************************************************************************************************************" << endl;
    cout << "********************************************              START               ***************************************" << endl;
    cout << "*********************************************************************************************************************" << endl;
    if (argc < 32) {      // (the reference tests argc < 27 and then reads 31 arguments)
        cout << "usage: LFBM3Ddenoising LF_dir SAI_name SAI_name_sep LF_awidth LF_aheight s_idx_start t_idx_start asw_size_ht asw_size_wien ang_major sigma lambda "
                "LF_dir_noisy LF_dir_basic LF_dir_denoised LF_dir_difference "
                "NHard nHard kHard pHard tau_2d_hard useSD_hard NWien nWien kWien pWien tau_2d_wien useSD_wien "
                "color_space nb_threads resultsFile" << endl;
        cout << "Problem while reading parameters from command line !" << endl;
        return EXIT_FAILURE;
    }
    unsigned i = 0;
    const char *LF_input_name = argv[++i];
    const char *sub_img_name = argv[++i]; if (strcmp(sub_img_name, "none") == 0) sub_img_name = "";
    const char *sep = argv[++i]; if (strcmp(sep, "none") == 0) sep = "";
    const bool gt_exists = strcmp(LF_input_name, "none") != 0;
    const unsigned awidth = atoi(argv[++i]), aheight = atoi(argv[++i]), s_start = atoi(argv[++i]), t_start = atoi(argv[++i]);
    i += 2;      // asw sizes: parsed and unused by the BM3D driver
    const unsigned ang_major = pick(argv[++i], { { "row", ROWMAJOR }, { "col", COLMAJOR } });
    if (ang_major == NONE) { cout << "ang_major is not known. Choice is :" << endl << " -row" << endl << " -col" << endl; return EXIT_FAILURE; }
    // sigma = auto: estimated from the noisy light field read back from disk (estimate_sigma_LF), so only without ground truth
    const bool sigma_auto = strcmp(argv[++i], "auto") == 0;
    float fSigma = sigma_auto ? 0.0f : atof(argv[i]);
    const float lambdaHard3D = atof(argv[++i]);
    if (sigma_auto && gt_exists) {
        cout << "sigma = auto needs LF_dir = none: with a ground-truth light field, noise of the given sigma is added to it. "
                "Give sigma as a number, or LF_dir = none to denoise the light field in LF_dir_noisy." << endl;
        return EXIT_FAILURE;
    }
    const char *LF_noisy_name = argv[++i], *LF_basic_name = argv[++i], *LF_denoised_name = argv[++i], *LF_diff_name = argv[++i];
    unsigned N[2], n[2], k[2], p[2], t2[2];
    bool useSD[2];
    for (int s = 0; s < 2; s++) {
        N[s] = atof(argv[++i]); n[s] = atof(argv[++i]); k[s] = atof(argv[++i]); p[s] = atof(argv[++i]);
        t2[s] = pick(argv[++i], { { "dct", DCT }, { "bior", BIOR } });
        if (t2[s] == NONE) { cout << "tau_2d_" << (s ? "wien" : "hard") << " is not known. Choice is :" << endl << " -dct" << endl << " -bior" << endl; return EXIT_FAILURE; }
        useSD[s] = (bool) atof(argv[++i]);
    }
    const unsigned color_space = pick(argv[++i], { { "rgb", RGB }, { "yuv", YUV }, { "ycbcr", YCBCR }, { "opp", OPP } });
    if (color_space == NONE) { cout << "color_space is not known. Choice is :" << endl << " -rgb" << endl << " -yuv" << endl << " -opp" << endl << " -ycbcr" << endl; return EXIT_FAILURE; }
    unsigned nb_threads = atof(argv[++i]);
    const char *psnr_file_name = argv[++i];
    if (!nb_threads) nb_threads = 1;

    vector<vector<float> > LF, LF_noisy, LF_basic, LF_denoised, LF_diff;
    vector<unsigned> LF_SAI_mask;
    unsigned width = 0, height = 0, chnls = 0;
    const unsigned awh = awidth * aheight;
    if (gt_exists) {
        double t0 = lfio::now();
        if (lfio::load_LF(LF_input_name, sub_img_name, sep, LF, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, &width, &height, &chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
        cout << "Loading LF elapsed time = " << float(lfio::now() - t0) << "s." << endl;
        LF_noisy.assign(awh, vector<float>());
        t0 = lfio::now();
        cout << endl << "Add noise [sigma = " << fSigma << "] ... " << flush;
        lfio::add_noise_LF(LF, LF_SAI_mask, LF_noisy, fSigma);
        cout << "done in " << float(lfio::now() - t0) << "s." << endl;
        cout << endl << "Save noisy light field..." << endl;
        t0 = lfio::now();
        if (lfio::save_LF(LF_noisy_name, sub_img_name, sep, LF_noisy, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, width, height, chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
        cout << "done in " << float(lfio::now() - t0) << "s." << endl;
    } else {
        const double t0 = lfio::now();
        if (lfio::load_LF(LF_noisy_name, sub_img_name, sep, LF_noisy, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, &width, &height, &chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
        cout << endl << "Loading noisy LF elapsed time = " << float(lfio::now() - t0) << "s." << endl;
    }
    const size_t whc = (size_t) width * height * chnls;
    LF_diff.assign(awh, vector<float>(whc, 0.0f)); LF_basic.assign(awh, vector<float>(whc, 0.0f)); LF_denoised.assign(awh, vector<float>(whc, 0.0f));
    for (unsigned st = 0; st < awh; st++) if (LF_noisy[st].size() != whc) LF_noisy[st].resize(whc, 0.0f);
    if (sigma_auto) {
        vector<float> sigma_chnl;
        if (estimate_sigma_LF(LF_noisy, LF_SAI_mask, width, height, chnls, &fSigma, &sigma_chnl) != EXIT_SUCCESS) return EXIT_FAILURE;
        char line[160];
        int n = snprintf(line, sizeof(line), "Estimated noise level: sigma = %.9g (per channel:", fSigma);
        for (float s : sigma_chnl) n += snprintf(line + n, sizeof(line) - n, " %.9g", s);
        cout << endl << line << ")" << endl;
    }
    vector<float> psnr_noisy, rmse_noisy, psnr_basic, rmse_basic, psnr, rmse;
    float apn = 0, arn = 0, spn = 0, srn = 0, apb = 0, arb = 0, spb = 0, srb = 0, ap = 0, ar = 0, sp = 0, sr = 0;
    if (gt_exists) {
        if (lfio::compute_psnr_LF(LF, LF_noisy, LF_SAI_mask, psnr_noisy, &apn, &spn, rmse_noisy, &arn, &srn) != EXIT_SUCCESS) return EXIT_FAILURE;
        cout << endl << "Average PSNR:" << endl << "- Noisy light field: " << apn << endl;
        lfio::write_psnr_LF(psnr_file_name, "noisy", LF_SAI_mask, ang_major, awidth, aheight, psnr_noisy, apn, spn, rmse_noisy, arn, srn, ROWMAJOR);
    }
    cout << endl << " ---> Running BM3D filter <--- " << endl << endl;
    const double start = lfio::now();
    char name[4] = "SAI";
    if (run_bm3d_LF(fSigma, LF_noisy, LF_SAI_mask, LF_basic, LF_denoised, width, height, chnls, n[0], n[1], k[0], k[1], N[0], N[1], p[0], p[1],
                    useSD[0], useSD[1], t2[0], t2[1], lambdaHard3D, color_space, nb_threads, name) != EXIT_SUCCESS) return EXIT_FAILURE;
    const float secs = float(lfio::now() - start);
    if (gt_exists) {
        if (lfio::compute_psnr_LF(LF, LF_basic, LF_SAI_mask, psnr_basic, &apb, &spb, rmse_basic, &arb, &srb) != EXIT_SUCCESS) return EXIT_FAILURE;
        lfio::write_psnr_LF(psnr_file_name, "basic", LF_SAI_mask, ang_major, awidth, aheight, psnr_basic, apb, spb, rmse_basic, arb, srb, ROWMAJOR);
    }
    cout << endl << "Save basic light field..." << endl;
    if (lfio::save_LF(LF_basic_name, sub_img_name, sep, LF_basic, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, width, height, chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
    if (gt_exists) {
        if (lfio::compute_psnr_LF(LF, LF_denoised, LF_SAI_mask, psnr, &ap, &sp, rmse, &ar, &sr) != EXIT_SUCCESS) return EXIT_FAILURE;
        cout << endl << "Average PSNR:" << endl << "- Noisy light field: " << apn << endl << "- Basic light field: " << apb << endl
             << "- Denoised light field: " << ap << endl << endl;
        lfio::write_psnr_LF(psnr_file_name, "denoised", LF_SAI_mask, ang_major, awidth, aheight, psnr, ap, sp, rmse, ar, sr, ROWMAJOR);
        lfio::compute_diff_LF(LF, LF_denoised, LF_SAI_mask, LF_diff, fSigma);
    }
    cout << endl << "Save denoised light field..." << endl;
    if (lfio::save_LF(LF_denoised_name, sub_img_name, sep, LF_denoised, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, width, height, chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
    if (gt_exists) {
        cout << endl << "Save diff light field..." << endl;
        if (lfio::save_LF(LF_diff_name, sub_img_name, sep, LF_diff, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, width, height, chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
    }
    cout << "Total BM3D computing time = " << secs << "s." << endl;
    cout << endl;
    cout << "*********************************************************************************************************************" << endl;
    cout << "********************************************         THIS IS THE END          ***************************************" << endl;
    cout << "*********************************************************************************************************************" << endl;
    return EXIT_SUCCESS;
}
