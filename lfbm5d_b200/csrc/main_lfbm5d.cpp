// LFBM5Ddenoising — same 37 positional arguments, console messages and report file as the reference's main.cpp:60-309
// (argument grammar: utilities_LF.cpp:1128-1312, README.md:80-118); the two denoising steps run on the GPU through
// run_bm5d_1st_step / run_bm5d_2nd_step (lfbm5d_host.h).
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
    if (argc < 38) {
        cout << "usage: LFBM5Ddenoising LF_dir SAI_name SAI_name_sep LF_awidth LF_aheight s_idx_start t_idx_start asw_size_ht asw_size_wien ang_major sigma lambda "
                "LF_dir_noisy LF_dir_basic LF_dir_denoised LF_dir_difference "
                "NHard nSimHard nDispHard khard pHard tau_2d_hard tau_4d_hard tau_5d_hard useSD_hard "
                "NWien nSimWien nDispWien kWien pWien tau_2d_wien tau_4d_wien tau_5d_wien useSD_wien "
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
    const unsigned anHard = atoi(argv[++i]), anWien = atoi(argv[++i]);
    const unsigned ang_major = pick(argv[++i], { { "row", ROWMAJOR }, { "col", COLMAJOR } });
    if (ang_major == NONE) { cout << "ang_major is not known. Choice is :" << endl << " -row" << endl << " -col" << endl; return EXIT_FAILURE; }
    // sigma = auto: estimated from the noisy light field read back from disk (estimate_sigma_LF), so only without ground truth
    const bool sigma_auto = strcmp(argv[++i], "auto") == 0;
    float fSigma = sigma_auto ? 0.0f : atof(argv[i]);
    const float lambdaHard5D = atof(argv[++i]);
    if (sigma_auto && gt_exists) {
        cout << "sigma = auto needs LF_dir = none: with a ground-truth light field, noise of the given sigma is added to it. "
                "Give sigma as a number, or LF_dir = none to denoise the light field in LF_dir_noisy." << endl;
        return EXIT_FAILURE;
    }
    const char *LF_noisy_name = argv[++i], *LF_basic_name = argv[++i], *LF_denoised_name = argv[++i], *LF_diff_name = argv[++i];
    unsigned N[2], nSim[2], nDisp[2], k[2], p[2], t2[2], t4[2], t5[2];
    bool useSD[2];
    for (int s = 0; s < 2; s++) {
        N[s] = atof(argv[++i]); nSim[s] = atof(argv[++i]); nDisp[s] = atof(argv[++i]); k[s] = atof(argv[++i]); p[s] = atof(argv[++i]);
        const char *nm = s == 0 ? "hard" : "wien";
        t2[s] = pick(argv[++i], { { "id", ID }, { "dct", DCT }, { "bior", BIOR } });
        if (t2[s] == NONE) { cout << "tau_2d_" << nm << " is not known. Choice is :" << endl << " -id" << endl << " -dct" << endl << " -bior" << endl; return EXIT_FAILURE; }
        t4[s] = pick(argv[++i], { { "id", ID }, { "dct", DCT }, { "sadct", SADCT } });
        if (t4[s] == NONE) { cout << "tau_4d_" << nm << " is not known. Choice is :" << endl << " -id" << endl << " -dct" << endl << " -sadct" << endl; return EXIT_FAILURE; }
        t5[s] = pick(argv[++i], { { "hw", HADAMARD }, { "haar", HAAR }, { "dct", DCT } });
        if (t5[s] == NONE) { cout << "tau_5d_hard is not known. Choice is :" << endl << " -hw" << endl << " -haar" << endl << " -dct" << endl; return EXIT_FAILURE; }
        useSD[s] = (bool) atof(argv[++i]);
    }
    const unsigned color_space = pick(argv[++i], { { "rgb", RGB }, { "yuv", YUV }, { "ycbcr", YCBCR }, { "opp", OPP } });
    if (color_space == NONE) { cout << "color_space is not known. Choice is :" << endl << " -rgb" << endl << " -yuv" << endl << " -opp" << endl << " -ycbcr" << endl; return EXIT_FAILURE; }
    unsigned nb_threads = atof(argv[++i]);
    const char *psnr_file_name = argv[++i];
    if (!nb_threads) nb_threads = 1;      // accepted and ignored: results always follow the reference's nb_threads = 1 semantics

    vector<vector<float> > LF, LF_noisy, LF_basic, LF_denoised, LF_diff;
    vector<unsigned> LF_SAI_mask;
    unsigned width = 0, height = 0, chnls = 0;
    const unsigned awh = awidth * aheight;
    if (gt_exists) {
        const double t0 = lfio::now();
        if (lfio::load_LF(LF_input_name, sub_img_name, sep, LF, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, &width, &height, &chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
        cout << "Loading LF elapsed time = " << float(lfio::now() - t0) << "s." << endl;
        LF_noisy.assign(awh, vector<float>());
        double t1 = lfio::now();
        cout << endl << "Add noise [sigma = " << fSigma << "] ... " << flush;
        lfio::add_noise_LF(LF, LF_SAI_mask, LF_noisy, fSigma);
        cout << "done in " << float(lfio::now() - t1) << "s." << endl;
        cout << endl << "Save noisy light field..." << endl;
        t1 = lfio::now();
        {   // save_image clips to [0, 255] before writing (utilities.cpp:129-130)
            if (lfio::save_LF(LF_noisy_name, sub_img_name, sep, LF_noisy, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, width, height, chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
        }
        cout << "done in " << float(lfio::now() - t1) << "s." << endl;
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

    vector<float> psnr_noisy, rmse_noisy, psnr_basic, rmse_basic;
    float avg_psnr_noisy = 0, avg_rmse_noisy = 0, std_psnr_noisy = 0, std_rmse_noisy = 0;
    float avg_psnr_basic = 0, avg_rmse_basic = 0, std_psnr_basic = 0, std_rmse_basic = 0;
    if (gt_exists) {
        if (lfio::compute_psnr_LF(LF, LF_noisy, LF_SAI_mask, psnr_noisy, &avg_psnr_noisy, &std_psnr_noisy, rmse_noisy, &avg_rmse_noisy, &std_rmse_noisy) != EXIT_SUCCESS) return EXIT_FAILURE;
        cout << endl << "Average PSNR:" << endl << "- Noisy light field: " << avg_psnr_noisy << endl;
        lfio::write_psnr_LF(psnr_file_name, "noisy", LF_SAI_mask, ang_major, awidth, aheight, psnr_noisy, avg_psnr_noisy, std_psnr_noisy, rmse_noisy, avg_rmse_noisy, std_rmse_noisy, ROWMAJOR);
    }

    cout << endl << " ---> Running LFBM5D filter <--- " << endl << endl;
    const double start_bm5d = lfio::now();
    cout << "Step 1 running..." << endl;
    double t0 = lfio::now();
    if (run_bm5d_1st_step(fSigma, lambdaHard5D, LF_noisy, LF_SAI_mask, LF_basic, ang_major, awidth, aheight, anHard, width, height, chnls,
                          N[0], nSim[0], nDisp[0], k[0], p[0], useSD[0], t2[0], t4[0], t5[0], color_space, nb_threads) != EXIT_SUCCESS) return EXIT_FAILURE;
    const float step1_elapsed_secs = float(lfio::now() - t0);
    cout << endl << "Step 1 done in " << step1_elapsed_secs << " secs." << endl << endl;
    if (gt_exists) {
        if (lfio::compute_psnr_LF(LF, LF_basic, LF_SAI_mask, psnr_basic, &avg_psnr_basic, &std_psnr_basic, rmse_basic, &avg_rmse_basic, &std_rmse_basic) != EXIT_SUCCESS) return EXIT_FAILURE;
        cout << endl << "Average PSNR:" << endl << "- Noisy light field: " << avg_psnr_noisy << endl << "- Basic light field: " << avg_psnr_basic << endl;
        lfio::write_psnr_LF(psnr_file_name, "basic", LF_SAI_mask, ang_major, awidth, aheight, psnr_basic, avg_psnr_basic, std_psnr_basic, rmse_basic, avg_rmse_basic, std_rmse_basic, ROWMAJOR);
        cout << endl << "Compute difference... ";
        t0 = lfio::now();
        lfio::compute_diff_LF(LF, LF_basic, LF_SAI_mask, LF_diff, fSigma);
        cout << "done. Compute diff LF elapsed time = " << float(lfio::now() - t0) << "s." << endl;
    }
    cout << endl << "Save basic light field..." << endl;
    t0 = lfio::now();
    if (lfio::save_LF(LF_basic_name, sub_img_name, sep, LF_basic, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, width, height, chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
    cout << "done in " << float(lfio::now() - t0) << "s." << endl;

    cout << endl << endl << "Step 2 running..." << endl;
    t0 = lfio::now();
    if (run_bm5d_2nd_step(fSigma, LF_noisy, LF_SAI_mask, LF_basic, LF_denoised, ang_major, awidth, aheight, anWien, width, height, chnls,
                          N[1], nSim[1], nDisp[1], k[1], p[1], useSD[1], t2[1], t4[1], t5[1], color_space, nb_threads) != EXIT_SUCCESS) return EXIT_FAILURE;
    const float step2_elapsed_secs = float(lfio::now() - t0);
    cout << endl << "Step 2 done in " << step2_elapsed_secs << " secs." << endl << endl;
    if (gt_exists) {
        vector<float> psnr, rmse;
        float avg_psnr, avg_rmse, std_psnr, std_rmse;
        if (lfio::compute_psnr_LF(LF, LF_denoised, LF_SAI_mask, psnr, &avg_psnr, &std_psnr, rmse, &avg_rmse, &std_rmse) != EXIT_SUCCESS) return EXIT_FAILURE;
        cout << endl << "Average PSNR:" << endl << "- Noisy light field: " << avg_psnr_noisy << endl << "- Basic light field: " << avg_psnr_basic << endl
             << "- Denoised light field: " << avg_psnr << endl << endl;
        lfio::write_psnr_LF(psnr_file_name, "denoised", LF_SAI_mask, ang_major, awidth, aheight, psnr, avg_psnr, std_psnr, rmse, avg_rmse, std_rmse, ROWMAJOR);
        cout << endl << "Compute difference... ";
        t0 = lfio::now();
        lfio::compute_diff_LF(LF, LF_denoised, LF_SAI_mask, LF_diff, fSigma);
        cout << "done in " << float(lfio::now() - t0) << "s." << endl;
    }
    cout << endl << "Save denoised light field..." << endl;
    t0 = lfio::now();
    if (lfio::save_LF(LF_denoised_name, sub_img_name, sep, LF_denoised, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, width, height, chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
    cout << "done in " << float(lfio::now() - t0) << "s." << endl;
    if (gt_exists) {
        cout << endl << "Save diff light field..." << endl;
        t0 = lfio::now();
        if (lfio::save_LF(LF_diff_name, sub_img_name, sep, LF_diff, LF_SAI_mask, ang_major, awidth, aheight, s_start, t_start, width, height, chnls, ROWMAJOR) != EXIT_SUCCESS) return EXIT_FAILURE;
        cout << "done in " << float(lfio::now() - t0) << "s." << endl << endl;
    }
    cout << "Total LFBM5D computing time = " << step1_elapsed_secs + step2_elapsed_secs << "s." << endl;
    cout << "Total elapsed time = " << float(lfio::now() - start_bm5d) << "s." << endl;
    cout << endl;
    cout << "*********************************************************************************************************************" << endl;
    cout << "********************************************         THIS IS THE END          ***************************************" << endl;
    cout << "*********************************************************************************************************************" << endl;
    return EXIT_SUCCESS;
}
