// TEST INFRASTRUCTURE (tests/test_gpu_tall_frames.py builds it into a temporary directory).
//
// The four float prefix arrays of the CPU oracle -- the Blelloch-order exclusive scans of disparity, valid, ground
// and sky that oracle/stixels_cpu.cpp computes per column, literally as the reference does over rows_power2 rows --
// which its own entry point keeps internal.  The oracle's source is compiled unchanged into this translation unit,
// with the flags of oracle/Makefile, so these are the very arrays its DP uses.
#include "../../oracle/stixels_cpu.cpp"

extern "C" {

// prefix: [realcols][4][rows + 1]: disparity, valid, ground, sky.  valid stays zero with invalid_disparity < 0,
// where the reference does not scan it.  Returns 0.
int orc_prefix_tables(const isx_config *cfg, int pairwise, const float *disparity, const int32_t *segmentation,
                      const isx_road *road, int nthreads, float *prefix) {
  Model m(*cfg);
  std::vector<float> gf, ng, ig;
  const int vhor = m.ground(*road, gf, ng, ig);
  Ctx c{m, gf, ng, ig, vhor, pairwise != 0};
  const int C = m.realcols, H = m.rows;
  std::vector<isx_section> sections((size_t)C * kMaxSections);
  if (nthreads <= 0) nthreads = omp_get_max_threads();
#pragma omp parallel num_threads(nthreads)
  {
    _mm_setcsr(_mm_getcsr() | 0x8040);  // FTZ + DAZ, as in orc_compute_frame
    ColumnWork w;
#pragma omp for schedule(dynamic, 1)
    for (int col = 0; col < C; col++) {
      process_column(c, col, disparity, segmentation, w, sections.data() + (size_t)col * kMaxSections);
      const std::vector<float> *ps[4] = {&w.disp_ps, &w.valid_ps, &w.ground_ps, &w.sky_ps};   // rows_power2 > rows
      for (int i = 0; i < 4; i++)
        std::memcpy(prefix + ((size_t)col * 4 + i) * (H + 1), ps[i]->data(), sizeof(float) * (H + 1));
    }
  }
  return 0;
}

}  // extern "C"
