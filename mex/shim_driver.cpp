// shim_driver.cpp -- exercises one gateway (compiled together with it) under the mex shim.
// Without a GPU only the argument validation is checked (it happens before any CUDA call and must
// raise the reference's identifiers); with a GPU (argv[1] == "gpu") a small real call runs too.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "mex.h"

static int expect_error(const char* want, int nlhs, int nrhs, const mxArray** in) {
  mxArray* out[4] = {nullptr, nullptr, nullptr, nullptr};
  try {
    mexFunction(nlhs, out, nrhs, in);
  } catch (const mexShimError& e) {
    if (e.id == want) return 0;
    std::printf("FAIL: expected %s, got %s (%s)\n", want, e.id.c_str(), e.what());
    return 1;
  }
  std::printf("FAIL: expected %s, no error raised\n", want);
  return 1;
}

// ---- file mode: `gate file in.bin out.bin` ---------------------------------------------------------------------
// in.bin : int32 nmat ; per matrix int32 cls (0 single, 1 uint8, 2 double, 4 uint8 wrapped in a binaryFeatures
//          object), int32 rows, int32 cols, column-major payload ; int32 nscalars ; doubles ; optionally (batched
//          gateway) int32 ngpus ; doubles = the trailing `gpus` vector (1-based GPU indices).
// out.bin: int32 nout ; per output int32 cls (0 single, 1 uint8, 2 double, 3 uint32, -1 empty), rows, cols, payload.
// tests/test_mex_gateways.py builds the inputs, runs the gateway on the GPU and compares the outputs with the oracle.
static mxArray* read_matrix(FILE* f) {
  int32_t h[3];
  if (std::fread(h, 4, 3, f) != 3) return nullptr;
  const mxClassID cls = h[0] == 0 ? mxSINGLE_CLASS : (h[0] == 2 ? mxDOUBLE_CLASS : mxUINT8_CLASS);
  mxArray* a = mxCreateNumericMatrix((mwSize)h[1], (mwSize)h[2], cls, mxREAL);
  const size_t bytes = (size_t)h[1] * h[2] * mxshim_elem_size(cls);
  if (bytes && std::fread(mxGetData(a), 1, bytes, f) != bytes) return nullptr;
  if (h[0] == 4) {
    mxArray* o = new mxArray();
    o->cls = mxUNKNOWN_CLASS;
    o->dims = {1, 1};
    o->class_name = "binaryFeatures";
    o->properties.push_back({"Features", a});
    return o;
  }
  return a;
}
static void write_matrix(FILE* f, const mxArray* a) {
  int32_t h[3] = {-1, 0, 0};
  if (a && !mxIsCell(a)) {
    h[0] = mxIsSingle(a) ? 0 : mxIsUint8(a) ? 1 : mxIsDouble(a) ? 2 : mxIsUint32(a) ? 3 : -1;
    h[1] = (int32_t)mxGetM(a);
    h[2] = (int32_t)mxGetN(a);
  }
  std::fwrite(h, 4, 3, f);
  if (h[0] >= 0) std::fwrite(mxGetData(a), mxshim_elem_size(mxGetClassID(a)), (size_t)h[1] * h[2], f);
}
static int file_mode(const char* in_path, const char* out_path) {
  FILE* f = std::fopen(in_path, "rb");
  if (!f) return 2;
  int32_t nmat = 0, nsc = 0;
  if (std::fread(&nmat, 4, 1, f) != 1) return 2;
  std::vector<mxArray*> mats;
  for (int i = 0; i < nmat; ++i) mats.push_back(read_matrix(f));
  if (std::fread(&nsc, 4, 1, f) != 1) return 2;
  std::vector<double> sc((size_t)nsc);
  if (nsc && std::fread(sc.data(), 8, (size_t)nsc, f) != (size_t)nsc) return 2;
  int32_t ngpu = 0;
  std::vector<double> gpus;
  if (std::fread(&ngpu, 4, 1, f) == 1 && ngpu > 0) {
    gpus.resize((size_t)ngpu);
    if (std::fread(gpus.data(), 8, (size_t)ngpu, f) != (size_t)ngpu) return 2;
  }
  std::fclose(f);
  mxArray* out[4] = {nullptr, nullptr, nullptr, nullptr};
  int nout = 0;
  std::vector<const mxArray*> outs;
  try {
#if defined(GATE_FLANN)   // scalars: k, use_bf ; matrices: train [, query]
    std::vector<const mxArray*> in(mats.begin(), mats.end());
    in.push_back(mxCreateDoubleScalar(sc[0]));
    if (sc.size() > 1 && sc[1] != 0.0) in.push_back(mxCreateString("bf"));
    mexFunction(2, out, (int)in.size(), in.data());
    outs = {out[0], out[1]};
#elif defined(GATE_HAMMING)
    const mxArray* in[] = {mats[0], mats[1]};
    mexFunction(3, out, 2, in);
    outs = {out[0], out[1], out[2]};
#elif defined(GATE_BATCHED)  // scalars: mode (0 global, 1 pairwise), then (k, ratio, useBF) or (MatchThreshold, MaxRatio)
    // 'globalsets': scalars 2, B, numImgs(1..B), k, ratio, useBF, mutual; 'pairwisesets': scalars 3, B, numImgs(1..B),
    // MatchThreshold, MaxRatio, method; matrices = all sets' images
    if (sc[0] == 2.0 || sc[0] == 3.0) {
      const int B = (int)sc[1];
      mxArray* sets = mxCreateCellMatrix(1, (mwSize)B);
      mxArray* nimg = mxCreateDoubleMatrix(1, (mwSize)B, mxREAL);
      for (int b = 0, m0 = 0; b < B; ++b) {
        const int n = (int)sc[2 + b];
        mxGetPr(nimg)[b] = n;
        mxArray* cb = mxCreateCellMatrix(1, (mwSize)n);
        for (int i = 0; i < n; ++i) mxSetCell(cb, (mwIndex)i, mats[m0 + i]);
        m0 += n;
        mxSetCell(sets, (mwIndex)b, cb);
      }
      std::vector<const mxArray*> in = {mxCreateString(sc[0] == 2.0 ? "globalsets" : "pairwisesets"), sets, nimg};
      for (size_t i = 2 + B; i < sc.size(); ++i) in.push_back(mxCreateDoubleScalar(sc[i]));
      mexFunction(1, out, (int)in.size(), in.data());
      for (int b = 0; b < B; ++b) {  // per set: upper-triangle cells in column-major order
        const mxArray* cb = mxGetCell(out[0], (mwIndex)b);
        const int n = (int)sc[2 + b];
        for (int j = 0; j < n; ++j)
          for (int i = 0; i < j; ++i) outs.push_back(mxGetCell(cb, (mwIndex)(i + j * n)));
      }
    } else {
    mxArray* cells = mxCreateCellMatrix(1, (mwSize)nmat);
    for (int i = 0; i < nmat; ++i) mxSetCell(cells, (mwIndex)i, mats[i]);
    std::vector<const mxArray*> in = {mxCreateString(sc[0] == 0.0 ? "global" : "pairwise"), cells,
                                      mxCreateDoubleScalar((double)nmat)};
    for (size_t i = 1; i < sc.size(); ++i) in.push_back(mxCreateDoubleScalar(sc[i]));
    if (!gpus.empty()) {  // after (k, ratio, useBF) / (MatchThreshold, MaxRatio, method)
      mxArray* g = mxCreateDoubleMatrix(1, (mwSize)gpus.size(), mxREAL);
      for (size_t i = 0; i < gpus.size(); ++i) mxGetPr(g)[i] = gpus[i];
      in.push_back(g);
    }
    mexFunction(1, out, (int)in.size(), in.data());
    for (int j = 0; j < nmat; ++j)   // upper-triangle cells in column-major order
      for (int i = 0; i < j; ++i) outs.push_back(mxGetCell(out[0], (mwIndex)(i + j * nmat)));
    }
#elif defined(GATE_MATCHF)   // scalars: kind, MatchThreshold, MaxRatio, Unique
    mxArray* uq = mxCreateLogicalMatrix(1, 1);
    ((unsigned char*)mxGetData(uq))[0] = sc[3] != 0.0;
    const mxArray* in[] = {mats[0], mats[1], mxCreateDoubleScalar(sc[0]), mxCreateDoubleScalar(sc[1]),
                           mxCreateDoubleScalar(sc[2]), uq};
    mexFunction(2, out, 6, in);
    outs = {out[0], out[1]};
#elif defined(GATE_IMATCH_SETS)  // scalars: B, numImgs(1..B), m, maxDistance, confidence, maxIter, seed ; matrices: per
    // set its n_b keypoint matrices, then its n_b^2 matchesAll cells in column-major order.  outputs per set: the n_b^2
    // allMatches cells (column-major), numMatches, the n_b^2 tforms cells
    const int B = (int)sc[0];
    mxArray *kps = mxCreateCellMatrix(1, (mwSize)B), *mcs = mxCreateCellMatrix(1, (mwSize)B);
    for (int b = 0, m0 = 0; b < B; ++b) {
      const int n = (int)sc[1 + b];
      mxArray *kc = mxCreateCellMatrix(1, (mwSize)n), *mc = mxCreateCellMatrix((mwSize)n, (mwSize)n);
      for (int i = 0; i < n; ++i) mxSetCell(kc, (mwIndex)i, mats[m0++]);
      for (int c = 0; c < n * n; ++c) mxSetCell(mc, (mwIndex)c, mats[m0++]);
      mxSetCell(kps, (mwIndex)b, kc);
      mxSetCell(mcs, (mwIndex)b, mc);
    }
    std::vector<const mxArray*> in = {kps, mcs};
    for (size_t i = 1 + B; i < sc.size(); ++i) in.push_back(mxCreateDoubleScalar(sc[i]));
    mexFunction(3, out, (int)in.size(), in.data());
    for (int b = 0; b < B; ++b) {
      const int n = (int)sc[1 + b];
      for (int c = 0; c < n * n; ++c) outs.push_back(mxGetCell(mxGetCell(out[0], (mwIndex)b), (mwIndex)c));
      outs.push_back(mxGetCell(out[1], (mwIndex)b));
      for (int c = 0; c < n * n; ++c) outs.push_back(mxGetCell(mxGetCell(out[2], (mwIndex)b), (mwIndex)c));
    }
#elif defined(GATE_GIMATCH)  // scalars: B, numImgs(1..B), k, ratio, m, maxDistance, confidence, maxIter, seed ; matrices:
    // per set its n_b descriptor matrices, then its n_b keypoint matrices.  outputs per set: the n_b^2 allMatches cells
    // (column-major), numMatches, the n_b^2 tforms cells
    const int B = (int)sc[0];
    mxArray *ds = mxCreateCellMatrix(1, (mwSize)B), *kps = mxCreateCellMatrix(1, (mwSize)B);
    mxArray* nums = mxCreateDoubleMatrix(1, (mwSize)B, mxREAL);
    for (int b = 0, m0 = 0; b < B; ++b) {
      const int n = (int)sc[1 + b];
      mxGetPr(nums)[b] = n;
      mxArray *dc = mxCreateCellMatrix(1, (mwSize)n), *kc = mxCreateCellMatrix(1, (mwSize)n);
      for (int i = 0; i < n; ++i) mxSetCell(dc, (mwIndex)i, mats[m0++]);
      for (int i = 0; i < n; ++i) mxSetCell(kc, (mwIndex)i, mats[m0++]);
      mxSetCell(ds, (mwIndex)b, dc);
      mxSetCell(kps, (mwIndex)b, kc);
    }
    const double* t = sc.data() + 1 + B;  // k, ratio, m, maxDistance, confidence, maxIter, seed
    std::vector<const mxArray*> in = {ds, nums, kps, mxCreateDoubleScalar(t[0]), mxCreateDoubleScalar(t[1]),
                                      mxCreateDoubleScalar(0)};
    for (int i = 2; i < 7; ++i) in.push_back(mxCreateDoubleScalar(t[i]));
    mexFunction(3, out, (int)in.size(), in.data());
    for (int b = 0; b < B; ++b) {
      const int n = (int)sc[1 + b];
      for (int c = 0; c < n * n; ++c) outs.push_back(mxGetCell(mxGetCell(out[0], (mwIndex)b), (mwIndex)c));
      outs.push_back(mxGetCell(out[1], (mwIndex)b));
      for (int c = 0; c < n * n; ++c) outs.push_back(mxGetCell(mxGetCell(out[2], (mwIndex)b), (mwIndex)c));
    }
#elif defined(GATE_PIMATCH)  // scalars: B, numImgs(1..B), matchThreshold, maxRatio, method, m, maxDistance, confidence,
    // maxIter, seed ; matrices and outputs as GATE_GIMATCH
    const int B = (int)sc[0];
    mxArray *ds = mxCreateCellMatrix(1, (mwSize)B), *kps = mxCreateCellMatrix(1, (mwSize)B);
    mxArray* nums = mxCreateDoubleMatrix(1, (mwSize)B, mxREAL);
    for (int b = 0, m0 = 0; b < B; ++b) {
      const int n = (int)sc[1 + b];
      mxGetPr(nums)[b] = n;
      mxArray *dc = mxCreateCellMatrix(1, (mwSize)n), *kc = mxCreateCellMatrix(1, (mwSize)n);
      for (int i = 0; i < n; ++i) mxSetCell(dc, (mwIndex)i, mats[m0++]);
      for (int i = 0; i < n; ++i) mxSetCell(kc, (mwIndex)i, mats[m0++]);
      mxSetCell(ds, (mwIndex)b, dc);
      mxSetCell(kps, (mwIndex)b, kc);
    }
    const double* t = sc.data() + 1 + B;  // matchThreshold, maxRatio, method, m, maxDistance, confidence, maxIter, seed
    std::vector<const mxArray*> in = {ds, nums, kps};
    for (int i = 0; i < 8; ++i) in.push_back(mxCreateDoubleScalar(t[i]));
    mexFunction(3, out, (int)in.size(), in.data());
    for (int b = 0; b < B; ++b) {
      const int n = (int)sc[1 + b];
      for (int c = 0; c < n * n; ++c) outs.push_back(mxGetCell(mxGetCell(out[0], (mwIndex)b), (mwIndex)c));
      outs.push_back(mxGetCell(out[1], (mwIndex)b));
      for (int c = 0; c < n * n; ++c) outs.push_back(mxGetCell(mxGetCell(out[2], (mwIndex)b), (mwIndex)c));
    }
#else
    (void)out;
    return 3;
#endif
  } catch (const mexShimError& e) {
    std::printf("ERROR %s: %s\n", e.id.c_str(), e.what());
    return 1;
  }
  nout = (int)outs.size();
  FILE* g = std::fopen(out_path, "wb");
  if (!g) return 2;
  std::fwrite(&nout, 4, 1, g);
  for (const mxArray* a : outs) write_matrix(g, a);
  std::fclose(g);
  std::printf("OK\n");
  return 0;
}

#if defined(GATE_BATCHED)
// `gate_batched gpus`: the trailing gpus argument of the batched gateway is validated before any device is touched;
// without a GPU a well-formed multi-GPU list reaches aps_group_create and fails with apsmatch:nogpu.
static int gpus_argument_checks() {
  int bad = 0;
  mxArray* cells = mxCreateCellMatrix(1, 2);
  mxArray* a = mxCreateNumericMatrix(6, 8, mxSINGLE_CLASS, mxREAL);
  mxSetCell(cells, 0, a);
  mxSetCell(cells, 1, mxCreateNumericMatrix(6, 8, mxSINGLE_CLASS, mxREAL));
  mxArray *n2 = mxCreateDoubleScalar(2), *k = mxCreateDoubleScalar(4), *r = mxCreateDoubleScalar(0.6);
  mxArray* opt = mxCreateDoubleScalar(1);  // useBF / method
  auto vec = [](std::vector<double> v) {
    mxArray* g = mxCreateDoubleMatrix(1, (mwSize)v.size(), mxREAL);
    for (size_t i = 0; i < v.size(); ++i) mxGetPr(g)[i] = v[i];
    return g;
  };
  mxArray* bad_lists[] = {vec({0}), vec({1, 1.5}), vec({2, 2}), vec({-1, 2}), vec({1, NAN}), mxCreateString("1:2"),
                          mxCreateNumericMatrix(1, 2, mxSINGLE_CLASS, mxREAL), mxCreateDoubleMatrix(2, 2, mxREAL)};
  for (const char* mode : {"global", "pairwise"}) {
    mxArray* m = mxCreateString(mode);
    for (mxArray* g : bad_lists) {
      const mxArray* in[] = {m, cells, n2, k, r, opt, g};
      bad += expect_error("apsmatch:args", 1, 7, in);
    }
    const mxArray* in[] = {m, cells, n2, k, r, opt, vec({1, 2})};
    bad += expect_error("apsmatch:nogpu", 1, 7, in);  // no CPU fallback for a device group either
  }
  std::printf(bad ? "FAILED (%d)\n" : "OK\n", bad);
  return bad ? 1 : 0;
}

// `gate_batched sets [nogpu]`: the argument checks of the 'globalsets' and 'pairwisesets' verbs, all made before any
// device is touched; with `nogpu` a well-formed call must then fail with apsmatch:nogpu (no CPU fallback)
static int sets_argument_checks(bool nogpu) {
  int bad = 0;
  for (const char* verb : {"globalsets", "pairwisesets"}) {
    auto set_of = [](std::vector<mxArray*> m) {
      mxArray* c = mxCreateCellMatrix(1, (mwSize)m.size());
      for (size_t i = 0; i < m.size(); ++i) mxSetCell(c, (mwIndex)i, m[i]);
      return c;
    };
    auto vec = [](std::vector<double> v) {
      mxArray* g = mxCreateDoubleMatrix(1, (mwSize)v.size(), mxREAL);
      for (size_t i = 0; i < v.size(); ++i) mxGetPr(g)[i] = v[i];
      return g;
    };
    mxArray* f8 = mxCreateNumericMatrix(6, 8, mxSINGLE_CLASS, mxREAL);
    mxArray* f16 = mxCreateNumericMatrix(6, 16, mxSINGLE_CLASS, mxREAL);
    mxArray* orb = new mxArray();
    orb->cls = mxUNKNOWN_CLASS;
    orb->dims = {1, 1};
    orb->class_name = "binaryFeatures";
    orb->properties.push_back({"Features", mxCreateNumericMatrix(6, 32, mxUINT8_CLASS, mxREAL)});
    mxArray *mode = mxCreateString(verb), *k = mxCreateDoubleScalar(4), *r = mxCreateDoubleScalar(0.6);
    mxArray* good = set_of({set_of({f8, f8}), set_of({f8})});
    {  // too few arguments, sets not a cell of cells, numImgs of the wrong length / not positive integers
      const mxArray* in[] = {mode, good, vec({2, 1}), k};
      bad += expect_error("apsmatch:args", 1, 4, in);
    }
    for (mxArray* sets : {f8, set_of({f8, f8})}) {
      const mxArray* in[] = {mode, sets, vec({2, 1}), k, r};
      bad += expect_error("apsmatch:args", 1, 5, in);
    }
    for (mxArray* n : {vec({2}), vec({2, 0}), vec({2, 1.5}), vec({2, NAN})}) {
      const mxArray* in[] = {mode, good, n, k, r};
      bad += expect_error("apsmatch:args", 1, 5, in);
    }
    {  // sets of different classes or widths
      const mxArray* in1[] = {mode, set_of({set_of({f8}), set_of({orb})}), vec({1, 1}), k, r};
      bad += expect_error("apsmatch:args", 1, 5, in1);
      const mxArray* in2[] = {mode, set_of({set_of({f8}), set_of({f16})}), vec({1, 1}), k, r};
      bad += expect_error("apsmatch:args", 1, 5, in2);
    }
    {  // every set empty: 1 x B cell of cell(numImgs(b)) without touching the GPU
      mxArray* out[1] = {nullptr};
      const mxArray* in[] = {mode, set_of({mxCreateCellMatrix(1, 2), mxCreateCellMatrix(1, 3)}), vec({2, 3}), k, r};
      mexFunction(1, out, 5, in);
      const mxArray* c1 = out[0] ? mxGetCell(out[0], 1) : nullptr;
      bad += !(out[0] && mxGetN(out[0]) == 2 && c1 && mxIsCell(c1) && mxGetM(c1) == 3 && mxGetN(c1) == 3);
    }
    if (nogpu) {
      const mxArray* in[] = {mode, good, vec({2, 1}), k, r};
      bad += expect_error("apsmatch:nogpu", 1, 5, in);
    }
  }
  std::printf(bad ? "FAILED (%d)\n" : "OK\n", bad);
  return bad ? 1 : 0;
}
#endif

int main(int argc, char** argv) {
  if (argc > 3 && !std::strcmp(argv[1], "file")) return file_mode(argv[2], argv[3]);
#if defined(GATE_BATCHED)
  if (argc > 1 && !std::strcmp(argv[1], "gpus")) return gpus_argument_checks();
  if (argc > 1 && !std::strcmp(argv[1], "sets")) return sets_argument_checks(argc > 2 && !std::strcmp(argv[2], "nogpu"));
#endif
  const bool gpu = argc > 1 && !std::strcmp(argv[1], "gpu");
  int bad = 0;
#if defined(GATE_FLANN)
  mxArray* T = mxCreateNumericMatrix(8, 4, mxSINGLE_CLASS, mxREAL);
  mxArray* Td = mxCreateDoubleMatrix(8, 4, mxREAL);
  mxArray* Q5 = mxCreateNumericMatrix(3, 5, mxSINGLE_CLASS, mxREAL);
  mxArray *k0 = mxCreateDoubleScalar(0), *k2 = mxCreateDoubleScalar(2), *bf = mxCreateString("bf");
  { const mxArray* in[] = {T}; bad += expect_error("flann_knn:args", 2, 1, in); }
  { const mxArray* in[] = {Td, k2}; bad += expect_error("flann_knn:type", 2, 2, in); }
  { const mxArray* in[] = {T, k0}; bad += expect_error("flann_knn:k", 2, 2, in); }
  { const mxArray* in[] = {T, Q5, k2}; bad += expect_error("flann_knn:dim", 2, 3, in); }
  if (gpu) {
    { const mxArray* in[] = {T, k2, bf}; bad += expect_error("flann_knn:bf", 2, 3, in); }
    float* t = (float*)mxGetData(T);
    for (int i = 0; i < 32; ++i) t[i] = (float)((i * 7) % 11);
    mxArray* out[2] = {nullptr, nullptr};
    const mxArray* in[] = {T, k2};
    mexFunction(2, out, 2, in);
    const uint32_t* idx = (const uint32_t*)mxGetData(out[0]);
    for (int r = 0; r < 8; ++r) bad += idx[r] != (uint32_t)(r + 1);  // nearest neighbour of a row is itself
  } else {
    const mxArray* in[] = {T, k2};
    bad += expect_error("apsmatch:nogpu", 2, 2, in);  // no CPU fallback
  }
#elif defined(GATE_HAMMING)
  mxArray* A = mxCreateNumericMatrix(4, 32, mxUINT8_CLASS, mxREAL);
  mxArray* B = mxCreateNumericMatrix(5, 16, mxUINT8_CLASS, mxREAL);
  mxArray* S = mxCreateNumericMatrix(4, 32, mxSINGLE_CLASS, mxREAL);
  { const mxArray* in[] = {A}; bad += expect_error("hamm2nn:nrhs", 3, 1, in); }
  { const mxArray* in[] = {A, S}; bad += expect_error("hamm2nn:type", 3, 2, in); }
  { const mxArray* in[] = {A, B}; bad += expect_error("hamm2nn:cols", 3, 2, in); }
  if (gpu) {
    mxArray* out[3] = {nullptr, nullptr, nullptr};
    const mxArray* in[] = {A, A};
    mexFunction(3, out, 2, in);
    bad += ((const float*)mxGetData(out[1]))[0] != 0.0f;
  }
#elif defined(GATE_BATCHED)
  mxArray* cells = mxCreateCellMatrix(1, 2);
  mxArray* n2 = mxCreateDoubleScalar(2);
  { const mxArray* in[] = {n2, cells, n2}; bad += expect_error("apsmatch:args", 1, 3, in); }
  {  // all-empty descriptors: cell(numImg) without touching the GPU
    mxArray* out[1] = {nullptr};
    mxArray* mode = mxCreateString("global");
    mxArray *k = mxCreateDoubleScalar(4), *r = mxCreateDoubleScalar(0.6);
    const mxArray* in[] = {mode, cells, n2, k, r};
    mexFunction(1, out, 5, in);
    bad += !(mxIsCell(out[0]) && mxGetM(out[0]) == 2 && mxGetN(out[0]) == 2 && mxGetCell(out[0], 2) == nullptr);
  }
  if (gpu) {
    mxArray* a = mxCreateNumericMatrix(6, 8, mxSINGLE_CLASS, mxREAL);
    mxArray* b = mxCreateNumericMatrix(6, 8, mxSINGLE_CLASS, mxREAL);
    float *pa = (float*)mxGetData(a), *pb = (float*)mxGetData(b);
    for (int i = 0; i < 48; ++i) { pa[i] = (float)((i * 13) % 17) - 8.f; pb[i] = pa[i] + ((i % 6) < 3 ? 0.001f : (float)((i * 5) % 7)); }
    mxSetCell(cells, 0, a);
    mxSetCell(cells, 1, b);
    mxArray* out[1] = {nullptr};
    mxArray* mode = mxCreateString("global");
    mxArray *k = mxCreateDoubleScalar(4), *r = mxCreateDoubleScalar(0.5);
    const mxArray* in[] = {mode, cells, n2, k, r};
    mexFunction(1, out, 5, in);
    const mxArray* c01 = mxGetCell(out[0], 2);  // cell (1,2) -> linear index 0 + 1*2
    bad += !(c01 && mxIsDouble(c01) && mxGetN(c01) == 2 && mxGetM(c01) >= 3);
  }
#elif defined(GATE_IMATCH)
  mxArray* kp = mxCreateCellMatrix(1, 2);
  mxArray* mm = mxCreateCellMatrix(2, 2);
  mxArray* m3 = mxCreateCellMatrix(2, 3);
  mxArray *six = mxCreateDoubleScalar(6), *md = mxCreateDoubleScalar(5.5), *cf = mxCreateDoubleScalar(99.9), *it = mxCreateDoubleScalar(500);
  { const mxArray* in[] = {kp, mm, six}; bad += expect_error("apsmatch:args", 3, 3, in); }
  { const mxArray* in[] = {kp, m3, six, md, cf, it}; bad += expect_error("imageMatching:InvalidMatchesAllSize", 3, 6, in); }
  { mxArray* kp3 = mxCreateCellMatrix(1, 3);
    const mxArray* in[] = {kp3, mm, six, md, cf, it}; bad += expect_error("imageMatching:InvalidKeypointsLength", 3, 6, in); }
  if (gpu) {
    // image 2 = image 1 shifted by (10, -5): 40 correspondences, 30 exact + 10 wrong
    const int N = 40;
    mxArray *k1 = mxCreateDoubleMatrix(N, 2, mxREAL), *k2 = mxCreateDoubleMatrix(N, 2, mxREAL), *m12 = mxCreateDoubleMatrix(N, 2, mxREAL);
    for (int r = 0; r < N; ++r) {
      const double x = (double)((r * 37) % 101) * 7.0, y = (double)((r * 53) % 89) * 9.0;
      mxGetPr(k1)[r] = x; mxGetPr(k1)[r + N] = y;
      mxGetPr(k2)[r] = (r < 30) ? x - 10.0 : (double)((r * 11) % 97) * 5.0;
      mxGetPr(k2)[r + N] = (r < 30) ? y + 5.0 : (double)((r * 29) % 83) * 3.0;
      mxGetPr(m12)[r] = r + 1; mxGetPr(m12)[r + N] = r + 1;
    }
    mxSetCell(kp, 0, k1); mxSetCell(kp, 1, k2); mxSetCell(mm, 2, m12);
    mxArray* out[3] = {nullptr, nullptr, nullptr};
    const mxArray* in[] = {kp, mm, six, md, cf, it};
    mexFunction(3, out, 6, in);
    const mxArray* a12 = mxGetCell(out[0], 2);
    const mxArray* t12 = mxGetCell(out[2], 2);
    bad += !(a12 && mxGetM(a12) == 30 && mxGetN(a12) == 2 && mxGetPr(out[1])[2] == 30.0);
    if (t12) {  // model maps image 2 keypoints to image 1: translation (+10, -5); column-major 3x3
      const double* t = mxGetPr(t12);
      bad += !(std::fabs(t[6] / t[8] - 10.0) < 1e-6 && std::fabs(t[7] / t[8] + 5.0) < 1e-6 && std::fabs(t[0] / t[8] - 1.0) < 1e-8);
    } else {
      ++bad;
    }
    bad += mxGetCell(out[2], 1) == nullptr;  // tforms{2,1} = inv(model)
  } else {
    mxArray *k1 = mxCreateDoubleMatrix(5, 2, mxREAL), *k2 = mxCreateDoubleMatrix(5, 2, mxREAL), *m12 = mxCreateDoubleMatrix(5, 2, mxREAL);
    for (int r = 0; r < 10; ++r) mxGetPr(m12)[r] = (r % 5) + 1;
    mxSetCell(kp, 0, k1); mxSetCell(kp, 1, k2); mxSetCell(mm, 2, m12);
    const mxArray* in[] = {kp, mm, six, md, cf, it};
    bad += expect_error("apsmatch:nogpu", 3, 6, in);  // no CPU fallback
  }
#elif defined(GATE_IMATCH_SETS)
  // two sets: set 1 = two images whose second is the first shifted by (10, -5) (40 correspondences, 30 exact), set 2 =
  // one image (no candidate pair)
  const int N = 40;
  mxArray *k1 = mxCreateDoubleMatrix(N, 2, mxREAL), *k2 = mxCreateDoubleMatrix(N, 2, mxREAL), *m12 = mxCreateDoubleMatrix(N, 2, mxREAL);
  for (int r = 0; r < N; ++r) {
    const double x = (double)((r * 37) % 101) * 7.0, y = (double)((r * 53) % 89) * 9.0;
    mxGetPr(k1)[r] = x; mxGetPr(k1)[r + N] = y;
    mxGetPr(k2)[r] = (r < 30) ? x - 10.0 : (double)((r * 11) % 97) * 5.0;
    mxGetPr(k2)[r + N] = (r < 30) ? y + 5.0 : (double)((r * 29) % 83) * 3.0;
    mxGetPr(m12)[r] = r + 1; mxGetPr(m12)[r + N] = r + 1;
  }
  auto cell_of = [](int m, int n, std::vector<mxArray*> e) {
    mxArray* c = mxCreateCellMatrix((mwSize)m, (mwSize)n);
    for (size_t i = 0; i < e.size(); ++i) mxSetCell(c, (mwIndex)i, e[i]);
    return c;
  };
  mxArray* kp1 = cell_of(1, 2, {k1, k2});
  mxArray* mm1 = cell_of(2, 2, {nullptr, nullptr, m12, nullptr});
  mxArray* kps = cell_of(1, 2, {kp1, cell_of(1, 1, {k1})});
  mxArray* mms = cell_of(1, 2, {mm1, mxCreateCellMatrix(1, 1)});
  mxArray *six = mxCreateDoubleScalar(6), *md = mxCreateDoubleScalar(5.5), *cf = mxCreateDoubleScalar(99.9), *it = mxCreateDoubleScalar(500);
  { const mxArray* in[] = {kps, mms, six}; bad += expect_error("apsmatch:args", 3, 3, in); }
  { const mxArray* in[] = {kp1, mms, six, md, cf, it}; bad += expect_error("apsmatch:args", 3, 6, in); }   // not one per set
  { const mxArray* in[] = {six, mms, six, md, cf, it}; bad += expect_error("apsmatch:args", 3, 6, in); }   // not a cell
  { const mxArray* in[] = {kps, cell_of(1, 2, {mm1, cell_of(1, 2, {nullptr, nullptr})}), six, md, cf, it};
    bad += expect_error("apsmatch:args", 3, 6, in); }                                                      // not n x n
  { const mxArray* in[] = {cell_of(1, 2, {kp1, cell_of(1, 2, {k1, k2})}), mms, six, md, cf, it};
    bad += expect_error("apsmatch:args", 3, 6, in); }                                                      // keypoints != n
  { const mxArray* in[] = {kps, mms, six, md, cf, mxCreateString("500")}; bad += expect_error("apsmatch:args", 3, 6, in); }
  if (gpu) {
    {  // a match index outside the keypoints of set 2 fails the whole call (the library checks it on the host, but the
       // gateway creates its context first)
      mxArray* m12b = mxCreateDoubleMatrix(N, 2, mxREAL);
      for (int r = 0; r < 2 * N; ++r) mxGetPr(m12b)[r] = mxGetPr(m12)[r];
      mxGetPr(m12b)[3] = N + 1;
      const mxArray* in[] = {cell_of(1, 2, {cell_of(1, 1, {k1}), kp1}),
                             cell_of(1, 2, {mxCreateCellMatrix(1, 1), cell_of(2, 2, {nullptr, nullptr, m12b, nullptr})}),
                             six, md, cf, it};
      bad += expect_error("refineMatch:MatchIndexOutOfBounds", 3, 6, in);
    }
    mxArray* out[3] = {nullptr, nullptr, nullptr};
    const mxArray* in[] = {kps, mms, six, md, cf, it};
    mexFunction(3, out, 6, in);
    const mxArray* a12 = mxGetCell(mxGetCell(out[0], 0), 2);
    const mxArray* t12 = mxGetCell(mxGetCell(out[2], 0), 2);
    bad += !(mxGetN(out[0]) == 2 && a12 && mxGetM(a12) == 30 && mxGetPr(mxGetCell(out[1], 0))[2] == 30.0);
    if (t12) {  // model maps image 2 keypoints to image 1: translation (+10, -5); column-major 3x3
      const double* t = mxGetPr(t12);
      bad += !(std::fabs(t[6] / t[8] - 10.0) < 1e-6 && std::fabs(t[7] / t[8] + 5.0) < 1e-6);
    } else {
      ++bad;
    }
    bad += !(mxGetM(mxGetCell(out[0], 1)) == 1 && mxGetCell(mxGetCell(out[0], 1), 0) == nullptr);
  } else {
    const mxArray* in[] = {kps, mms, six, md, cf, it};
    bad += expect_error("apsmatch:nogpu", 3, 6, in);  // no CPU fallback
  }
#elif defined(GATE_GIMATCH)
  // two sets: set 1 = two images of 40 float descriptors, the second a copy of the first, its keypoints the first's
  // shifted by (10, -5); set 2 = one image
  const int N = 40, Dd = 16;
  mxArray *d1 = mxCreateNumericMatrix(N, Dd, mxSINGLE_CLASS, mxREAL), *d2 = mxCreateNumericMatrix(N, Dd, mxSINGLE_CLASS, mxREAL);
  mxArray *k1 = mxCreateDoubleMatrix(N, 2, mxREAL), *k2 = mxCreateDoubleMatrix(N, 2, mxREAL);
  for (int r = 0; r < N; ++r) {
    for (int c = 0; c < Dd; ++c)
      ((float*)mxGetData(d1))[r + c * N] = ((float*)mxGetData(d2))[r + c * N] = (float)(((r + 3) * (c + 7) * 31) % 97);
    const double x = (double)((r * 37) % 101) * 7.0, y = (double)((r * 53) % 89) * 9.0;
    mxGetPr(k1)[r] = x; mxGetPr(k1)[r + N] = y;
    mxGetPr(k2)[r] = x - 10.0; mxGetPr(k2)[r + N] = y + 5.0;
  }
  auto cell_of = [](int m, int n, std::vector<mxArray*> e) {
    mxArray* c = mxCreateCellMatrix((mwSize)m, (mwSize)n);
    for (size_t i = 0; i < e.size(); ++i) mxSetCell(c, (mwIndex)i, e[i]);
    return c;
  };
  mxArray* ds = cell_of(1, 2, {cell_of(1, 2, {d1, d2}), cell_of(1, 1, {d1})});
  mxArray* kps = cell_of(1, 2, {cell_of(1, 2, {k1, k2}), cell_of(1, 1, {k1})});
  mxArray* nums = mxCreateDoubleMatrix(1, 2, mxREAL);
  mxGetPr(nums)[0] = 2; mxGetPr(nums)[1] = 1;
  mxArray *k = mxCreateDoubleScalar(2), *ratio = mxCreateDoubleScalar(0.8), *bf = mxCreateDoubleScalar(0),
          *six = mxCreateDoubleScalar(6), *md = mxCreateDoubleScalar(5.5), *cf = mxCreateDoubleScalar(99.9),
          *it = mxCreateDoubleScalar(500);
  { const mxArray* in[] = {ds, nums, kps, k, ratio, bf}; bad += expect_error("apsmatch:args", 3, 6, in); }
  { const mxArray* in[] = {ds, six, kps, k, ratio, bf, six, md, cf, it}; bad += expect_error("apsmatch:args", 3, 10, in); }
  { const mxArray* in[] = {six, nums, kps, k, ratio, bf, six, md, cf, it}; bad += expect_error("apsmatch:args", 3, 10, in); }
  { const mxArray* in[] = {ds, nums, cell_of(1, 2, {cell_of(1, 1, {k1}), cell_of(1, 1, {k1})}), k, ratio, bf, six, md,
                           cf, it};
    bad += expect_error("apsmatch:args", 3, 10, in); }                                    // keypoints != n
  { const mxArray* in[] = {ds, nums, cell_of(1, 2, {cell_of(1, 2, {k1, mxCreateDoubleMatrix(N - 1, 2, mxREAL)}),
                                                    cell_of(1, 1, {k1})}), k, ratio, bf, six, md, cf, it};
    bad += expect_error("apsmatch:args", 3, 10, in); }                                    // a row per descriptor
  { const mxArray* in[] = {cell_of(1, 2, {cell_of(1, 2, {d1, mxCreateDoubleMatrix(N, Dd + 1, mxREAL)}),
                                          cell_of(1, 1, {d1})}), nums, kps, k, ratio, bf, six, md, cf, it};
    bad += expect_error("flann_knn:dim", 3, 10, in); }
  if (gpu) {  // the library's own checks (the gateway creates its context first)
    { const mxArray* in[] = {ds, nums, kps, mxCreateDoubleScalar(0), ratio, bf, six, md, cf, it};
      bad += expect_error("flann_knn:k", 3, 10, in); }
    { const mxArray* in[] = {ds, nums, kps, k, ratio, bf, six, md, cf, mxCreateDoubleScalar(0)};
      bad += expect_error("apsmatch:args", 3, 10, in); }                                  // maxIter <= 0
    mxArray* out[4] = {nullptr, nullptr, nullptr, nullptr};
    const mxArray* in[] = {ds, nums, kps, k, ratio, bf, six, md, cf, it};
    mexFunction(4, out, 10, in);
    const mxArray* a12 = mxGetCell(mxGetCell(out[0], 0), 2);
    const mxArray* t12 = mxGetCell(mxGetCell(out[2], 0), 2);
    const mxArray* m12 = mxGetCell(mxGetCell(out[3], 0), 2);
    bad += !(mxGetN(out[0]) == 2 && a12 && mxGetM(a12) == N && mxGetPr(mxGetCell(out[1], 0))[2] == N);
    bad += !(m12 && mxGetM(m12) == 2 * N);  // both directions of every row: featureMatchingGlobal.m:149-159
    if (t12) {  // model maps image 2 keypoints to image 1: translation (+10, -5); column-major 3x3
      const double* t = mxGetPr(t12);
      bad += !(std::fabs(t[6] / t[8] - 10.0) < 1e-6 && std::fabs(t[7] / t[8] + 5.0) < 1e-6);
    } else {
      ++bad;
    }
    bad += !(mxGetM(mxGetCell(out[0], 1)) == 1 && mxGetCell(mxGetCell(out[0], 1), 0) == nullptr);
  } else {
    const mxArray* in[] = {ds, nums, kps, k, ratio, bf, six, md, cf, it};
    bad += expect_error("apsmatch:nogpu", 3, 10, in);  // no CPU fallback
  }
#elif defined(GATE_PIMATCH)
  // the sets of GATE_GIMATCH: set 1 = two images, the second a copy of the first with keypoints shifted by (10, -5);
  // set 2 = one image.  Arguments: matchThreshold, maxRatio, method (exhaustive), m, maxDistance, confidence, maxIter
  const int N = 40, Dd = 16;
  mxArray *d1 = mxCreateNumericMatrix(N, Dd, mxSINGLE_CLASS, mxREAL), *d2 = mxCreateNumericMatrix(N, Dd, mxSINGLE_CLASS, mxREAL);
  mxArray *k1 = mxCreateDoubleMatrix(N, 2, mxREAL), *k2 = mxCreateDoubleMatrix(N, 2, mxREAL);
  for (int r = 0; r < N; ++r) {
    for (int c = 0; c < Dd; ++c)
      ((float*)mxGetData(d1))[r + c * N] = ((float*)mxGetData(d2))[r + c * N] = (float)(((r + 3) * (c + 7) * 31) % 97);
    const double x = (double)((r * 37) % 101) * 7.0, y = (double)((r * 53) % 89) * 9.0;
    mxGetPr(k1)[r] = x; mxGetPr(k1)[r + N] = y;
    mxGetPr(k2)[r] = x - 10.0; mxGetPr(k2)[r + N] = y + 5.0;
  }
  auto cell_of = [](int m, int n, std::vector<mxArray*> e) {
    mxArray* c = mxCreateCellMatrix((mwSize)m, (mwSize)n);
    for (size_t i = 0; i < e.size(); ++i) mxSetCell(c, (mwIndex)i, e[i]);
    return c;
  };
  mxArray* ds = cell_of(1, 2, {cell_of(1, 2, {d1, d2}), cell_of(1, 1, {d1})});
  mxArray* kps = cell_of(1, 2, {cell_of(1, 2, {k1, k2}), cell_of(1, 1, {k1})});
  mxArray* nums = mxCreateDoubleMatrix(1, 2, mxREAL);
  mxGetPr(nums)[0] = 2; mxGetPr(nums)[1] = 1;
  mxArray *thr = mxCreateDoubleScalar(1.5), *ratio = mxCreateDoubleScalar(0.8), *meth = mxCreateDoubleScalar(0),
          *six = mxCreateDoubleScalar(6), *md = mxCreateDoubleScalar(5.5), *cf = mxCreateDoubleScalar(99.9),
          *it = mxCreateDoubleScalar(500);
  { const mxArray* in[] = {ds, nums, kps, thr, ratio, meth}; bad += expect_error("apsmatch:args", 3, 6, in); }
  { const mxArray* in[] = {ds, six, kps, thr, ratio, meth, six, md, cf, it}; bad += expect_error("apsmatch:args", 3, 10, in); }
  { const mxArray* in[] = {six, nums, kps, thr, ratio, meth, six, md, cf, it}; bad += expect_error("apsmatch:args", 3, 10, in); }
  { const mxArray* in[] = {ds, nums, kps, thr, ratio, mxCreateString("x"), six, md, cf, it};
    bad += expect_error("apsmatch:args", 3, 10, in); }                                    // scalars only
  { const mxArray* in[] = {ds, nums, cell_of(1, 2, {cell_of(1, 1, {k1}), cell_of(1, 1, {k1})}), thr, ratio, meth, six,
                           md, cf, it};
    bad += expect_error("apsmatch:args", 3, 10, in); }                                    // keypoints != n
  { const mxArray* in[] = {ds, nums, cell_of(1, 2, {cell_of(1, 2, {k1, mxCreateDoubleMatrix(N - 1, 2, mxREAL)}),
                                                    cell_of(1, 1, {k1})}), thr, ratio, meth, six, md, cf, it};
    bad += expect_error("apsmatch:args", 3, 10, in); }                                    // a row per descriptor
  { const mxArray* in[] = {cell_of(1, 2, {cell_of(1, 2, {d1, mxCreateDoubleMatrix(N, Dd + 1, mxREAL)}),
                                          cell_of(1, 1, {d1})}), nums, kps, thr, ratio, meth, six, md, cf, it};
    bad += expect_error("flann_knn:dim", 3, 10, in); }
  if (gpu) {  // the library's own checks (the gateway creates its context first)
    { const mxArray* in[] = {ds, nums, kps, thr, ratio, mxCreateDoubleScalar(7), six, md, cf, it};
      bad += expect_error("apsmatch:args", 3, 10, in); }                                  // method 7
    { const mxArray* in[] = {ds, nums, kps, thr, ratio, meth, six, md, cf, mxCreateDoubleScalar(0)};
      bad += expect_error("apsmatch:args", 3, 10, in); }                                  // maxIter <= 0
    mxArray* out[4] = {nullptr, nullptr, nullptr, nullptr};
    const mxArray* in[] = {ds, nums, kps, thr, ratio, meth, six, md, cf, it};
    mexFunction(4, out, 10, in);
    const mxArray* a12 = mxGetCell(mxGetCell(out[0], 0), 2);
    const mxArray* t12 = mxGetCell(mxGetCell(out[2], 0), 2);
    const mxArray* m12 = mxGetCell(mxGetCell(out[3], 0), 2);
    bad += !(mxGetN(out[0]) == 2 && a12 && mxGetM(a12) >= 4 && mxGetPr(mxGetCell(out[1], 0))[2] == (double)mxGetM(a12));
    bad += !(m12 && mxGetM(m12) >= mxGetM(a12) && mxGetM(m12) <= (size_t)N);  // one row per query row at most
    if (t12) {  // model maps image 2 keypoints to image 1: translation (+10, -5); column-major 3x3
      const double* t = mxGetPr(t12);
      bad += !(std::fabs(t[6] / t[8] - 10.0) < 1e-6 && std::fabs(t[7] / t[8] + 5.0) < 1e-6);
    } else {
      ++bad;
    }
    bad += !(mxGetM(mxGetCell(out[0], 1)) == 1 && mxGetCell(mxGetCell(out[0], 1), 0) == nullptr);
  } else {
    const mxArray* in[] = {ds, nums, kps, thr, ratio, meth, six, md, cf, it};
    bad += expect_error("apsmatch:nogpu", 3, 10, in);  // no CPU fallback
  }
#elif defined(GATE_MATCHF)
  mxArray* A = mxCreateNumericMatrix(6, 8, mxSINGLE_CLASS, mxREAL);
  mxArray* B = mxCreateNumericMatrix(7, 8, mxSINGLE_CLASS, mxREAL);
  mxArray* B5 = mxCreateNumericMatrix(7, 5, mxSINGLE_CLASS, mxREAL);
  mxArray* E = mxCreateNumericMatrix(0, 8, mxSINGLE_CLASS, mxREAL);
  mxArray* U = mxCreateNumericMatrix(4, 32, mxUINT8_CLASS, mxREAL);
  mxArray* U0 = mxCreateNumericMatrix(0, 32, mxUINT8_CLASS, mxREAL);
  mxArray *kf = mxCreateDoubleScalar(0), *kb = mxCreateDoubleScalar(1), *k9 = mxCreateDoubleScalar(9);
  mxArray *thr = mxCreateDoubleScalar(3.5), *ratio = mxCreateDoubleScalar(0.6), *r2 = mxCreateDoubleScalar(1.5);
  mxArray* uq = mxCreateLogicalMatrix(1, 1);
  ((unsigned char*)mxGetData(uq))[0] = 1;
  { const mxArray* in[] = {A, B, kf}; bad += expect_error("apsmatch:args", 2, 3, in); }
  { const mxArray* in[] = {A, B, k9, thr, ratio, uq}; bad += expect_error("apsmatch:args", 2, 6, in); }
  { const mxArray* in[] = {A, B, kf, thr, r2, uq}; bad += expect_error("apsmatch:args", 2, 6, in); }     // MaxRatio > 1
  { const mxArray* in[] = {A, B5, kf, thr, ratio, uq}; bad += expect_error("apsmatch:dim", 2, 6, in); }
  { const mxArray* in[] = {A, U, kf, thr, ratio, uq}; bad += expect_error("apsmatch:type", 2, 6, in); }
  { const mxArray* in[] = {A, B, kb, thr, ratio, uq}; bad += expect_error("apsmatch:type", 2, 6, in); }   // float data as bytes
  { const mxArray* in[] = {E, B, kf, thr, ratio, uq}; bad += expect_error("MATLAB:expectedNonempty", 2, 6, in); }
  {  // binary early exit (matchFeaturesScratch.m:84-88): zeros(0,2,'uint32'), zeros(0,1,'single'), no GPU touched
    mxArray* out[2] = {nullptr, nullptr};
    const mxArray* in[] = {U0, U, kb, thr, ratio, uq};
    mexFunction(2, out, 6, in);
    bad += !(mxIsUint32(out[0]) && mxGetM(out[0]) == 0 && mxGetN(out[0]) == 2 && mxIsSingle(out[1]) && mxGetM(out[1]) == 0);
  }
  if (gpu) {
    float *pa = (float*)mxGetData(A), *pb = (float*)mxGetData(B);
    // rows 0..3 of B are near copies of rows 0..3 of A (unit-scale values: no normalisation), the rest far away
    for (int r = 0; r < 6; ++r)
      for (int c = 0; c < 8; ++c) pa[r + 6 * c] = (float)(((r * 5 + c * 3) % 11) - 5) * 0.15f;
    for (int r = 0; r < 7; ++r)
      for (int c = 0; c < 8; ++c)
        pb[r + 7 * c] = r < 4 ? pa[r + 6 * c] + 0.001f * (float)(c + 1) : (float)(((r * 7 + c * 5) % 13) - 6) * 0.3f;
    mxArray* out[2] = {nullptr, nullptr};
    const mxArray* in[] = {A, B, kf, thr, ratio, uq};
    mexFunction(2, out, 6, in);
    bad += !(mxIsUint32(out[0]) && mxGetN(out[0]) == 2 && mxGetM(out[0]) >= 4 && mxIsDouble(out[1]) && mxGetM(out[1]) == mxGetM(out[0]));
    const uint32_t* m = (const uint32_t*)mxGetData(out[0]);
    const size_t K = mxGetM(out[0]);
    for (size_t r = 0; r < K; ++r)
      if (m[r] <= 4) bad += m[r + K] != m[r];                       // planted copies match their source row
    for (size_t r = 1; r < K; ++r) bad += mxGetPr(out[1])[r] < mxGetPr(out[1])[r - 1];  // Unique: ascending metric
    // packed bytes: identical sets match row to row at 0 percent, metric is single
    unsigned char* u = (unsigned char*)mxGetData(U);
    for (int i = 0; i < 4 * 32; ++i) u[i] = (unsigned char)((i * 37 + (i % 4) * 101) & 0xff);
    mxArray* o2[2] = {nullptr, nullptr};
    mxArray* t10 = mxCreateDoubleScalar(10.0);
    const mxArray* in2[] = {U, U, kb, t10, ratio, uq};
    mexFunction(2, o2, 6, in2);
    bad += !(mxGetM(o2[0]) == 4 && mxIsSingle(o2[1]) && ((const float*)mxGetData(o2[1]))[0] == 0.0f);
  } else {
    const mxArray* in[] = {A, B, kf, thr, ratio, uq};
    bad += expect_error("apsmatch:nogpu", 2, 6, in);  // no CPU fallback
  }
#endif
  std::printf(bad ? "FAILED (%d)\n" : "OK\n", bad);
  return bad ? 1 : 0;
}
