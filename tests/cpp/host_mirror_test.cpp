// C++ host-mirror test (include/nova_b200.hpp).  Reads a case file written by the Python test
// (inputs + oracle answers), runs the calls through the C++ layer -- including COMMITS ISSUED
// CONCURRENTLY FROM SEVERAL THREADS, as rayon workers do in the reference (r1cs/mod.rs:509-512) --
// and prints OK / MISMATCH lines.  Usage: host_mirror_test <case.bin>      (needs a GPU)
//        host_mirror_test --compile-check                                   (no GPU: links only)
#include <cstdio>
#include <fstream>
#include <memory>
#include <thread>

#include "../../include/nova_b200.hpp"
using namespace nova::b200;

template <class T>
static std::vector<T> rd(std::ifstream& f) {
  uint64_t n;
  f.read((char*)&n, 8);
  std::vector<T> v(n);
  f.read((char*)v.data(), n * sizeof(T));
  return v;
}

// --fold <case.bin>: the device-resident folding step through the C++ layer (R1CSShapeDev::commit_T,
// fold_witness_resident, WitnessStream, validate_key); the Python test checks the dumped results against
// the oracle.  Case file: A, B, C as (data, indices, indptr), then W1, E1, W2, X1, X2, [u1, u_sum, r, r_T, r_W],
// bases, h.
static SparseMatrix* read_matrix(std::ifstream& f, int field, size_t cols) {
  auto data = rd<Scalar>(f);
  auto idx = rd<uint64_t>(f);
  auto ptr = rd<uint64_t>(f);
  return new SparseMatrix(field, data, idx, ptr, cols);
}
static int fold_mode(const char* path) {
  std::ifstream f(path, std::ios::binary);
  check(b200_init(0), "b200_init");
  const int field = BN254::scalar_field;
  auto dims = rd<uint64_t>(f);  // num_cons, num_vars, num_io
  const size_t num_cons = dims[0], num_vars = dims[1], num_io = dims[2], cols = num_vars + 1 + num_io;
  std::unique_ptr<SparseMatrix> A(read_matrix(f, field, cols)), B(read_matrix(f, field, cols)), C(read_matrix(f, field, cols));
  auto W1 = rd<Scalar>(f), E1 = rd<Scalar>(f), W2 = rd<Scalar>(f), X1 = rd<Scalar>(f), X2 = rd<Scalar>(f), sc = rd<Scalar>(f);
  auto bases = rd<Affine>(f);
  auto h = rd<Affine>(f);
  const Scalar &u1 = sc[0], &u_sum = sc[1], &r = sc[2], &r_T = sc[3], &r_W = sc[4], &one = sc[5];
  // the key arrives "from a file": validated on the device before its tables are built
  CommitmentKey<BN254> ck(CommitmentKey<BN254>::Untrusted{}, bases, &h[0]);
  uint64_t rejected_at = UINT64_MAX;  // ... and a copy with one corrupted point is refused with that point's index
  {
    auto broken = bases;
    broken[bases.size() / 2].y.limbs[0] ^= 1;
    try {
      CommitmentKey<BN254> nope(CommitmentKey<BN254>::Untrusted{}, broken, &h[0]);
    } catch (const CommitmentKey<BN254>::InvalidCommitmentKey& e) {
      rejected_at = e.index;
    }
  }
  R1CSShapeDev S{*A, *B, *C, field, num_cons, num_vars, num_io};
  size_t bad = validate_key<BN254>(bases);
  // the fresh witness arrives through the stream in three ragged chunks
  WitnessStream<BN254> ws(ck, num_vars);
  size_t c1 = num_vars / 3, c2 = num_vars / 2;
  ws.append(W2.data(), c1);
  ws.append(W2.data() + c1, c2 - c1);
  ws.append(W2.data() + c2, num_vars - c2);
  void* dW2 = nullptr;
  Point comm_W2 = ws.finish(&r_W, &dW2);
  DeviceVec W2d(W2), W1d(W1), E1d(E1);
  DeviceVec Z1 = S.z(W1d, u1, X1), Z2 = S.z(W2d, one, X2);
  auto tc = S.commit_T(ck, Z1, Z2, u_sum, E1d, nullptr, &r_T);
  RelaxedR1CSWitnessDev run{std::move(W1d), std::move(E1d)};
  RelaxedR1CSWitnessDev folded = fold_witness_resident(field, run, W2d, tc.first, r);
  auto T = tc.first.to_host(), Wf = folded.W.to_host(), Ef = folded.E.to_host();
  std::ofstream o(std::string(path) + ".out", std::ios::binary);
  auto dump = [&](const void* p, uint64_t n, size_t sz) { o.write((char*)&n, 8); o.write((const char*)p, n * sz); };
  uint64_t b64 = bad;
  dump(&b64, 1, 8);
  dump(&rejected_at, 1, 8);
  dump(&comm_W2, 1, 96);
  dump(&tc.second, 1, 96);
  dump(T.data(), T.size(), 32);
  dump(Wf.data(), Wf.size(), 32);
  dump(Ef.data(), Ef.size(), 32);
  std::printf("fold ok\n");
  return 0;
}

// --sumcheck <case.bin>: the two fused sum-check loops through the C++ wrappers (prove_quad_prod,
// prove_cubic_with_three_inputs with a TranscriptState carrying pending absorbs); dumps every prover message and the
// transcript afterwards for the Python test to compare with the oracle.  Case: [l], A, B, C, taus, [claim_q, claim_c],
// transcript (72 bytes as 9 u64), pending bytes.
static int sumcheck_mode(const char* path) {
  std::ifstream f(path, std::ios::binary);
  check(b200_init(0), "b200_init");
  const int field = BN254::scalar_field;
  auto dims = rd<uint64_t>(f);
  auto A = rd<Scalar>(f), B = rd<Scalar>(f), C = rd<Scalar>(f), taus = rd<Scalar>(f), claims = rd<Scalar>(f);
  auto trw = rd<uint64_t>(f);
  auto pending = rd<unsigned char>(f);
  const int l = (int)dims[0];
  std::ofstream o(std::string(path) + ".out", std::ios::binary);
  auto dump = [&](const void* p, uint64_t n, size_t sz) { o.write((char*)&n, 8); o.write((const char*)p, n * sz); };
  for (int which = 0; which < 2; which++) {
    TranscriptState t;
    memcpy(&t.tr, trw.data(), sizeof(b200_transcript));
    t.pending = pending;
    DeviceVec dA(A), dB(B), dC(C);
    SumcheckProofOut out = which == 0 ? prove_quad_prod(field, claims[0], l, dA.ptr(), dB.ptr(), t)
                                      : prove_cubic_with_three_inputs(field, claims[1], taus, dA.ptr(), dB.ptr(), dC.ptr(), t);
    std::vector<Scalar> flat;
    for (auto& q : out.compressed_polys) flat.insert(flat.end(), q.begin(), q.end());
    dump(flat.data(), flat.size(), 32);
    dump(out.r.data(), out.r.size(), 32);
    dump(out.final_evals.data(), out.final_evals.size(), 32);
    dump(&t.tr, 1, sizeof(b200_transcript));
    uint64_t left = t.pending.size();
    dump(&left, 1, 8);
  }
  std::printf("sumcheck ok\n");
  return 0;
}

// --concurrency <log2n> <threads> <points.bin>: the same `threads` commitments issued from ONE thread one after the other
// and from `threads` threads at once (what rayon does in the reference: src/spartan/ppsnark.rs:457-470); the results must
// be the same points (written to points.bin) and the ratio of the two wall times is printed.  Synthetic key, pinned host
// scalars.
#include <chrono>
static int concurrency_mode(int log2n, int nthreads, const char* points_path) {
  check(b200_init(0), "b200_init");
  const size_t n = (size_t)1 << log2n;
  // generator of BN254 G1 (1, 2) in Montgomery form is not needed here: any valid affine point works as the seed of
  // the synthetic key -- take it from a one-point key the library builds from the curve generator it is given
  unsigned char gen[64] = {0};
  {  // (1, 2) in Montgomery form: R mod q and 2R mod q for BN254 Fq
    const uint64_t one[4] = {0xd35d438dc58f0d9dull, 0x0a78eb28f5c70b3dull, 0x666ea36f7879462cull, 0x0e0a77c19a07df2full};
    const uint64_t two[4] = {0xa6ba871b8b1e1b3aull, 0x14f1d651eb8e167bull, 0xccdd46def0f28c58ull, 0x1c14ef83340fbe5eull};
    memcpy(gen, one, 32);
    memcpy(gen + 32, two, 32);
  }
  uint64_t ck = 0;
  check(b200_ck_setup_synthetic(0, gen, 0x5EED, n, 0, 0, &ck), "ck_setup_synthetic");
  std::vector<void*> bufs(nthreads);
  for (int t = 0; t < nthreads; t++) {
    check(b200_host_alloc(32 * n, &bufs[t]), "host_alloc");
    uint64_t* w = (uint64_t*)bufs[t];
    uint64_t x = 0x9E3779B97F4A7C15ull * (t + 1);
    for (size_t i = 0; i < 4 * n; i++) {  // xorshift words; top limb masked below the modulus
      x ^= x << 13; x ^= x >> 7; x ^= x << 17;
      w[i] = (i % 4 == 3) ? (x & 0x0FFFFFFFFFFFFFFFull) : x;
    }
  }
  std::vector<Point> serial(nthreads), conc(nthreads);
  auto commit = [&](int t, Point* out) { check(b200_commit(ck, bufs[t], n, nullptr, out), "commit"); };
  for (int t = 0; t < nthreads; t++) commit(t, &serial[t]);  // warm-up (workspaces)
  {
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; t++) th.emplace_back([&, t] { commit(t, &conc[t]); });
    for (auto& x : th) x.join();
  }
  const int reps = 5;
  auto t0 = std::chrono::steady_clock::now();
  for (int r = 0; r < reps; r++)
    for (int t = 0; t < nthreads; t++) commit(t, &serial[t]);
  auto t1 = std::chrono::steady_clock::now();
  for (int r = 0; r < reps; r++) {
    std::vector<std::thread> th;
    for (int t = 0; t < nthreads; t++) th.emplace_back([&, t] { commit(t, &conc[t]); });
    for (auto& x : th) x.join();
  }
  auto t2 = std::chrono::steady_clock::now();
  double ms_serial = std::chrono::duration<double, std::milli>(t1 - t0).count() / reps;
  double ms_conc = std::chrono::duration<double, std::milli>(t2 - t1).count() / reps;
  // same points?  compare cross-multiplied (Jacobian coordinates differ between runs): done by the Python side from the dump
  std::printf("{\"what\": \"%d commits of 2^%d scalars, serial vs %d threads\", \"ms_serial\": %.4f, \"ms_concurrent\": %.4f, "
              "\"speedup\": %.3f}\n", nthreads, log2n, nthreads, ms_serial, ms_conc, ms_serial / ms_conc);
  FILE* f = std::fopen(points_path, "wb");
  if (!f) {
    std::fprintf(stderr, "cannot write %s\n", points_path);
    return 1;
  }
  std::fwrite(serial.data(), sizeof(Point), nthreads, f);
  std::fwrite(conc.data(), sizeof(Point), nthreads, f);
  std::fclose(f);
  for (void* b : bufs) b200_host_free(b);
  b200_ck_release(ck);
  return 0;
}

// --mgpu <case.bin> <ndev>: MultiGpuCommitmentKey (one process, ndev devices -- virtual devices on one GPU are allowed) against
// the single-device CommitmentKey on the same key and vectors; dumps both sets of points for the Python side.
static int mgpu_mode(const char* path, int ndev) {
  std::ifstream f(path, std::ios::binary);
  check(b200_init(0), "b200_init");
  auto bases = rd<Affine>(f);
  auto h = rd<Affine>(f);
  auto scalars = rd<Scalar>(f);
  auto r = rd<Scalar>(f);
  std::vector<int> devs(ndev, 0);  // all on device 0 unless the box has more
  int have = 0;
  b200_device_count(&have);
  for (int d = 0; d < ndev; d++) devs[d] = have > 1 ? d % have : 0;
  MultiGpuCommitmentKey<BN254> mk(bases, &h[0], ndev, devs);
  CommitmentKey<BN254> ck(bases, &h[0]);
  std::vector<Point> a, b;
  for (size_t len : {scalars.size(), scalars.size() / 2 + 1, (size_t)1, (size_t)0}) {
    std::vector<Scalar> v(scalars.begin(), scalars.begin() + len);
    a.push_back(mk.commit(v, &r[0]));
    b.push_back(CommitmentEngine<BN254>::commit(ck, v, &r[0]));
    a.push_back(mk.commit(v));
    b.push_back(DlogGroup<BN254>::vartime_multiscalar_mul(v, ck));
  }
  std::ofstream o(std::string(path) + ".out", std::ios::binary);
  uint64_t n = a.size();
  o.write((char*)&n, 8);
  o.write((char*)a.data(), n * sizeof(Point));
  o.write((char*)b.data(), n * sizeof(Point));
  std::printf("mgpu ok %d devices\n", ndev);
  return 0;
}

// Jacobian -> compare with expected affine without inversion: X == x*Z^2, Y == y*Z^3 is checked on
// the Python side; here we only dump the raw result bytes.
int main(int argc, char** argv) {
  if (argc < 2) return 2;
  if (std::string(argv[1]) == "--compile-check") {
    std::printf("compiled against %s\n", b200_version());
    return 0;
  }
  if (std::string(argv[1]) == "--fold") return argc > 2 ? fold_mode(argv[2]) : 2;
  if (std::string(argv[1]) == "--sumcheck") return argc > 2 ? sumcheck_mode(argv[2]) : 2;
  if (std::string(argv[1]) == "--mgpu") return argc > 3 ? mgpu_mode(argv[2], std::atoi(argv[3])) : 2;
  if (std::string(argv[1]) == "--concurrency")
    return argc > 4 ? concurrency_mode(std::atoi(argv[2]), std::atoi(argv[3]), argv[4]) : 2;
  std::ifstream f(argv[1], std::ios::binary);
  check(b200_init(0), "b200_init");
  auto bases = rd<Affine>(f);
  auto h = rd<Affine>(f);
  auto scalars = rd<Scalar>(f);
  auto r = rd<Scalar>(f);
  CommitmentKey<BN254> ck(bases, &h[0]);
  // 1) single commit with blind, 2) 8 threads x 4 concurrent commits of different prefixes
  std::vector<Point> results;
  results.push_back(CommitmentEngine<BN254>::commit(ck, scalars, &r[0]));
  const int NT = 8, PER = 4;
  std::vector<Point> conc(NT * PER);
  std::vector<std::thread> th;
  for (int t = 0; t < NT; t++)
    th.emplace_back([&, t] {
      for (int k = 0; k < PER; k++) {
        size_t len = scalars.size() / (1 + (t * PER + k) % 5);
        std::vector<Scalar> v(scalars.begin(), scalars.begin() + len);
        conc[t * PER + k] = DlogGroup<BN254>::vartime_multiscalar_mul(v, ck);
      }
    });
  for (auto& x : th) x.join();
  results.insert(results.end(), conc.begin(), conc.end());
  // 3) length mismatch must throw logic_error (msm.rs:226)
  bool threw = false;
  try {
    std::vector<Scalar> too_long(bases.size() + 1);
    DlogGroup<BN254>::vartime_multiscalar_mul(too_long, ck);
  } catch (const std::logic_error&) { threw = true; }
  // 4) fold + bind through the mirror
  auto folded = fold_witness(BN254::scalar_field, scalars, scalars, r[0]);
  std::vector<Scalar> z(scalars.begin(), scalars.begin() + (scalars.size() & ~(size_t)1));
  bind_poly_var_top(BN254::scalar_field, z, r[0]);
  std::ofstream o(std::string(argv[1]) + ".out", std::ios::binary);
  uint64_t n = results.size();
  o.write((char*)&n, 8);
  o.write((char*)results.data(), n * sizeof(Point));
  n = folded.size(); o.write((char*)&n, 8); o.write((char*)folded.data(), n * 32);
  n = z.size(); o.write((char*)&n, 8); o.write((char*)z.data(), n * 32);
  std::printf("threw=%d results=%zu\n", (int)threw, results.size());
  return threw ? 0 : 1;
}
