// ractip_prob.hpp -- header-only C++17 shim over the C ABI (ractip_prob.h) that
// speaks RactIP's own types.  It reproduces what RactIP::rnafold and
// RactIP::rnaduplex leave in the members RactIP::solve consumes
// (reference src/ractip.cpp:185-191, typedefs :82-85):
//
//     VF  bp      bp[offset[i]+j], 1-based, i<j            (:314-317, :365-367)
//     VI  offset  offset[i] = i*((L+1)+(L+1)-i-1)/2        (:316-317)
//     VVF up      up[i][d], 0-based start i, window i..i+d (:370-375)
//     VVF hp      hp[i][j], 1-based both                   (:393-397, :404-405, :451-453)
//
// A RactIP build swaps the three calls at src/ractip.cpp:546-548 for
// rp::ProbabilityStage::solve_probabilities(), and the body of the z-score loop
// (:1638-1657) for one solve_batch() over all shuffles (see INTEGRATION.md).
#ifndef RACTIP_PROB_HPP
#define RACTIP_PROB_HPP

#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "ractip_prob.h"

namespace rp {

typedef std::vector<float> VF;
typedef std::vector<VF> VVF;
typedef std::vector<int> VI;

struct PairProbabilities {
  VF bp1, bp2;
  VI offset1, offset2;
  VVF up1, up2;
  VVF hp;
};

class ProbabilityStage {
 public:
  // model == nullptr: the tables a default `ractip` run uses (BL* over Turner-2004).
  explicit ProbabilityStage(const rp_model* model = nullptr, int device = 0) {
    rp_model m;
    if (!model) {
      check(rp_model_default(&m, 1), nullptr);
      model = &m;
    }
    check(rp_create(&ctx_, model, device), nullptr);
    rp_opts_default(&opts_);
  }
  // All (n_gpus <= 0) or the first n_gpus visible devices behind one stage: solve_batch() then cuts the batch
  // into one contiguous block per device (rp_multi_*), which is how the z-score loop uses a multi-GPU box.
  ProbabilityStage(const rp_model* model, int /*first_device*/, int n_gpus) {
    rp_model m;
    if (!model) {
      check(rp_model_default(&m, 1), nullptr);
      model = &m;
    }
    const int rc = rp_multi_create(&multi_, model, nullptr, n_gpus);
    if (rc) throw std::runtime_error(std::string("ractip_prob: ") + rp_strerror(rc) + " -- " + rp_multi_last_error(nullptr));
    rp_opts_default(&opts_);
  }
  ~ProbabilityStage() {
    rp_destroy(ctx_);
    rp_multi_destroy(multi_);
  }
  int devices() const { return multi_ ? rp_multi_devices(multi_) : 1; }
  ProbabilityStage(const ProbabilityStage&) = delete;
  ProbabilityStage& operator=(const ProbabilityStage&) = delete;

  rp_opts& options() { return opts_; }

  // rnafold(fa1,...), rnafold(fa2,...), rnaduplex(fa1,fa2,...) of src/ractip.cpp:546-548
  void solve_probabilities(const std::string& s1, const std::string& s2, PairProbabilities& out) {
    std::vector<std::pair<std::string, std::string> > one(1, std::make_pair(s1, s2));
    std::vector<PairProbabilities> res;
    solve_batch(one, res);
    out = std::move(res[0]);
  }

  // The same under structure constraints c1 over s1, c2 over s2 (RactIP -c: the FASTA records' structure lines in
  // the alphabet .x()[] of rp_constraint; an empty string leaves its sequence unconstrained).  One context only.
  void solve_probabilities(const std::string& s1, const std::string& s2, const std::string& c1, const std::string& c2,
                           PairProbabilities& out) {
    if (!ctx_) throw std::runtime_error("ractip_prob: constrained problems run on a single-device stage");
    rp_pair pair = {s1.data(), static_cast<int>(s1.size()), s2.data(), static_cast<int>(s2.size())};
    rp_constraint con = {c1.empty() ? nullptr : c1.c_str(), c2.empty() ? nullptr : c2.c_str()};
    rp_dense_layout lay;
    size_t total = 0;
    check(rp_dense_plan(&pair, 1, &opts_, &lay, &total), ctx_);
    std::vector<float> flat(total ? total : 1);
    rp_batch* b = nullptr;
    check(rp_batch_create_constrained(ctx_, &pair, &con, 1, &opts_, &b), ctx_);
    int rc = rp_batch_run(b);
    if (!rc) rc = rp_batch_fetch_dense(b, flat.data(), flat.size());
    rp_batch_destroy(b);
    check(rc, ctx_);
    unpack(pair, lay, flat.data(), out);
  }

  // the same for a whole batch (the shuffles of src/ractip.cpp:1638-1657) in one call
  void solve_batch(const std::vector<std::pair<std::string, std::string> >& seqs, std::vector<PairProbabilities>& out) {
    const int n = static_cast<int>(seqs.size());
    std::vector<rp_pair> pairs(n);
    for (int k = 0; k < n; k++) {
      pairs[k].s1 = seqs[k].first.data();
      pairs[k].n1 = static_cast<int>(seqs[k].first.size());
      pairs[k].s2 = seqs[k].second.data();
      pairs[k].n2 = static_cast<int>(seqs[k].second.size());
    }
    std::vector<rp_dense_layout> lay(n ? n : 1);
    size_t total = 0;
    check(rp_dense_plan(pairs.data(), n, &opts_, lay.data(), &total), ctx_);
    std::vector<float> flat(total ? total : 1);
    if (multi_) {
      const int rc = rp_multi_run_dense(multi_, pairs.data(), n, &opts_, flat.data(), flat.size());
      if (rc) throw std::runtime_error(std::string("ractip_prob: ") + rp_strerror(rc) + " -- " + rp_multi_last_error(multi_));
    } else {
      check(rp_run_dense(ctx_, pairs.data(), n, &opts_, flat.data(), flat.size()), ctx_);
    }
    out.assign(n, PairProbabilities());
    for (int k = 0; k < n; k++) unpack(pairs[k], lay[k], flat.data(), out[k]);
  }

  // RactIP::rnafold(fa, bp, offset, up, max_w), src/ractip.cpp:308-382: a pair with an empty second
  // sequence computes s1's sections only.  (The reference calls it with std::max(1, max_w_), :546.)
  void rnafold(const std::string& seq, VF& bp, VI& offset, VVF& up, unsigned max_w) {
    const int keep = opts_.max_w;
    opts_.max_w = static_cast<int>(max_w < 1 ? 1 : max_w);
    PairProbabilities r;
    solve_probabilities(seq, std::string(), r);
    opts_.max_w = keep;
    bp.swap(r.bp1);
    offset.swap(r.offset1);
    up.swap(r.up1);
  }

  // RactIP::rnaduplex(fa1, fa2, hp), src/ractip.cpp:384-459
  void rnaduplex(const std::string& s1, const std::string& s2, VVF& hp) {
    PairProbabilities r;
    solve_probabilities(s1, s2, r);
    hp.swap(r.hp);
  }

 private:
  static void check(int rc, rp_ctx* ctx) {
    if (rc) throw std::runtime_error(std::string("ractip_prob: ") + rp_strerror(rc) + " -- " + rp_last_error(ctx));
  }
  // one pair's sections of a dense output buffer
  void unpack(const rp_pair& p, const rp_dense_layout& L, const float* flat, PairProbabilities& r) const {
    const int w = opts_.max_w > 0 ? opts_.max_w : 0;
    fill_bp(flat + L.bp1, p.n1, r.bp1, r.offset1);
    fill_bp(flat + L.bp2, p.n2, r.bp2, r.offset2);
    fill_rows(flat + L.up1, p.n1, w, r.up1);
    fill_rows(flat + L.up2, p.n2, w, r.up2);
    fill_rows(flat + L.hp, p.n1 + 1, p.n2 + 1, r.hp);
  }
  static void fill_bp(const float* src, int L, VF& bp, VI& offset) {
    bp.assign(src, src + static_cast<size_t>(L + 1) * (L + 2) / 2);
    offset.resize(L + 1);
    for (int i = 0; i <= L; i++) offset[i] = i * ((L + 1) + (L + 1) - i - 1) / 2;
  }
  static void fill_rows(const float* src, int rows, int cols, VVF& out) {
    out.assign(rows, VF(cols));
    for (int i = 0; i < rows; i++) out[i].assign(src + static_cast<size_t>(i) * cols, src + static_cast<size_t>(i + 1) * cols);
  }
  rp_ctx* ctx_ = nullptr;
  rp_multi* multi_ = nullptr;
  rp_opts opts_;
};

// the shuffled sequences of the z-score loop, src/ractip.cpp:1636-1643
inline void zscore_shuffles(const std::string& s1, const std::string& s2, int mode, unsigned seed, int num,
                            std::vector<std::pair<std::string, std::string> >& out) {
  std::string o1(static_cast<size_t>(num) * s1.size(), ' '), o2(static_cast<size_t>(num) * s2.size(), ' ');
  int rc = rp_zscore_shuffles(s1.data(), static_cast<int>(s1.size()), s2.data(), static_cast<int>(s2.size()), mode, seed,
                              num, 2, &o1[0], &o2[0]);
  if (rc) throw std::runtime_error(std::string("ractip_prob: ") + rp_strerror(rc));
  out.clear();
  for (int r = 0; r < num; r++) out.emplace_back(o1.substr(r * s1.size(), s1.size()), o2.substr(r * s2.size(), s2.size()));
}

}  // namespace rp
#endif
