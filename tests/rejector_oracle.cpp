// rejector_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle's ICP with a correspondence rejector chain.
//
// oracle/pcl_oracle.cpp is included unchanged; this file adds PCL 1.10's MedianDistance, OneToOne and Trimmed
// rejectors (and the Distance rejector at any place of a chain), restated from recollection like the rest of the
// oracle (include/pe_b200.h : peb_rejector, DESIGN.md section 12), and an align that applies them in the order they
// were added.  tests/rejector_oracle.py compiles it, with the oracle's parity flags, into a temporary directory.
//   score: the median rejector's DataContainer score of each pair, (src - tgt).squaredNorm() over the Vector4f maps (w = 1
//   on both sides), with the association of Eigen's 4-lane reduction: (v0 + v2) + (v1 + v3), v3 = 0 -> (dx dx + dz dz) + dy dy.
#include "../oracle/pcl_oracle.cpp"

namespace orc {

struct ScoredCorr {
  Corr c;
  float score;
};

static float median_score(const float* s, const float* t) {
  const float dx = s[0] - t[0], dy = s[1] - t[1], dz = s[2] - t[2];
  return (dx * dx + dz * dz) + dy * dy;
}

static void reject_chain(std::vector<ScoredCorr>& pairs, const peb_rejector* chain, size_t n_chain) {
  for (size_t r = 0; r < n_chain; ++r) {
    const peb_rejector& rj = chain[r];
    const size_t m = pairs.size();
    std::vector<ScoredCorr> out;
    out.reserve(m);
    if (rj.kind == PEB_REJECTOR_DISTANCE) {
      // setMaximumDistance(d): max_distance_ = d * d, a float; keep iff distance < max_distance_
      const float lim = static_cast<float>(rj.value * rj.value);
      for (const ScoredCorr& p : pairs)
        if (p.c.d2 < lim) out.push_back(p);
    } else if (rj.kind == PEB_REJECTOR_MEDIAN_DISTANCE) {
      // the scores as doubles, nth_element at m / 2 (the upper median), keep iff score <= median * factor
      if (m > 0) {
        std::vector<double> d(m);
        for (size_t k = 0; k < m; ++k) d[k] = pairs[k].score;
        std::nth_element(d.begin(), d.begin() + static_cast<std::ptrdiff_t>(m / 2), d.end());
        const double lim = d[m / 2] * rj.value;
        for (const ScoredCorr& p : pairs)
          if (static_cast<double>(p.score) <= lim) out.push_back(p);
      }
    } else if (rj.kind == PEB_REJECTOR_ONE_TO_ONE) {
      // sorted by (index_match, distance); the first pair of every target index stays.  std::sort leaves the order of
      // full ties open: the smaller source index first.  The output stays in that order.
      out = pairs;
      std::sort(out.begin(), out.end(), [](const ScoredCorr& a, const ScoredCorr& b) {
        if (a.c.m != b.c.m) return a.c.m < b.c.m;
        if (a.c.d2 != b.c.d2) return a.c.d2 < b.c.d2;
        return a.c.q < b.c.q;
      });
      size_t w = 0;
      for (size_t k = 0; k < out.size(); ++k)
        if (w == 0 || out[k].c.m != out[w - 1].c.m) out[w++] = out[k];
      out.resize(w);
    } else {  // PEB_REJECTOR_TRIMMED
      // setOverlapRatio clamps a float to [0, 1]; n_keep = max(floor(ratio * m) in float, min_correspondences); fewer than
      // m: partial_sort by distance (ties: smaller source index first) and the first n_keep, in that order
      const float ratio = std::min(1.0f, std::max(0.0f, static_cast<float>(rj.value)));
      const int n_keep = std::max(static_cast<int>(std::floor(ratio * static_cast<float>(m))), rj.min_correspondences);
      out = pairs;
      if (static_cast<size_t>(std::max(n_keep, 0)) < m) {
        std::partial_sort(out.begin(), out.begin() + n_keep, out.end(), [](const ScoredCorr& a, const ScoredCorr& b) {
          if (a.c.d2 != b.c.d2) return a.c.d2 < b.c.d2;
          return a.c.q < b.c.q;
        });
        out.resize(static_cast<size_t>(n_keep));
      }
    }
    pairs.swap(out);
  }
}

// Icp::align with the rejector chain after the correspondence loop
struct IcpChain : Icp {
  void align_ex(const void* src, size_t n, size_t stride, const M4& guess, const peb_icp_params& prm,
                const peb_rejector* chain, size_t n_chain, peb_icp_result* res, float* out_aligned, int32_t* out_idx,
                float* out_d2, IcpTrace* trace) const {
    // working cloud (input_transformed), xyz1 records
    std::vector<float> work(4 * n);
    std::vector<char> valid(n);
    bool guess_is_identity = true;
    {
      M4 I = M4::identity();
      for (int i = 0; i < 16; ++i)
        if (guess.m[i] != I.m[i]) guess_is_identity = false;
    }
    for (size_t i = 0; i < n; ++i) {
      const float* p = rec(src, i, stride);
      valid[i] = finite3(p[0], p[1], p[2]);
      work[4 * i + 0] = p[0];
      work[4 * i + 1] = p[1];
      work[4 * i + 2] = p[2];
      work[4 * i + 3] = 1.0f;
      if (!guess_is_identity && valid[i]) transform_icp(guess, p, &work[4 * i]);
    }
    M4 final_t = guess;
    M4 transformation = M4::identity();
    int nr_iterations = 0;
    bool converged = false;

    Criteria crit;
    crit.max_similar = prm.max_iterations_similar;
    crit.mse_abs = prm.abs_mse_threshold;
    crit.max_iterations = prm.max_iterations;
    crit.mse_rel = prm.euclidean_fitness_epsilon;
    crit.translation_threshold = prm.transformation_epsilon;
    crit.rotation_threshold = prm.rotation_epsilon > 0 ? prm.rotation_epsilon : 1.0 - prm.transformation_epsilon;

    const double max_dist_sqr = prm.max_corr_dist * prm.max_corr_dist;
    const bool use_rejector = prm.rejector_max_dist > 0;
    const float rej_max2 = static_cast<float>(prm.rejector_max_dist * prm.rejector_max_dist);
    const float* tn = static_cast<const float*>(tgt_normals);
    std::vector<Corr> corrs;
    corrs.reserve(n);
    std::vector<float> ms, md;
    if (out_idx)
      for (size_t i = 0; i < n; ++i) out_idx[i] = -1;
    if (out_d2)
      for (size_t i = 0; i < n; ++i) out_d2[i] = 0.0f;

    do {
      corrs.clear();
      for (size_t i = 0; i < n; ++i) {
        if (!valid[i]) continue;
        int id;
        float d2;
        if (tree.knn(&work[4 * i], 1, &id, &d2) == 0) continue;
        if (d2 > max_dist_sqr) continue;                 // determineCorrespondences: strict >
        if (use_rejector && !(d2 < rej_max2)) continue;  // CorrespondenceRejectorDistance: keep iff <
        corrs.push_back({static_cast<int>(i), id, d2});
      }
      // the rejector chain, in the order the rejectors were added (the only difference from Icp::align)
      {
        std::vector<ScoredCorr> pairs(corrs.size());
        for (size_t k = 0; k < corrs.size(); ++k)
          pairs[k] = {corrs[k], median_score(&work[4 * static_cast<size_t>(corrs[k].q)], rec(tgt, corrs[k].m, tgt_stride))};
        reject_chain(pairs, chain, n_chain);
        corrs.resize(pairs.size());
        for (size_t k = 0; k < pairs.size(); ++k) corrs[k] = pairs[k].c;
      }
      if (out_idx || out_d2) {
        if (out_idx)
          for (size_t i = 0; i < n; ++i) out_idx[i] = -1;
        if (out_d2)
          for (size_t i = 0; i < n; ++i) out_d2[i] = 0.0f;
        for (const Corr& c : corrs) {
          if (out_idx) out_idx[c.q] = c.m;
          if (out_d2) out_d2[c.q] = c.d2;
        }
      }
      if (static_cast<int>(corrs.size()) < prm.min_correspondences) {
        crit.state = PEB_NO_CORRESPONDENCES;
        converged = false;
        break;
      }
      if (prm.estimator == PEB_ESTIMATOR_SVD) {
        size_t nc = corrs.size();
        if (wide_accum) {
          std::vector<double> s(3 * nc), d(3 * nc);
          for (size_t k = 0; k < nc; ++k) {
            const float* t = rec(tgt, corrs[k].m, tgt_stride);
            for (int c = 0; c < 3; ++c) {
              s[3 * k + c] = work[4 * static_cast<size_t>(corrs[k].q) + c];
              d[3 * k + c] = t[c];
            }
          }
          transformation = umeyama<double>(s, d, nc);
        } else {
          ms.resize(3 * nc);
          md.resize(3 * nc);
          for (size_t k = 0; k < nc; ++k) {
            const float* t = rec(tgt, corrs[k].m, tgt_stride);
            for (int c = 0; c < 3; ++c) {
              ms[3 * k + c] = work[4 * static_cast<size_t>(corrs[k].q) + c];
              md[3 * k + c] = t[c];
            }
          }
          transformation = umeyama<float>(ms, md, nc);
        }
      } else {
        transformation = point_to_plane_lls(work, static_cast<const float*>(tgt), tgt_stride / 4, tn,
                                            tgt_nstride / 4, corrs);
      }
      for (size_t i = 0; i < n; ++i) {
        if (!valid[i]) continue;
        float o[3];
        transform_icp(transformation, &work[4 * i], o);
        work[4 * i] = o[0];
        work[4 * i + 1] = o[1];
        work[4 * i + 2] = o[2];
      }
      final_t = mul(transformation, final_t);
      ++nr_iterations;
      if (trace) {
        trace->increments.push_back(transformation);
        trace->ncorr.push_back(static_cast<int>(corrs.size()));
      }
      converged = crit.hasConverged(nr_iterations, transformation, corrs);
      if (trace) trace->mse.push_back(crit.cur_mse);
    } while (crit.state == PEB_NOT_CONVERGED);

    if (out_aligned) {
      for (size_t i = 0; i < n; ++i) {
        const float* p = rec(src, i, stride);
        float* o = out_aligned + 4 * i;
        o[0] = p[0];
        o[1] = p[1];
        o[2] = p[2];
        o[3] = 1.0f;
        if (finite3(p[0], p[1], p[2])) transform_icp(final_t, p, o);
      }
    }
    std::memcpy(res->T, final_t.m, sizeof(res->T));
    res->iterations = nr_iterations;
    res->converged = converged ? 1 : 0;
    res->state = crit.state;
    res->last_mse = crit.cur_mse;
    res->n_correspondences = static_cast<int32_t>(corrs.size());
    res->fitness = fitness(src, n, stride, final_t, prm.fitness_max_range, nullptr);
  }
};

}  // namespace orc

extern "C" {

ORC_API void* orc_icp_chain_create(void) { return new orc::IcpChain(); }
ORC_API void orc_icp_chain_destroy(void* h) { delete static_cast<orc::IcpChain*>(h); }
// (the handle is also an orc::Icp: orc_icp_set_target / orc_icp_set_wide_accum / orc_icp_align apply to it)
ORC_API void* orc_icp_chain_as_icp(void* h) { return static_cast<orc::Icp*>(static_cast<orc::IcpChain*>(h)); }

// the same with a rejector chain (include/pe_b200.h : peb_rejector)
ORC_API void orc_icp_align_ex(const void* h, const void* src, size_t n, size_t stride, const float* guess,
                              const peb_icp_params* prm, const peb_rejector* chain, size_t n_chain, peb_icp_result* res,
                              float* out_aligned, int32_t* out_idx, float* out_d2, float* trace_T, double* trace_mse,
                              size_t cap, size_t* trace_n) {
  orc::M4 g = orc::M4::identity();
  if (guess) std::memcpy(g.m, guess, sizeof(g.m));
  orc::IcpTrace tr;
  static_cast<const orc::IcpChain*>(h)->align_ex(src, n, stride, g, *prm, chain, n_chain, res, out_aligned, out_idx,
                                                  out_d2, (trace_T || trace_mse) ? &tr : nullptr);
  size_t cnt = std::min(cap, tr.increments.size());
  for (size_t i = 0; i < cnt; ++i) {
    if (trace_T) std::memcpy(trace_T + 16 * i, tr.increments[i].m, 16 * sizeof(float));
    if (trace_mse) trace_mse[i] = tr.mse[i];
  }
  if (trace_n) *trace_n = cnt;
}

ORC_API void orc_icp_align_batch_ex(const void* h, const void* src, size_t n, size_t stride, const float* guesses,
                                    size_t H, const peb_icp_params* prm, const peb_rejector* chain, size_t n_chain,
                                    peb_icp_result* res, int threads) {
#ifdef _OPENMP
  if (threads <= 0) threads = omp_get_max_threads();
#pragma omp parallel for num_threads(threads) schedule(dynamic, 1)
#endif
  for (int64_t i = 0; i < static_cast<int64_t>(H); ++i) {
    orc::M4 g;
    std::memcpy(g.m, guesses + 16 * i, sizeof(g.m));
    static_cast<const orc::IcpChain*>(h)->align_ex(src, n, stride, g, *prm, chain, n_chain, &res[i], nullptr, nullptr,
                                                   nullptr, nullptr);
  }
  (void)threads;
}

// the chain over a scripted pair set: q (source), m (target), d2, score (the median rejector's) per pair, in order;
// out_k (capacity n): which input pairs are left, in the order the chain leaves them; returns their count
ORC_API size_t orc_reject_pairs(const int32_t* q, const int32_t* m, const float* d2, const float* score, size_t n,
                                const peb_rejector* chain, size_t n_chain, int32_t* out_k) {
  std::vector<orc::ScoredCorr> pairs(n);
  for (size_t k = 0; k < n; ++k) pairs[k] = {{q[k], m[k], d2[k]}, score[k]};
  std::vector<int> pos_of_q;  // scripted q are unique: map back to the input position
  for (size_t k = 0; k < n; ++k) {
    if (static_cast<size_t>(q[k]) >= pos_of_q.size()) pos_of_q.resize(static_cast<size_t>(q[k]) + 1, -1);
    pos_of_q[static_cast<size_t>(q[k])] = static_cast<int>(k);
  }
  orc::reject_chain(pairs, chain, n_chain);
  for (size_t k = 0; k < pairs.size(); ++k) out_k[k] = pos_of_q[static_cast<size_t>(pairs[k].c.q)];
  return pairs.size();
}

}  // extern "C"
