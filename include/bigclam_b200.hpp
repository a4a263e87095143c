// bigclam_b200.hpp — header-only C++17 mirror of the reference's spark-shell surface over the C ABI (bigclam_b200.h).
//
// The reference's host side is JVM code (three Scala scripts); the image has no JVM, so the compiled host mirror is C++
// (the Python one is bigclam_apachespark_b200/driver.py — same names, same argument meaning).  Script-level names are
// kept so that a driver reads like the script:
//
//   script (codes/bigclam4-7.scala)                              here
//   numCore/minCom/maxCom/divCom/alpha/beta/MaxInter  :14-26     public members of BigClam (same defaults)
//   GraphLoader.edgeListFile + collectNeighborIds     :45,50-51  load_edge_list / set_graph
//   conductanceLocalMin()                             :58-73     conductanceLocalMin()
//   initNeighborComF(K)                               :81-108    initNeighborComF(K)
//   Kset()                                            :116-133   Kset()
//   backtrackingLineSearchs(uset)                     :152-223   backtrackingLineSearchs(uset)
//   loglikelihood()           bigclamv3-7.scala:106-120          loglikelihood()
//   SGDFindC()                                        :225-243   SGDFindC()
//   MBSGD()       bigclamv3-7.scala:206-222, Bigclamv2.scala:203-219   MBSGD(version)
//   K sweep                                           :244-266   sweep_K()
//   community extraction         Bigclamv2.scala:223-230         delta_threshold(), extract(delta)
//
// Errors: the reference throws JVM exceptions; here every negative return code of the C ABI becomes a bigclam::Error
// (std::runtime_error carrying the code and bigclam_last_error()).  There is no CPU path: without a CUDA device
// set_K() throws BIGCLAM_ECUDA.  One BigClam is driven by one thread at a time (like the script's driver thread).
#ifndef BIGCLAM_B200_HPP
#define BIGCLAM_B200_HPP

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "bigclam_b200.h"

namespace bigclam {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &msg) : std::runtime_error("bigclam_b200 error " + std::to_string(c) + ": " + msg), code(c) {}
};

// Geometric grid of K values (:116-133).  `maxCom / minCom` is an Int division in the script (both are Int vars): the
// pasted REPL value at :268 is only reproduced with that quirk, so it is the default.
inline std::vector<int> Kset(int minCom, int maxCom, int divCom, bool int_division = true) {
    const double ratio = int_division ? (double)(maxCom / minCom) : (double)maxCom / (double)minCom;
    const double conGap = std::exp(std::log(ratio) / divCom);
    std::vector<int> ks{minCom};
    for (int x = minCom;;) {
        int next = (int)(x * conGap);
        if (next == x) ++next;
        x = next;
        if (x >= maxCom) break;
        ks.push_back(x);
    }
    ks.push_back(maxCom);
    return ks;
}

class BigClam {
public:
    // script variables (:14-26), the script's values as defaults
    int numCore = 36;                                // :14 (Spark parallelism; informational here: numGPUs plays that role)
    int minCom = 1000, maxCom = 9000, divCom = 100;
    double alpha = 0.05, beta = 0.1;
    int MaxInter = 15;
    // outcome of the most recent call
    int64_t last_n_updated = 0, last_calls = 0;
    std::vector<double> last_trace;                  // LLH returned by every hot-path call of the last SGDFindC / MBSGD

    explicit BigClam(int numGPUs = 1, int device = 0, bool sparse_rows = true, bool exhaustive_linesearch = false)
        : world_(numGPUs), device_(device),
          flags_((sparse_rows || numGPUs > 1 ? BIGCLAM_F_SPARSE_ROWS : 0) | (exhaustive_linesearch ? BIGCLAM_F_LS_EXHAUSTIVE : 0)) {}
    BigClam(const BigClam &) = delete;
    BigClam &operator=(const BigClam &) = delete;
    ~BigClam() { close(); }

    void close() {
        if (ctx_ != nullptr) bigclam_destroy(ctx_);
        if (multi_ != nullptr) bigclam_multi_destroy(multi_);
        ctx_ = nullptr;
        multi_ = nullptr;
    }

    // GraphLoader.edgeListFile + collectNeighborIds(Either) (:45,50-51).  dedup: simple undirected graph; false = one
    // neighbour entry per edge line and endpoint (literal GraphX).  Vertex ids are relabelled 0..n-1 in ascending order.
    BigClam &load_edge_list(const std::string &path, bool dedup = true) {
        bigclam_graph g{};
        char err[512] = {0};
        const int rc = bigclam_graph_read_edgelist(path.c_str(), dedup ? 1 : 0, &g, err, (int64_t)sizeof(err));
        if (rc != BIGCLAM_OK) throw Error(rc, err);
        ids.assign(g.ids, g.ids + g.n);
        set_graph(g.n, g.rowptr, g.col);
        bigclam_graph_free(&g);
        return *this;
    }
    BigClam &set_graph(int64_t n, const int64_t *rowptr, const int32_t *col) {
        close();
        n_ = n;
        rowptr_.assign(rowptr, rowptr + n + 1);
        col_.assign(col, col + rowptr[n]);
        Sbc.clear();
        return *this;
    }

    // K = sc.broadcast(i) (:249): (re)creates the device context for this K.
    BigClam &set_K(int K) {
        close();
        bigclam_params p;
        check(bigclam_default_params(&p, K), "bigclam_default_params");
        p.alpha = alpha;
        p.beta = beta;
        p.max_inter = MaxInter;
        p.device = device_;
        p.flags = flags_;
        if (world_ > 1) {
            const int rc = bigclam_multi_create(&multi_, n_, rowptr_.data(), col_.data(), &p, world_, nullptr);
            if (rc != BIGCLAM_OK) throw Error(rc, str(bigclam_multi_last_error(nullptr)));
        } else {
            const int rc = bigclam_create(&ctx_, n_, rowptr_.data(), col_.data(), &p);
            if (rc != BIGCLAM_OK) throw Error(rc, str(bigclam_last_error(nullptr)));
        }
        K_ = K;
        return *this;
    }

    // F <- n x K row-major; sumF <- column sums (:105-107), or an injected sumF (the script never recomputes it, :192)
    BigClam &set_F(const std::vector<double> &F, const std::vector<double> *sumF = nullptr) {
        need();
        if ((int64_t)F.size() != n_ * K_) throw Error(BIGCLAM_EINVAL, "F must be n x K");
        check(multi_ ? bigclam_multi_set_F(multi_, F.data()) : bigclam_set_F(ctx_, F.data()), "set_F");
        if (sumF != nullptr) check(multi_ ? bigclam_multi_set_sumF(multi_, sumF->data()) : bigclam_set_sumF(ctx_, sumF->data()), "set_sumF");
        return *this;
    }
    std::vector<double> F() {
        need();
        std::vector<double> out((size_t)(n_ * K_));
        check(multi_ ? bigclam_multi_get_F(multi_, 0, out.data()) : bigclam_get_F(ctx_, out.data()), "get_F");
        return out;
    }
    std::vector<double> sumF() {
        need();
        std::vector<double> out((size_t)K_);
        check(multi_ ? bigclam_multi_get_sumF(multi_, 0, out.data()) : bigclam_get_sumF(ctx_, out.data()), "get_sumF");
        return out;
    }

    // conductanceLocalMin() (:58-73): ranked seed candidates `Sbc` (:75) and every vertex's ego-net conductance.
    const std::vector<int32_t> &conductanceLocalMin(bool on_gpu = true) {
        conductance.assign((size_t)n_, 0.0);
        Sbc.assign((size_t)n_, 0);
        int64_t cnt = 0;
        const int rc = on_gpu ? bigclam_conductance_seeds_gpu(n_, rowptr_.data(), col_.data(), device_, conductance.data(), Sbc.data(), &cnt)
                              : bigclam_conductance_seeds(n_, rowptr_.data(), col_.data(), conductance.data(), Sbc.data(), &cnt);
        if (rc != BIGCLAM_OK) throw Error(rc, "bigclam_conductance_seeds failed");
        Sbc.resize((size_t)cnt);
        return Sbc;
    }
    // initNeighborComF(K) (:81-108): builds F0 from the ranked seeds and loads it.
    std::vector<double> initNeighborComF(int K, bool include_self = false, uint64_t pad_seed = 1234) {
        if (Sbc.empty()) conductanceLocalMin();
        if (K != K_ || (ctx_ == nullptr && multi_ == nullptr)) set_K(K);
        std::vector<double> F0((size_t)(n_ * K));
        const int rc = bigclam_init_neighbor_com_F(n_, rowptr_.data(), col_.data(), K, Sbc.data(), (int64_t)Sbc.size(), include_self ? 1 : 0,
                                                   pad_seed, F0.data());
        if (rc != BIGCLAM_OK) throw Error(rc, "bigclam_init_neighbor_com_F failed");
        set_F(F0);
        return F0;
    }

    // ---- the hot path (:152-223).  uset: nullptr = all vertices (what the script always passes, :227)
    double backtrackingLineSearchs(const std::vector<int64_t> *uset = nullptr) {
        need();
        std::vector<uint8_t> mask;
        if (uset != nullptr) {
            mask.assign((size_t)n_, 0);
            for (int64_t u : *uset) mask.at((size_t)u) = 1;
        }
        double llh = 0.0;
        const uint8_t *m = uset != nullptr ? mask.data() : nullptr;
        check(multi_ ? bigclam_multi_step(multi_, m, &llh, &last_n_updated) : bigclam_step(ctx_, m, &llh, &last_n_updated), "step");
        return llh;
    }
    double loglikelihood() {
        need();
        double llh = 0.0;
        check(multi_ ? bigclam_multi_loglikelihood(multi_, &llh) : bigclam_loglikelihood(ctx_, &llh), "loglikelihood");
        return llh;
    }
    // :225-243: one call for LLHold, then until |1 - new/old| < 1e-4; returns what the script returns (:242).
    double SGDFindC(double rel_tol = 1e-4, int64_t max_outer = 0) { return run(4, rel_tol, max_outer); }
    void MBSGD(int version = 3, double rel_tol = 1e-4, int64_t max_outer = 0) {
        if (version != 2 && version != 3) throw Error(BIGCLAM_EINVAL, "version must be 2 or 3");
        run(version, rel_tol, max_outer);
    }

    // Held-out pairs (bigclam_set_holdout: sparse rows, one GPU): the masked objective from now on; an empty ho_rowptr
    // clears the lists.  holdout_loglikelihood(): L_HO of the current F (n_pairs: unordered pairs scored).
    void set_holdout(const std::vector<int64_t> &ho_rowptr, const std::vector<int32_t> &ho_col, const std::vector<uint8_t> &ho_is_edge) {
        need();
        if (multi_ != nullptr) throw Error(BIGCLAM_EUNSUPPORTED, "set_holdout: single-GPU contexts only");
        if (ho_rowptr.empty()) { check(bigclam_set_holdout(ctx_, nullptr, nullptr, nullptr), "set_holdout"); return; }
        if ((int64_t)ho_rowptr.size() != n_ + 1 || (int64_t)ho_col.size() != ho_rowptr.back() || ho_is_edge.size() != ho_col.size())
            throw Error(BIGCLAM_EINVAL, "set_holdout: the arrays do not describe n rows");
        check(bigclam_set_holdout(ctx_, ho_rowptr.data(), ho_col.data(), ho_is_edge.data()), "set_holdout");
    }
    double holdout_loglikelihood(int64_t *n_pairs = nullptr) {
        need();
        if (multi_ != nullptr) throw Error(BIGCLAM_EUNSUPPORTED, "holdout_loglikelihood: single-GPU contexts only");
        double llh = 0.0;
        check(bigclam_holdout_loglikelihood(ctx_, &llh, n_pairs), "holdout_loglikelihood");
        return llh;
    }

    // Community extraction as coded in Bigclamv2.scala:223-230.  delta_threshold: `e = 2.0*count/(N*(N-1)); sqrt(-log(1-e))`
    // (:223-224; in the script `count` is the number of vertices that have edges, the thesis uses |E|: pass what you mean).
    // extract(): communities[c] = vertices u with F_uc >= delta, or, when the row maximum is below delta, with F_uc equal to
    // the row maximum (:227); the flatMap / groupByKey of :229-230 is the regrouping by community id done here.
    static double delta_threshold(int64_t n_vertices, int64_t count) {
        const double e = 2.0 * (double)count / ((double)n_vertices * ((double)n_vertices - 1.0));
        return std::sqrt(-std::log(1.0 - e));
    }
    std::vector<std::vector<int32_t>> extract(double delta) {
        need();
        if (multi_ != nullptr) throw Error(BIGCLAM_EUNSUPPORTED, "extract: single-GPU contexts only (read F() and regroup on the host)");
        std::vector<uint8_t> member((size_t)(n_ * K_));
        std::vector<double> fmax((size_t)n_);
        check(bigclam_extract(ctx_, delta, member.data(), fmax.data()), "extract");
        std::vector<std::vector<int32_t>> comms((size_t)K_);
        for (int64_t u = 0; u < n_; ++u)
            for (int c = 0; c < K_; ++c)
                if (member[(size_t)(u * K_ + c)]) comms[(size_t)c].push_back((int32_t)u);
        return comms;
    }

    std::vector<int> Kset() const { return bigclam::Kset(minCom, maxCom, divCom); }
    // The K sweep (:244-266): for K in Kset: initNeighborComF(K), SGDFindC(); stops at the first K whose gain
    // `1 - new/old` is below 0.1 %.  As coded LLHKold starts at 0.0, so the first K never stops the sweep.
    // Returns KforC (0 when the grid ran out, :245) and fills hist with (K, LLH).
    int sweep_K(std::vector<std::pair<int, double>> *hist = nullptr, double rel_gain = 0.001, int64_t max_outer = 0) {
        double LLHKold = 0.0;
        for (int k : Kset()) {
            initNeighborComF(k);
            const double LLHKnew = SGDFindC(1e-4, max_outer);
            if (hist != nullptr) hist->emplace_back(k, LLHKnew);
            if (1.0 - LLHKnew / LLHKold < rel_gain) return k;          // (x / 0.0 = -inf or nan: never below, like the JVM)
            LLHKold = LLHKnew;
        }
        return 0;
    }

    int64_t n() const { return n_; }
    int K() const { return K_; }
    std::vector<int64_t> ids;                         // original vertex id of dense index i (load_edge_list)
    std::vector<int32_t> Sbc;                         // ranked seeds (:75)
    std::vector<double> conductance;

private:
    double run(int variant, double rel_tol, int64_t max_outer) {
        need();
        std::vector<double> trace(65536);
        double llh = 0.0;
        check(multi_ ? bigclam_multi_run(multi_, variant, rel_tol, max_outer, &llh, &last_calls, trace.data(), (int64_t)trace.size())
                     : bigclam_run(ctx_, variant, rel_tol, max_outer, &llh, &last_calls, trace.data(), (int64_t)trace.size()),
              "run");
        trace.resize((size_t)std::min<int64_t>(last_calls, (int64_t)trace.size()));
        last_trace = std::move(trace);
        return llh;
    }
    void need() const {
        if (ctx_ == nullptr && multi_ == nullptr) throw Error(BIGCLAM_EINVAL, "no context: call set_graph()/load_edge_list() and set_K() first");
    }
    static std::string str(const char *s) { return s != nullptr ? s : "unknown error"; }
    void check(int rc, const char *what) const {
        if (rc == BIGCLAM_OK) return;
        const char *msg = multi_ ? bigclam_multi_last_error(multi_) : bigclam_last_error(ctx_);
        throw Error(rc, std::string(what) + ": " + str(msg));
    }

    int world_, device_, flags_;
    int64_t n_ = 0;
    int K_ = 0;
    std::vector<int64_t> rowptr_;
    std::vector<int32_t> col_;
    bigclam_ctx *ctx_ = nullptr;
    bigclam_multi *multi_ = nullptr;
};

}  // namespace bigclam
#endif  // BIGCLAM_B200_HPP
