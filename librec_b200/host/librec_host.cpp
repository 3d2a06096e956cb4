// Host-side mirror of the reference's recommender plugin interface; see librec_host.hpp.
#include "librec_host.hpp"
#include <sys/stat.h>
#include <dirent.h>
#include <deque>
#include <unordered_map>
#include <string_view>

#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <set>
#include <sstream>

namespace librec {

// ------------------------------------------------------------------------------------------------
// Java number formatting (the per-iteration log line concatenates a double and a float:
// recommender/AbstractRecommender.java:253-257)
// ------------------------------------------------------------------------------------------------
template <typename T>
static std::string java_fp_to_string(T v) {
    if (std::isnan(v)) return "NaN";
    if (std::isinf(v)) return v > 0 ? "Infinity" : "-Infinity";
    if (v == 0) return std::signbit(v) ? "-0.0" : "0.0";
    char buf[64];
    auto r = std::to_chars(buf, buf + sizeof buf, v, std::chars_format::scientific);   // shortest round-trip digits
    std::string s(buf, r.ptr);                       // d[.ddd]e[+-]XX
    const size_t epos = s.find('e');
    std::string mant = s.substr(0, epos);
    const int exp10 = std::stoi(s.substr(epos + 1));
    bool neg = false;
    if (mant[0] == '-') { neg = true; mant = mant.substr(1); }
    std::string digits;
    for (char c : mant) if (c != '.') digits.push_back(c);
    std::string out;
    const double a = std::fabs((double)v);
    if (a >= 1e-3 && a < 1e7) {
        if (exp10 >= 0) {
            std::string ip = digits.substr(0, std::min((size_t)exp10 + 1, digits.size()));
            while ((int)ip.size() < exp10 + 1) ip.push_back('0');
            std::string fp = (int)digits.size() > exp10 + 1 ? digits.substr((size_t)exp10 + 1) : "0";
            out = ip + "." + fp;
        } else {
            out = "0." + std::string((size_t)(-exp10 - 1), '0') + digits;
        }
    } else {
        std::string fp = digits.size() > 1 ? digits.substr(1) : "0";
        out = digits.substr(0, 1) + "." + fp + "E" + std::to_string(exp10);
    }
    return neg ? "-" + out : out;
}
std::string java_double_to_string(double v) { return java_fp_to_string<double>(v); }
std::string java_float_to_string(float v) { return java_fp_to_string<float>(v); }

// ------------------------------------------------------------------------------------------------
// Configuration
// ------------------------------------------------------------------------------------------------
static std::string trim(const std::string& s) {
    size_t a = 0, b = s.size();
    while (a < b && (unsigned char)s[a] <= ' ') ++a;
    while (b > a && (unsigned char)s[b - 1] <= ' ') --b;
    return s.substr(a, b - a);
}
void Configuration::load_properties(const std::string& text) {
    std::istringstream in(text);
    std::string line;
    while (std::getline(in, line)) {
        std::string t = trim(line);
        if (t.empty() || t[0] == '#' || t[0] == '!') continue;
        size_t p = t.find_first_of("=:");
        if (p == std::string::npos) { props_[t] = ""; continue; }
        props_[trim(t.substr(0, p))] = trim(t.substr(p + 1));
    }
}
static bool is_blank(const std::string& s) { return trim(s).empty(); }
bool Configuration::has(const std::string& k) const { auto it = props_.find(k); return it != props_.end() && !is_blank(it->second); }
std::string Configuration::get(const std::string& k, const std::string& def) const {
    auto it = props_.find(k);
    return it == props_.end() ? def : it->second;
}
int Configuration::getInt(const std::string& k, int def) const { return has(k) ? std::stoi(get(k)) : def; }
long long Configuration::getLong(const std::string& k, long long def) const { return has(k) ? std::stoll(get(k)) : def; }
float Configuration::getFloat(const std::string& k, float def) const { return has(k) ? std::strtof(get(k).c_str(), nullptr) : def; }
double Configuration::getDouble(const std::string& k, double def) const { return has(k) ? std::strtod(get(k).c_str(), nullptr) : def; }
bool Configuration::getBoolean(const std::string& k, bool def) const {
    if (!has(k)) return def;
    std::string v = trim(get(k));
    std::transform(v.begin(), v.end(), v.begin(), [](unsigned char c) { return (char)std::tolower(c); });
    return v == "true";                                 // Boolean.valueOf
}

// ------------------------------------------------------------------------------------------------
// java.util.Random (JDK 8): LCG 0x5DEECE66D; nextInt(bound) rejection; nextDouble 26+27 bits;
// nextGaussian = Marsaglia polar with StrictMath.log (fdlibm __ieee754_log) and a cached second value.
// ------------------------------------------------------------------------------------------------
namespace {
struct JavaRandom {
    uint64_t seed = 0;
    bool have = false;
    double next_gauss = 0.0;
    void setSeed(long long s) { seed = ((uint64_t)s ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1); have = false; }
    int32_t next(int bits) {
        seed = (seed * 0x5DEECE66DULL + 0xBULL) & ((1ULL << 48) - 1);
        return (int32_t)(uint32_t)(seed >> (48 - bits));
    }
    int32_t nextInt(int32_t bound) {
        int32_t r = next(31);
        const int32_t m = bound - 1;
        if ((bound & m) == 0) return (int32_t)(((int64_t)bound * (int64_t)r) >> 31);
        for (int32_t u = r;; u = next(31)) {
            r = u % bound;
            if ((int32_t)((uint32_t)u - (uint32_t)r + (uint32_t)m) >= 0) return r;
        }
    }
    double nextDouble() {
        const int64_t a = next(26), b = next(27);
        return (double)((a << 27) + b) * 0x1.0p-53;
    }
    static double strict_log(double x);
    double nextGaussian() {
        if (have) { have = false; return next_gauss; }
        double v1, v2, s;
        do { v1 = 2 * nextDouble() - 1; v2 = 2 * nextDouble() - 1; s = v1 * v1 + v2 * v2; } while (s >= 1 || s == 0);
        const double mul = std::sqrt(-2 * strict_log(s) / s);
        next_gauss = v2 * mul; have = true;
        return v1 * mul;
    }
};
// fdlibm e_log.c (freely distributable, Sun Microsystems 1993) restated: what StrictMath.log executes
double JavaRandom::strict_log(double x) {
    static const double ln2_hi = 6.93147180369123816490e-01, ln2_lo = 1.90821492927058770002e-10, two54 = 1.80143985094819840000e+16,
                        Lg1 = 6.666666666666735130e-01, Lg2 = 3.999999999940941908e-01, Lg3 = 2.857142874366239149e-01,
                        Lg4 = 2.222219843214978396e-01, Lg5 = 1.818357216161805012e-01, Lg6 = 1.531383769920937332e-01,
                        Lg7 = 1.479819860511658591e-01;
    auto hi = [](double d) { uint64_t b; memcpy(&b, &d, 8); return (int32_t)(b >> 32); };
    auto lo = [](double d) { uint64_t b; memcpy(&b, &d, 8); return (uint32_t)b; };
    auto sethi = [](double d, int32_t h) { uint64_t b; memcpy(&b, &d, 8); b = (b & 0xffffffffULL) | ((uint64_t)(uint32_t)h << 32); memcpy(&d, &b, 8); return d; };
    int32_t hx = hi(x), k = 0, i, j;
    const uint32_t lx = lo(x);
    if (hx < 0x00100000) {
        if (((hx & 0x7fffffff) | lx) == 0) return -two54 / 0.0;
        if (hx < 0) return (x - x) / 0.0;
        k -= 54; x *= two54; hx = hi(x);
    }
    if (hx >= 0x7ff00000) return x + x;
    k += (hx >> 20) - 1023;
    hx &= 0x000fffff;
    i = (hx + 0x95f64) & 0x100000;
    x = sethi(x, hx | (i ^ 0x3ff00000));
    k += (i >> 20);
    const double f = x - 1.0;
    double dk, R;
    if ((0x000fffff & (2 + hx)) < 3) {
        if (f == 0.0) { if (k == 0) return 0.0; dk = (double)k; return dk * ln2_hi + dk * ln2_lo; }
        R = f * f * (0.5 - 0.33333333333333333 * f);
        if (k == 0) return f - R;
        dk = (double)k; return dk * ln2_hi - ((R - dk * ln2_lo) - f);
    }
    const double s = f / (2.0 + f);
    dk = (double)k;
    const double z = s * s;
    i = hx - 0x6147a;
    const double w = z * z;
    j = 0x6b851 - hx;
    const double t1 = w * (Lg2 + w * (Lg4 + w * Lg6));
    const double t2 = z * (Lg1 + w * (Lg3 + w * (Lg5 + w * Lg7)));
    i |= j;
    R = t2 + t1;
    if (i > 0) {
        const double hfsq = 0.5 * f * f;
        if (k == 0) return f - (hfsq - s * (hfsq + R));
        return dk * ln2_hi - ((hfsq - (s * (hfsq + R) + dk * ln2_lo)) - f);
    }
    if (k == 0) return f - s * (f - R);
    return dk * ln2_hi - ((s * (f - R) - dk * ln2_lo) - f);
}
JavaRandom g_r;
}  // namespace

void Randoms::seed(long long s) { g_r.setSeed(s); }
int Randoms::uniform(int range) { return 0 + g_r.nextInt(range - 0); }
double Randoms::uniform() { return 0.0 + (1.0 - 0.0) * g_r.nextDouble(); }
double Randoms::gaussian(double mu, double sigma) { return mu + sigma * g_r.nextGaussian(); }
uint64_t Randoms::state() { return g_r.seed; }
void Randoms::setState(uint64_t s) { g_r.seed = s & ((1ULL << 48) - 1); }

void DenseMatrix::init(double mean, double sigma) { for (double& v : values) v = Randoms::gaussian(mean, sigma); }
void VectorBasedDenseVector::init(double mean, double sigma) { for (double& v : values) v = Randoms::gaussian(mean, sigma); }
double SequentialAccessSparseMatrix::mean() const {
    double m = 0.0;
    for (double v : val) m += v;
    return m / (double)val.size();
}

// ------------------------------------------------------------------------------------------------
// AbstractRecommender / MatrixRecommender / MatrixFactorizationRecommender
// ------------------------------------------------------------------------------------------------
void AbstractRecommender::train(const Configuration& c, const SequentialAccessSparseMatrix& tr, const SequentialAccessSparseMatrix& te) {
    conf = c; trainMatrix = &tr; testMatrix = &te;
    setup();
    info("Job Setup completed.");
    trainModel();
    info("Job Train completed.");
    cleanup();
}
void AbstractRecommender::setup() {
    isRanking = conf.getBoolean("rec.recommender.isranking");
    if (isRanking) {
        topN = conf.getInt("rec.recommender.ranking.topn", 10);
        if (topN <= 0) throw std::out_of_range("rec.recommender.ranking.topn should be more than 0!");
    }
    earlyStop = conf.getBoolean("rec.recommender.earlystop", false);
    verbose = conf.getBoolean("rec.recommender.verbose", true);
}
bool AbstractRecommender::isConverged(int iter) {
    const float delta_loss = (float)(lastLoss - loss);
    if (verbose)
        info(simpleName() + " iter " + std::to_string(iter) + ": loss = " + java_double_to_string(loss) + ", delta_loss = " +
             java_float_to_string(delta_loss));
    if (std::isnan(loss) || std::isinf(loss))
        throw LibrecException("Loss = NaN or Infinity: current settings does not fit the recommender! Change the settings and try again!");
    return std::fabs(delta_loss) < 1e-5;
}

void MatrixRecommender::setup() {
    AbstractRecommender::setup();
    numUsers = trainMatrix->rowSize();
    numItems = trainMatrix->columnSize();
    numRates = trainMatrix->size();
    std::set<double> rs(trainMatrix->val.begin(), trainMatrix->val.end());
    ratingScale.assign(rs.begin(), rs.end());
    if (ratingScale.empty()) throw LibrecException("empty train matrix");
    maxRate = ratingScale.back(); minRate = ratingScale.front();
    if (minRate == maxRate) minRate = 0;
    globalMean = trainMatrix->mean();
}
double MatrixRecommender::predict(int u, int i, bool bound) {
    double p = predict(u, i);
    if (bound) { if (p > maxRate) p = maxRate; else if (p < minRate) p = minRate; }
    return p;
}

void MatrixFactorizationRecommender::setup() {
    MatrixRecommender::setup();
    numIterations = conf.getInt("rec.iterator.maximum", 100);
    learnRate = conf.getFloat("rec.iterator.learnrate", 0.01f);
    maxLearnRate = conf.getFloat("rec.iterator.learnrate.maximum", 1000.0f);
    regUser = conf.getFloat("rec.user.regularization", 0.01f);
    regItem = conf.getFloat("rec.item.regularization", 0.01f);
    numFactors = conf.getInt("rec.factor.number", 10);
    isBoldDriver = conf.getBoolean("rec.learnrate.bolddriver", false);
    decay = conf.getFloat("rec.learnrate.decay", 1.0f);
    userFactors = DenseMatrix(numUsers, numFactors);
    itemFactors = DenseMatrix(numItems, numFactors);
    impUserFactors = DenseMatrix(numUsers, numFactors);     // the fork's two extra matrices: they consume RNG draws
    impItemFactors = DenseMatrix(numItems, numFactors);
    initMean = 0.0f; initStd = 0.001f;
    userFactors.init(initMean, initStd);
    itemFactors.init(initMean, initStd);
    impUserFactors.init(initMean, initStd);
    impItemFactors.init(initMean, initStd);
}
double MatrixFactorizationRecommender::predict(int u, int i) {
    const double* p = userFactors.row(u); const double* q = itemFactors.row(i);
    double r = 0.0;
    for (int f = 0; f < numFactors; ++f) r += q[f] * p[f];             // DenseVector.java:104-111
    return r;
}
void MatrixFactorizationRecommender::updateLRate(int iter) {
    if (learnRate < 0.0) { lastLoss = loss; return; }
    if (isBoldDriver && iter > 1) learnRate = std::fabs(lastLoss) > std::fabs(loss) ? learnRate * 1.05f : learnRate * 0.5f;
    else if (decay > 0 && decay < 1) learnRate *= decay;
    if (maxLearnRate > 0 && learnRate > maxLearnRate) learnRate = maxLearnRate;
    lastLoss = loss;
}

// ------------------------------------------------------------------------------------------------
// the CUDA drop-ins
// ------------------------------------------------------------------------------------------------
MatrixFactorizationCudaRecommender::~MatrixFactorizationCudaRecommender() {
    if (handle) lrk_destroy(handle);
}
void MatrixFactorizationCudaRecommender::check(int status) const {
    if (status != LRK_OK) throw LibrecException(lrk_last_error(handle));
}
void MatrixFactorizationCudaRecommender::setup() {
    MatrixFactorizationRecommender::setup();
    biased = model() == LRK_MODEL_BIASEDMF;
    lrk_config_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.device = conf.getInt("rec.cuda.device", 0);
    cfg.model = model();
    cfg.num_factors = numFactors;
    cfg.update_mode = conf.get("rec.cuda.order", "shuffled") == "reference" ? LRK_UPDATE_REFERENCE_ORDER : LRK_UPDATE_ATOMIC;
    cfg.seed = (uint64_t)conf.getLong("rec.cuda.seed", 1);
    cfg.topn_path = conf.getInt("rec.cuda.topn.path", 0);
    if (handle) { lrk_destroy(handle); handle = nullptr; }
    if (lrk_create(&cfg, &handle) != LRK_OK) throw LibrecException(lrk_last_error(nullptr));
    check(lrk_set_train_csr(handle, numUsers, numItems, trainMatrix->rowptr.data(), trainMatrix->col.data(), trainMatrix->val.data()));
}
void MatrixFactorizationCudaRecommender::trainModel() {
    check(lrk_set_factors(handle, userFactors.values.data(), itemFactors.values.data(),
                          biased ? userBiases.values.data() : nullptr, biased ? itemBiases.values.data() : nullptr, globalMean));
    for (int iter = 1; iter <= numIterations; ++iter) {
        const int st = lrk_sgd_epoch(handle, learnRate, regUser, regItem, regBias, iter, &loss);
        if (st != LRK_OK && st != LRK_ERR_DIVERGED) check(st);      // a NaN/Inf loss is reported by isConverged, like the reference
        if (isConverged(iter) && earlyStop) break;
        updateLRate(iter);
    }
    check(lrk_get_factors(handle, userFactors.values.data(), itemFactors.values.data(),
                          biased ? userBiases.values.data() : nullptr, biased ? itemBiases.values.data() : nullptr));
}
void BPRCudaRecommender::trainModel() {
    const bool reference = conf.get("rec.cuda.order", "shuffled") == "reference";
    if (reference) {
        const double s = (double)Randoms::state();                  // < 2^48: exact
        check(lrk_set_matrix(handle, "jdk.random.state", &s));
    }
    MatrixFactorizationCudaRecommender::trainModel();
    if (reference) {
        double s = 0.0;
        check(lrk_get_matrix(handle, "jdk.random.state", &s));
        Randoms::setState((uint64_t)s);
    }
}
RecommendedList MatrixFactorizationCudaRecommender::recommendRank() {
    std::vector<int> all((size_t)numUsers);
    for (int u = 0; u < numUsers; ++u) all[(size_t)u] = u;
    return recommendRank(all);
}
RecommendedList MatrixFactorizationCudaRecommender::recommendRank(const std::vector<int>& userIds) {
    info("begin recommend");
    const int n = (int)userIds.size();
    std::vector<int32_t> items((size_t)n * topN), counts((size_t)n);
    std::vector<double> scores((size_t)n * topN);
    check(lrk_topn(handle, userIds.data(), n, topN, 1, items.data(), scores.data(), counts.data()));
    RecommendedList list;
    for (int c = 0; c < n; ++c) {
        list.addList();
        for (int t = 0; t < counts[(size_t)c]; ++t) list.add(c, items[(size_t)c * topN + t], scores[(size_t)c * topN + t]);
    }
    if (list.size() == 0)
        throw std::out_of_range("No item is recommended, there is something error in the recommendation algorithm! Please check it!");
    info("end recommend");
    return list;
}
RecommendedList MatrixFactorizationCudaRecommender::recommendRankAndEvaluate(const SequentialAccessSparseMatrix& test,
                                                                             std::map<std::string, double>* measures) {
    info("begin recommend");
    const int n = numUsers;
    std::vector<int32_t> items((size_t)n * topN), counts((size_t)n);
    std::vector<double> scores((size_t)n * topN);
    double m[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    check(lrk_eval_ranking(handle, topN, test.rowptr.data(), test.col.data(), test.val.data(), items.data(), scores.data(),
                           counts.data(), m));
    RecommendedList list;
    for (int c = 0; c < n; ++c) {
        list.addList();
        for (int t = 0; t < counts[(size_t)c]; ++t) list.add(c, items[(size_t)c * topN + t], scores[(size_t)c * topN + t]);
    }
    if (list.size() == 0)
        throw std::out_of_range("No item is recommended, there is something error in the recommendation algorithm! Please check it!");
    info("end recommend");
    static const char* names[8] = {"AUC", "AP", "NDCG", "PRECISION", "RECALL", "RR", "Novelty", "Entropy"};   // eval/Measure.java
    if (measures) for (int i = 0; i < 8; ++i) (*measures)[std::string(names[i]) + " top " + std::to_string(topN)] = m[i];
    return list;
}
RecommendedList MatrixFactorizationCudaRecommender::recommendRating(const SequentialAccessSparseMatrix& pm) {
    std::vector<double> pred((size_t)pm.size());
    double rmse = 0, mae = 0;
    check(lrk_eval_rating(handle, pm.numRows, pm.rowptr.data(), pm.col.data(), pm.val.data(), minRate, maxRate,
                          pred.data(), &rmse, &mae));
    RecommendedList list;
    for (int u = 0; u < pm.numRows; ++u) {
        list.addList();
        for (int64_t e = pm.rowptr[(size_t)u]; e < pm.rowptr[(size_t)u + 1]; ++e) list.add(u, pm.col[(size_t)e], pred[(size_t)e]);
    }
    return list;
}

void BiasedMFCudaRecommender::setup() {
    MatrixFactorizationCudaRecommender::setup();
    regBias = conf.getDouble("rec.bias.regularization", 0.01);
    userBiases = VectorBasedDenseVector(numUsers);
    itemBiases = VectorBasedDenseVector(numItems);
    userBiases.init(initMean, initStd);
    itemBiases.init(initMean, initStd);
}
double BiasedMFCudaRecommender::predict(int u, int i) {
    return MatrixFactorizationRecommender::predict(u, i) + userBiases.get(u) + itemBiases.get(i) + globalMean;
}

std::unique_ptr<MatrixFactorizationCudaRecommender> newRecommender(const std::string& name) {
    std::string n = name;
    std::transform(n.begin(), n.end(), n.begin(), [](unsigned char c) { return (char)std::tolower(c); });
    if (n == "biasedmf" || n == "net.librec.recommender.cuda.biasedmfcudarecommender") return std::make_unique<BiasedMFCudaRecommender>();
    if (n == "pmf" || n == "net.librec.recommender.cuda.pmfcudarecommender") return std::make_unique<PMFCudaRecommender>();
    if (n == "bpr" || n == "net.librec.recommender.cuda.bprcudarecommender") return std::make_unique<BPRCudaRecommender>();
    if (n == "ranksgd" || n == "net.librec.recommender.cuda.ranksgdcudarecommender") return std::make_unique<RankSGDCudaRecommender>();
    throw LibrecException("ClassNotFoundException: " + name);
}

// ------------------------------------------------------------------------------------------------
// evaluators + job
// ------------------------------------------------------------------------------------------------
static void zip_eval(const SequentialAccessSparseMatrix& test, const RecommendedList& rec, double* se, double* ae, int64_t* n) {
    *se = 0; *ae = 0; *n = 0;
    for (int u = 0; u < test.numRows; ++u) {
        const auto& lst = rec.lists[(size_t)u];
        size_t t = 0;
        for (int64_t e = test.rowptr[(size_t)u]; e < test.rowptr[(size_t)u + 1]; ++e, ++t) {
            if (t >= lst.size()) throw std::out_of_range("index cardinality of recommendedList does not equal testMatrix index cardinality");
            if (lst[t].key != test.col[(size_t)e]) throw std::out_of_range("index of recommendedList does not equal testMatrix index");
            const double d = test.val[(size_t)e] - lst[t].value;
            *se += d * d; *ae += std::fabs(d); ++*n;
        }
    }
}
double evaluateRMSE(const SequentialAccessSparseMatrix& test, const RecommendedList& rec) {
    if (test.size() == 0) return 0.0;
    double se, ae; int64_t n; zip_eval(test, rec, &se, &ae, &n);
    return n > 0 ? std::sqrt(se / (double)n) : 0.0;
}
double evaluateMAE(const SequentialAccessSparseMatrix& test, const RecommendedList& rec) {
    if (test.size() == 0) return 0.0;
    double se, ae; int64_t n; zip_eval(test, rec, &se, &ae, &n);
    return n > 0 ? ae / (double)n : 0.0;
}
double evaluateMSE(const SequentialAccessSparseMatrix& test, const RecommendedList& rec) {        // eval/rating/MSEEvaluator.java:33-66
    if (test.size() == 0) return 0.0;
    double se, ae; int64_t n; zip_eval(test, rec, &se, &ae, &n);
    return n > 0 ? se / (double)n : 0.0;
}
double evaluateMPE(const SequentialAccessSparseMatrix& test, const RecommendedList& rec, double mpe) {   // eval/rating/MPEEvaluator.java:33-73
    if (test.size() == 0) return 0.0;
    int64_t n = 0, over = 0;
    for (int u = 0; u < test.numRows; ++u) {
        const auto& lst = rec.lists[(size_t)u];
        size_t t = 0;
        for (int64_t e = test.rowptr[(size_t)u]; e < test.rowptr[(size_t)u + 1]; ++e, ++t) {
            if (t >= lst.size()) throw std::out_of_range("index cardinality of recommendedList does not equal testMatrix index cardinality");
            if (lst[t].key != test.col[(size_t)e]) throw std::out_of_range("index of recommendedList does not equal testMatrix index");
            if (std::fabs(test.val[(size_t)e] - lst[t].value) > mpe) ++over;
            ++n;
        }
    }
    return n > 0 ? ((double)over + 0.0) / (double)n : 0.0;
}

// ---------------------------------------------------------------------------------------------------------------------
// Ranking measures on the host -- used when rec.recommender.ranking.topn exceeds what the device evaluator keeps per thread
// (64).  One pass per user over its list and its test row; semantics of eval/ranking/*.java:
//   PRECISION hits / topN (PrecisionEvaluator.java:41);  RECALL hits / |test row| (RecallEvaluator.java);
//   AP  sum over hit positions of hits-so-far / position, divided by min(|test row|, list length), users with an empty list
//       skipped (AveragePrecisionEvaluator.java);  RR 1 / position of the first hit (ReciprocalRankEvaluator.java);
//   NDCG dcg / idcg with gains = TEST RATINGS of the hits, discount log2(position + 1), ideal = the same hits sorted by
//       rating (NormalizedDCGEvaluator.java:84-120);
//   AUC (AUCEvaluator.java:56-98) pair count with the dropped-items correction; the test items are walked in
//       java.util.HashSet<Integer> order (ascending bucket of h ^ h>>>16 in a table of the set's capacity);
//   Novelty (NoveltyEvaluator.java) sum over recommended items of -ln(purchases / numUsers), / (numUsers ln 2);
//   Entropy (EntropyEvaluator.java:60-90) of the items' share of the lists, in bits.
// Users without test entries do not count for the first six.
// ---------------------------------------------------------------------------------------------------------------------
void evaluateRanking(const SequentialAccessSparseMatrix& train, const SequentialAccessSparseMatrix& test, const RecommendedList& rec,
                     int topN, std::map<std::string, double>* measures) {
    const int numUsers = test.numRows, numItems = test.numCols;
    std::vector<int> purchases((size_t)numItems, 0), listed((size_t)numItems, 0);
    for (int32_t c : train.col) purchases[(size_t)c]++;
    for (int32_t c : test.col) purchases[(size_t)c]++;
    double novelty = 0.0;
    double auc = 0, ap = 0, ndcg = 0, prec = 0, recall = 0, rr = 0;
    int64_t usersWithTest = 0, usersWithList = 0;
    std::vector<double> gains;
    std::vector<std::pair<uint64_t, int32_t>> hashOrder;
    for (int u = 0; u < numUsers; ++u) {
        const auto& lst = rec.lists[(size_t)u];
        const int len = (int)std::min<size_t>(lst.size(), (size_t)topN);
        for (int t = 0; t < len; ++t) {
            const int item = lst[(size_t)t].key;
            listed[(size_t)item]++;
            if (purchases[(size_t)item] > 0) novelty += -std::log((double)purchases[(size_t)item] / numUsers);
        }
        const int64_t tb = test.rowptr[(size_t)u], te = test.rowptr[(size_t)u + 1];
        const int64_t nTest = te - tb;
        if (nTest <= 0) continue;
        ++usersWithTest;
        auto testValue = [&](int item, double* v) {
            const int32_t* b = test.col.data() + tb;
            const int32_t* e = test.col.data() + te;
            const int32_t* f = std::lower_bound(b, e, item);
            if (f == e || *f != item) return false;
            if (v) *v = test.val[(size_t)(f - test.col.data())];
            return true;
        };
        int hits = 0, misses = 0;
        double precSum = 0.0, dcg = 0.0;
        bool firstHit = true;
        gains.clear();
        for (int t = 0; t < len; ++t) {
            double v = 0.0;
            if (!testValue(lst[(size_t)t].key, &v)) { ++misses; continue; }
            ++hits;
            precSum += 1.0 * hits / (t + 1);
            if (firstHit) { rr += 1.0 / (t + 1.0); firstHit = false; }
            dcg += v / (std::log((double)(t + 2)) / std::log(2.0));
            gains.push_back(v);
        }
        prec += hits / (topN + 0.0);
        recall += hits / (nTest + 0.0);
        if (len != 0) { ap += precSum / (double)(nTest < len ? nTest : len); ++usersWithList; }
        if (!gains.empty() && dcg != 0.0) {
            std::sort(gains.begin(), gains.end(), std::greater<double>());
            double idcg = 0.0;
            for (size_t t = 0; t < gains.size(); ++t) idcg += gains[t] / (std::log((double)(t + 2)) / std::log(2.0));
            if (idcg != 0.0) ndcg += dcg / idcg;
        }
        // AUC: items never scored (numItems - |train row| - list length) rank below every listed item
        const int64_t dropped = (int64_t)numItems - (train.rowptr[(size_t)u + 1] - train.rowptr[(size_t)u]) - len;
        const int64_t pairs = ((dropped + len) - hits) * (int64_t)hits;
        if (pairs == 0) { auc += 0.5; continue; }
        uint32_t cap = 16;
        while ((double)nTest > 0.75 * (double)cap) cap <<= 1;
        hashOrder.clear();
        for (int64_t e = tb; e < te; ++e) {
            const uint32_t h = (uint32_t)test.col[(size_t)e];
            hashOrder.push_back({((uint64_t)((h ^ (h >> 16)) & (cap - 1)) << 32) | (uint32_t)(e - tb), test.col[(size_t)e]});
        }
        std::sort(hashOrder.begin(), hashOrder.end());
        int64_t correct = 0;
        int seenHits = 0;
        for (const auto& o : hashOrder) {
            bool inList = false;
            for (int t = 0; t < len; ++t) if (lst[(size_t)t].key == o.second) { inList = true; break; }
            if (inList) ++seenHits; else correct += seenHits;
        }
        correct += (int64_t)seenHits * (dropped - misses);
        auc += (correct + 0.0) / (double)pairs;
    }
    double entropy = 0.0;
    for (int i = 0; i < numItems; ++i)
        if (listed[(size_t)i] > 0) { const double p = (double)listed[(size_t)i] / numUsers; entropy += p * (-std::log(p)); }
    const std::string suffix = " top " + std::to_string(topN);
    (*measures)["AUC" + suffix] = usersWithTest ? auc / usersWithTest : 0.0;
    (*measures)["AP" + suffix] = usersWithList ? ap / usersWithList : 0.0;
    (*measures)["NDCG" + suffix] = usersWithTest ? ndcg / usersWithTest : 0.0;
    (*measures)["PRECISION" + suffix] = usersWithTest ? prec / usersWithTest : 0.0;
    (*measures)["RECALL" + suffix] = usersWithTest ? recall / usersWithTest : 0.0;
    (*measures)["RR" + suffix] = usersWithTest ? rr / usersWithTest : 0.0;
    (*measures)["Novelty" + suffix] = novelty / (numUsers * std::log(2.0));
    (*measures)["Entropy" + suffix] = entropy / std::log(2.0);
}

// The ranking evaluators outside the default list (rec.eval.classes = hitrate, arhr, idcg): HitRateEvaluator.java:33-62 (leave-one-out
// only: throws when a user has more than one test item), AverageReciprocalHitRankEvaluator.java:33-56 (the user's FIRST test item),
// IdealDCGEvaluator.java:34-52.  Keys "HitRate" / "ARHR" / "IDCG" + " top <N>".
void evaluateRankingExtra(const SequentialAccessSparseMatrix& test, const RecommendedList& rec, int topN, bool wantHitRate,
                          std::map<std::string, double>* measures) {
    int64_t hits = 0, usersWithTest = 0;
    double arhr = 0.0, idcgSum = 0.0;
    for (int u = 0; u < test.numRows; ++u) {
        const int64_t tb = test.rowptr[(size_t)u], nTest = test.rowptr[(size_t)u + 1] - tb;
        if (nTest <= 0) continue;
        if (wantHitRate && nTest > 1)
            throw std::out_of_range("It is not a leave-one-out validation method! Please use leave-one-out validation method");
        ++usersWithTest;
        const auto& lst = rec.lists[(size_t)u];
        const int len = (int)std::min<size_t>(lst.size(), (size_t)topN);
        const int first = test.col[(size_t)tb];
        for (int t = 0; t < len; ++t)
            if (lst[(size_t)t].key == first) { ++hits; arhr += 1.0 / (t + 1.0); break; }
        double idcg = 0.0;                                   // IdealDCGEvaluator sums per user first, then adds
        for (int64_t i = 0; i < nTest; ++i) idcg += 1 / (std::log((double)i + 2.0) / std::log(2.0));
        idcgSum += idcg;
    }
    const std::string suffix = " top " + std::to_string(topN);
    if (wantHitRate) (*measures)["HitRate" + suffix] = usersWithTest ? 1.0 * hits / usersWithTest : 0.0;
    (*measures)["ARHR" + suffix] = usersWithTest ? arhr / usersWithTest : 0.0;
    (*measures)["IDCG" + suffix] = usersWithTest ? idcgSum / usersWithTest : 0.0;
}

// ---------------------------------------------------------------------------------------------------------------------
// TextDataModel: text file -> flat CSR -> ratio split
// ---------------------------------------------------------------------------------------------------------------------
namespace {
struct SvHash { size_t operator()(const std::string_view& v) const { return std::hash<std::string_view>()(v); } };
inline bool is_sep(char c) { return c == '\t' || c == ';' || c == ',' || c == ' '; }
inline bool is_blank_line(const char* b, const char* e) {       // String.trim().isEmpty(): every char <= U+0020
    for (; b < e; ++b) if ((unsigned char)*b > ' ') return false;
    return true;
}
}  // namespace

// Files.walkFileTree (TextDataConvertor.java:157-169): a path that is a directory contributes every regular file below it.
// The JDK visits a directory in the order the file system lists it; here the listing is sorted by name so that inner ids
// (first-seen order) do not depend on the file system.
static void collect_files(const std::string& path, std::vector<std::string>& out) {
    struct stat st;
    if (stat(path.c_str(), &st) != 0) throw LibrecException("TextDataConvertor: cannot read " + path);
    if (!S_ISDIR(st.st_mode)) { out.push_back(path); return; }
    DIR* d = opendir(path.c_str());
    if (!d) throw LibrecException("TextDataConvertor: cannot list " + path);
    std::vector<std::string> names;
    while (struct dirent* e = readdir(d)) {
        const std::string n = e->d_name;
        if (n != "." && n != "..") names.push_back(n);
    }
    closedir(d);
    std::sort(names.begin(), names.end());
    for (const std::string& n : names) collect_files(path + "/" + n, out);
}

void TextDataModel::buildConvert() {
    const std::string dir = conf.get("dfs.data.dir", "");
    const std::string fmt = conf.get("data.column.format", "UIR");
    const double binThold = conf.getDouble("data.convert.binarize.threshold", -1.0);
    const size_t nfields = (fmt == "UIRT" || fmt == "uirt") ? 4 : 3;
    std::deque<std::string> bufs;                  // ids are views into these buffers
    std::unordered_map<std::string_view, int32_t, SvHash> umap, imap;      // DataFrame's static id maps: shared by the test-set load
    std::vector<std::string_view> uview, iview;
    struct Lines { std::vector<uint64_t> keys; std::vector<double> rates; std::vector<int64_t> dates; };   // key = user << 32 | item, line order

    // a ':'-separated path list, each entry relative to dfs.data.dir, file or directory (TextDataModel.java:58-64)
    auto collect = [&](const std::string& spec, std::string& shown) {
        std::vector<std::string> files;
        std::string all = spec;
        size_t b = all.find_first_not_of(" \t\r\n"), e = all.find_last_not_of(" \t\r\n");
        all = b == std::string::npos ? std::string() : all.substr(b, e - b + 1);
        size_t from = 0;
        for (;;) {
            const size_t c = all.find(':', from);
            std::string one = all.substr(from, c == std::string::npos ? std::string::npos : c - from);
            const size_t ob = one.find_first_not_of(" \t");
            one = ob == std::string::npos ? std::string() : one.substr(ob, one.find_last_not_of(" \t") - ob + 1);
            const std::string full = (dir.empty() ? std::string() : dir + "/") + one;
            shown += (shown.empty() ? "" : ", ") + full;
            collect_files(full, files);
            if (c == std::string::npos) break;
            from = c + 1;
        }
        return files;
    };
    // pass 1: one (user, item, rating[, date]) per line, inner ids in first-seen order; the first blank line ends THAT file
    auto parse = [&](const std::vector<std::string>& files, Lines& L) {
        for (const std::string& path : files) {
            FILE* fp = fopen(path.c_str(), "rb");
            if (!fp) throw LibrecException("TextDataConvertor: cannot read " + path);
            bufs.emplace_back();
            std::string& buf = bufs.back();
            {
                char tmp[1 << 16];
                size_t got;
                while ((got = fread(tmp, 1, sizeof tmp, fp)) > 0) buf.append(tmp, got);
                fclose(fp);
            }
            const char* p = buf.data();
            const char* const end = p + buf.size();
            while (p < end) {
                const char* eol = (const char*)memchr(p, '\n', (size_t)(end - p));
                const char* le = eol ? eol : end;
                const char* lend = (le > p && le[-1] == '\r') ? le - 1 : le;
                if (is_blank_line(p, lend)) break;                                           // TextDataConvertor.java:176-178
                // fields: split at every separator character, drop trailing empty fields
                std::string_view f[4]; size_t nf = 0, total = 0;
                const char* fb = p;
                for (const char* c = p;; ++c) {
                    if (c == lend || is_sep(*c)) {
                        if (nf < 4) f[nf] = std::string_view(fb, (size_t)(c - fb));
                        if (c > fb) total = nf + 1;                                          // index of the last non-empty field + 1
                        ++nf;
                        if (c == lend) break;
                        fb = c + 1;
                    }
                }
                if (total < nfields) throw std::out_of_range("TextDataConvertor: line with fewer than " + std::to_string(nfields) + " fields: " + std::string(p, (size_t)(lend - p)));
                auto idOf = [](std::unordered_map<std::string_view, int32_t, SvHash>& m, std::vector<std::string_view>& views, std::string_view key) {
                    auto it = m.find(key);
                    if (it != m.end()) return it->second;
                    const int32_t id = (int32_t)m.size();                                    // DataFrame.java:370-379
                    m.emplace(key, id); views.push_back(key);
                    return id;
                };
                const int32_t u = idOf(umap, uview, f[0]), i = idOf(imap, iview, f[1]);
                const std::string rs(f[2]);
                char* pe = nullptr;
                const double r = strtod(rs.c_str(), &pe);
                if (rs.empty() || (pe && *pe != 0)) throw std::invalid_argument("NumberFormatException: For input string: \"" + rs + "\"");
                L.keys.push_back(((uint64_t)(uint32_t)u << 32) | (uint32_t)i);
                L.rates.push_back(r);
                if (nfields == 4) {                                                          // DataFrame.java:112-113 Long.parseLong
                    const std::string ds(f[3]);
                    char* de = nullptr;
                    const long long d = strtoll(ds.c_str(), &de, 10);
                    if (ds.empty() || (de && *de != 0)) throw std::invalid_argument("NumberFormatException: For input string: \"" + ds + "\"");
                    L.dates.push_back((int64_t)d);
                }
                p = eol ? eol + 1 : end;
            }
        }
    };
    // pass 2: order by (user, item, line); the first entry of every (user, item) run is the earliest line -> it wins
    auto build = [&](const Lines& L, int32_t U, int32_t I, SequentialAccessSparseMatrix& out, std::vector<int64_t>* outDates) {
        const size_t n = L.keys.size();
        std::vector<uint32_t> ord(n);
        for (size_t t = 0; t < n; ++t) ord[t] = (uint32_t)t;
        std::sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return L.keys[a] != L.keys[b] ? L.keys[a] < L.keys[b] : a < b; });
        out = SequentialAccessSparseMatrix();
        if (outDates) outDates->clear();
        out.numRows = U; out.numCols = I;
        out.rowptr.assign((size_t)U + 1, 0);
        out.col.reserve(n); out.val.reserve(n);
        for (size_t t = 0; t < n; ++t) {
            const uint32_t a = ord[t];
            if (t > 0 && L.keys[ord[t - 1]] == L.keys[a]) continue;
            double r = L.rates[a];
            if (binThold >= 0) r = r > binThold ? 1.0 : -1.0;                                // DataFrame.java:251-253
            out.col.push_back((int32_t)(L.keys[a] & 0xffffffffu));
            out.val.push_back(r);
            if (outDates && nfields == 4) outDates->push_back(L.dates[a]);
            out.rowptr[(size_t)(L.keys[a] >> 32) + 1]++;
        }
        for (int32_t u = 0; u < U; ++u) out.rowptr[(size_t)u + 1] += out.rowptr[(size_t)u];
    };

    std::string shown;
    Lines mainLines, testLines;
    parse(collect(conf.get("data.input.path", ""), shown), mainLines);
    log.push_back("Dataset: [" + shown + "]");
    std::string splitter = conf.get("data.model.splitter", "ratio");
    std::transform(splitter.begin(), splitter.end(), splitter.begin(), [](unsigned char c) { return (char)std::tolower(c); });
    const bool testset = splitter == "testset" || splitter == "net.librec.data.splitter.giventestsetdatasplitter";
    if (testset) {
        // GivenTestSetDataSplitter.java:64-84: the test file(s) (data.testset.path, same list syntax) go through a second
        // convertor that continues the id maps; both matrices get the final dimensions
        if (!conf.has("data.testset.path")) throw LibrecException("data.model.splitter=testset needs data.testset.path");
        std::string shownTest;
        parse(collect(conf.get("data.testset.path", ""), shownTest), testLines);
        log.push_back("Dataset: [" + shownTest + "]");
    }
    const int32_t U = (int32_t)umap.size(), I = (int32_t)imap.size();
    build(mainLines, U, I, preference, &datetime);
    givenTest = SequentialAccessSparseMatrix();
    if (testset) build(testLines, U, I, givenTest, nullptr);
    userIds.assign(uview.begin(), uview.end());
    itemIds.assign(iview.begin(), iview.end());
    log.push_back("user number: " + std::to_string(U) + ",\t item number is: " + std::to_string(I));
}

// (train, test) from a per-entry flag; entries whose value is exactly 0.0 vanish from both (reshape())
static void two_way(const SequentialAccessSparseMatrix& pref, const std::vector<uint8_t>& isTrain,
                    SequentialAccessSparseMatrix& train, SequentialAccessSparseMatrix& test) {
    auto start = [&](SequentialAccessSparseMatrix& m) {
        m = SequentialAccessSparseMatrix();
        m.numRows = pref.numRows; m.numCols = pref.numCols;
        m.rowptr.assign((size_t)pref.numRows + 1, 0);
    };
    start(train); start(test);
    for (int u = 0; u < pref.numRows; ++u) {
        for (int64_t e = pref.rowptr[(size_t)u]; e < pref.rowptr[(size_t)u + 1]; ++e) {
            const double v = pref.val[(size_t)e];
            if (v == 0.0) continue;
            SequentialAccessSparseMatrix& dst = isTrain[(size_t)e] ? train : test;
            dst.col.push_back(pref.col[(size_t)e]); dst.val.push_back(v);
            dst.rowptr[(size_t)u + 1]++;
        }
    }
    for (int u = 0; u < pref.numRows; ++u) {
        train.rowptr[(size_t)u + 1] += train.rowptr[(size_t)u];
        test.rowptr[(size_t)u + 1] += test.rowptr[(size_t)u];
    }
}
// column walk of the CSR matrix (SequentialAccessSparseMatrix.column(j): rows ascending): csc[colptr[j] + t] = entry index
static void csc_order(const SequentialAccessSparseMatrix& m, std::vector<int64_t>& colptr, std::vector<int64_t>& csc) {
    const size_t nnz = m.col.size();
    colptr.assign((size_t)m.numCols + 1, 0);
    for (size_t e = 0; e < nnz; ++e) colptr[(size_t)m.col[e] + 1]++;
    for (int j = 0; j < m.numCols; ++j) colptr[(size_t)j + 1] += colptr[(size_t)j];
    csc.assign(nnz, 0);
    std::vector<int64_t> fill(colptr.begin(), colptr.end() - 1);
    for (int u = 0; u < m.numRows; ++u)
        for (int64_t e = m.rowptr[(size_t)u]; e < m.rowptr[(size_t)u + 1]; ++e) csc[(size_t)fill[(size_t)m.col[(size_t)e]]++] = e;
}
// Randoms.nextIntArray(length, range): math/algorithm/Randoms.java:576-604 (nextInt :520-535)
static void next_int_array(int length, int range, std::vector<int>& out) {
    out.clear();
    if (range == length) { for (int i = 0; i < length; ++i) out.push_back(i); return; }
    while ((int)out.size() < length) {
        const int next = Randoms::uniform(range);
        if (std::find(out.begin(), out.end(), next) == out.end()) out.push_back(next);
    }
    std::sort(out.begin(), out.end());
}

// date-ordered cuts (util/RatingContext.java:35-44, stable Collections.sort): mode 0 ratio ratingdate, 1 ratio userdate,
// 2 ratio itemdate, 3 loocv userdate, 4 loocv itemdate, 5 givenn userdate, 6 givenn itemdate.  QUIRK kept from the
// reference: modes 1 and 5 walk preferenceMatrix.row(u) and use (long) RATING as the timestamp (RatioDataSplitter.java:297,
// GivenNDataSplitter.java:189), the others read the datetime matrix.
static void split_by_date(const SequentialAccessSparseMatrix& pref, const std::vector<int64_t>& date, int mode, double ratio, int given,
                          std::vector<uint8_t>& isTrain) {
    const bool byCol = mode == 2 || mode == 4 || mode == 6;
    const bool needDate = !(mode == 1 || mode == 5);
    if (needDate && date.size() != pref.col.size()) throw LibrecException("this splitter needs data.column.format=UIRT (a date column)");
    std::vector<int64_t> colptr, csc;
    if (byCol) csc_order(pref, colptr, csc);
    std::vector<std::pair<int64_t, int64_t>> ctx;
    auto cut = [&](const int64_t* entries, size_t n, bool identity, int64_t first) {
        if (n == 0) return;
        ctx.resize(n);
        for (size_t t = 0; t < n; ++t) {
            const int64_t e = identity ? first + (int64_t)t : entries[t];
            ctx[t] = {needDate ? date[(size_t)e] : (int64_t)pref.val[(size_t)e], e};
        }
        std::stable_sort(ctx.begin(), ctx.end(), [](const std::pair<int64_t, int64_t>& a, const std::pair<int64_t, int64_t>& b) {
            return (double)a.first - (double)b.first < 0;
        });
        size_t nTrain;
        if (mode <= 2) nTrain = (size_t)(int)((double)n * ratio);
        else if (mode <= 4) nTrain = n - 1;
        else nTrain = (size_t)std::min<int64_t>((int64_t)n, given);
        for (size_t t = 0; t < n; ++t) isTrain[(size_t)ctx[t].second] = t < nTrain;
    };
    if (mode == 0) cut(nullptr, pref.col.size(), true, 0);
    else if (!byCol) for (int u = 0; u < pref.numRows; ++u) cut(nullptr, (size_t)(pref.rowptr[(size_t)u + 1] - pref.rowptr[(size_t)u]), true, pref.rowptr[(size_t)u]);
    else for (int j = 0; j < pref.numCols; ++j) cut(csc.data() + colptr[(size_t)j], (size_t)(colptr[(size_t)j + 1] - colptr[(size_t)j]), false, 0);
}

void TextDataModel::buildSplitter() {
    std::string splitter = conf.get("data.model.splitter", "ratio");
    std::transform(splitter.begin(), splitter.end(), splitter.begin(), [](unsigned char c) { return (char)std::tolower(c); });
    auto lower = [](std::string v) { std::transform(v.begin(), v.end(), v.begin(), [](unsigned char c) { return (char)std::tolower(c); }); return v; };
    const size_t nnz = preference.col.size();
    std::vector<uint8_t> isTrain(nnz, 1);
    numFolds = 1; foldCursor = 0; assign.clear();
    valid = SequentialAccessSparseMatrix();
    std::vector<int64_t> colptr, csc;
    if (splitter == "ratio" || splitter == "net.librec.data.splitter.ratiodatasplitter") {
        const std::string by = lower(conf.get("data.splitter.ratio", "rating"));
        const double ratio = conf.getDouble("data.splitter.trainset.ratio", 0.8);
        if (by == "rating" || by == "user") {                                                // RatioDataSplitter.java:136-156, 232-249
            for (size_t e = 0; e < nnz; ++e) isTrain[e] = Randoms::uniform() < ratio;
        } else if (by == "item") {                                                           // :315-334, column order
            csc_order(preference, colptr, csc);
            for (size_t t = 0; t < nnz; ++t) isTrain[(size_t)csc[t]] = Randoms::uniform() < ratio;
        } else if (by == "valid") {                                                          // getRatio :382-412, three-way
            const double validRatio = conf.getDouble("data.splitter.validset.ratio", 0.0);
            if (!((ratio > 0 && validRatio > 0) && (ratio + validRatio) < 1))
                throw LibrecException("data.splitter.ratio=valid needs positive trainset / validset ratios with a sum below 1");
            std::vector<uint8_t> isValid(nnz, 0), inTrainOrValid(nnz, 0);
            for (size_t e = 0; e < nnz; ++e) {
                const double rdm = Randoms::uniform();
                isTrain[e] = rdm < ratio;
                isValid[e] = !isTrain[e] && rdm < ratio + validRatio;
                inTrainOrValid[e] = isTrain[e] || isValid[e];
            }
            SequentialAccessSparseMatrix rest;
            two_way(preference, inTrainOrValid, rest, test);                                 // test = neither
            two_way(preference, isValid, valid, rest);                                       // valid
            two_way(preference, isTrain, train, rest);                                       // train
            return;
        } else if (by == "ratingdate" || by == "userdate" || by == "itemdate") {             // :190-221, 283-313, 339-373
            if (ratio > 0 && ratio < 1) split_by_date(preference, datetime, by == "ratingdate" ? 0 : (by == "userdate" ? 1 : 2), ratio, 0, isTrain);
        } else {
            throw LibrecException("data.splitter.ratio=" + by + " is not implemented (rating, user, item, valid, ratingdate, userdate, itemdate are; userfixed is broken in the reference: its train and test sets overlap)");
        }
    } else if (splitter == "loocv" || splitter == "net.librec.data.splitter.loocvdatasplitter") {
        const std::string by = lower(conf.get("data.splitter.loocv", "user"));
        if (by == "user") {                                                                  // LOOCVDataSplitter.java:144-165
            for (int u = 0; u < preference.numRows; ++u) {
                const int64_t n = preference.rowptr[(size_t)u + 1] - preference.rowptr[(size_t)u];
                if (n == 0) continue;
                isTrain[(size_t)(preference.rowptr[(size_t)u] + (int64_t)((double)n * Randoms::uniform()))] = 0;
            }
        } else if (by == "item") {                                                           // :197-216
            csc_order(preference, colptr, csc);
            for (int j = 0; j < preference.numCols; ++j) {
                const int64_t n = colptr[(size_t)j + 1] - colptr[(size_t)j];
                if (n == 0) continue;
                isTrain[(size_t)csc[(size_t)(colptr[(size_t)j] + (int64_t)((double)n * Randoms::uniform()))]] = 0;
            }
        } else if (by == "userdate" || by == "itemdate") {                                   // :171-191, 222-250
            split_by_date(preference, datetime, by == "userdate" ? 3 : 4, 0.0, 0, isTrain);
        } else {
            throw LibrecException("data.splitter.loocv=" + by + " is not implemented (user, item, userdate, itemdate are)");
        }
    } else if (splitter == "givenn" || splitter == "net.librec.data.splitter.givenndatasplitter") {
        const std::string by = lower(conf.get("data.splitter.givenn", "user"));
        const int given = (int)conf.getLong("data.splitter.givenn.n", 1);
        if (by == "userdate" || by == "itemdate") {                                          // GivenNDataSplitter.java:176-207, 254-284
            if (given > 0) split_by_date(preference, datetime, by == "userdate" ? 5 : 6, 0.0, given, isTrain);
            two_way(preference, isTrain, train, test);
            return;
        }
        if (by != "user" && by != "item") throw LibrecException("data.splitter.givenn=" + by + " is not implemented (user, item, userdate, itemdate are)");
        const bool byItem = by == "item";                                                    // GivenNDataSplitter.java:137-167, 217-245
        if (byItem) csc_order(preference, colptr, csc);
        std::vector<int> keep;
        const int lines = byItem ? preference.numCols : preference.numRows;
        for (int l = 0; given > 0 && l < lines; ++l) {
            const int64_t b = byItem ? colptr[(size_t)l] : preference.rowptr[(size_t)l];
            const int64_t n = (byItem ? colptr[(size_t)l + 1] : preference.rowptr[(size_t)l + 1]) - b;
            if (n <= given) continue;
            next_int_array(given, (int)n, keep);
            size_t g = 0;
            for (int64_t pos = 0; pos < n; ++pos) {
                const int64_t e = byItem ? csc[(size_t)(b + pos)] : b + pos;
                if (g < keep.size() && keep[g] == pos) ++g; else isTrain[(size_t)e] = 0;
            }
        }
    } else if (splitter == "kcv" || splitter == "net.librec.data.splitter.kcvdatasplitter") {
        const int64_t kFold = conf.getLong("data.splitter.cv.number", 5);                    // KCVDataSplitter.java:84-123,133-138
        if (kFold <= 0 || nnz == 0) throw LibrecException("data.splitter.cv.number must be positive and the data non-empty");
        const int64_t numFold = kFold > (int64_t)nnz ? (int64_t)nnz : kFold;
        const double indv = ((double)nnz + 0.0) / (double)numFold;
        std::vector<std::pair<int32_t, double>> rdm(nnz);
        for (size_t i = 0; i < nnz; ++i) rdm[i] = {(int32_t)((double)i / indv) + 1, Randoms::uniform()};
        std::stable_sort(rdm.begin(), rdm.end(), [](const std::pair<int32_t, double>& a, const std::pair<int32_t, double>& b) { return a.second > b.second; });
        assign.resize(nnz);
        for (size_t i = 0; i < nnz; ++i) assign[i] = rdm[i].first;
        numFolds = (int)numFold;
        train = SequentialAccessSparseMatrix(); test = SequentialAccessSparseMatrix();
        return;                                                                              // the folds are cut by hasNextFold()
    } else if (splitter == "testset" || splitter == "net.librec.data.splitter.giventestsetdatasplitter") {
        // GivenTestSetDataSplitter.java:86-93: every (user, item) of the test matrix is zeroed in the train matrix
        for (int u = 0; u < preference.numRows; ++u) {
            const int32_t* tb = givenTest.col.data() + givenTest.rowptr[(size_t)u];
            const int32_t* te = givenTest.col.data() + givenTest.rowptr[(size_t)u + 1];
            for (int64_t e = preference.rowptr[(size_t)u]; e < preference.rowptr[(size_t)u + 1]; ++e)
                if (std::binary_search(tb, te, preference.col[(size_t)e])) isTrain[(size_t)e] = 0;
        }
        SequentialAccessSparseMatrix dropped;
        two_way(preference, isTrain, train, dropped);
        test = givenTest;
        return;
    } else {
        throw LibrecException("data.model.splitter=" + splitter + " is not implemented (ratio, kcv, loocv, givenn, testset are)");
    }
    two_way(preference, isTrain, train, test);
}

bool TextDataModel::hasNextFold() {
    if (foldCursor >= numFolds) return false;
    ++foldCursor;
    if (!assign.empty()) {
        std::vector<uint8_t> isTrain(assign.size());
        for (size_t e = 0; e < assign.size(); ++e) isTrain[e] = assign[e] != foldCursor;
        two_way(preference, isTrain, train, test);
    }
    return true;
}

void TextDataModel::buildDataModel() {
    buildConvert();
    buildSplitter();
    log.push_back("Transform data and split data set successfully!");                        // AbstractDataModel.java:110
}

RecommenderJob::RecommenderJob(const Configuration& c) : conf(c) {
    if (conf.has("rec.random.seed")) Randoms::seed(conf.getLong("rec.random.seed", 1));      // RecommenderJob.java:74-77
}
void RecommenderJob::setData(const SequentialAccessSparseMatrix& tr, const SequentialAccessSparseMatrix& te) { train = tr; test = te; }
// RecommenderJob.java:121-133 with a k-fold splitter: `while (dataModel.hasNextFold())` trains and evaluates once per fold on
// the SAME recommender instance, collects every evaluator value (collectCVResults :335-343) and prints the averages
// (printCVAverageResult :311-326); the recommended list that is saved is the last fold's.
void RecommenderJob::runCrossValidation() {
    recommender = newRecommender(conf.get("rec.recommender.class"));
    const bool ranking = conf.getBoolean("rec.recommender.isranking");
    std::map<std::string, std::vector<double>> cv;
    std::vector<std::string> lines(dataModel->log.begin(), dataModel->log.end());
    size_t logSeen = 0;
    while (dataModel->hasNextFold()) {
        dataModel->nextFold();
        train = dataModel->train; test = dataModel->test;
        recommender->train(conf, train, test);
        evaluatedMap.clear();
        if (conf.getBoolean("rec.eval.enable", true)) {
            if (ranking && recommender->rankingTopN() <= 64) recommendedList = recommender->recommendRankAndEvaluate(test, &evaluatedMap);
            else recommendedList = ranking ? recommender->recommendRank() : recommender->recommendRating(test);
            if (ranking && evaluatedMap.empty()) evaluateRanking(train, test, recommendedList, recommender->rankingTopN(), &evaluatedMap);
            if (!ranking) {
                evaluatedMap["RMSE"] = evaluateRMSE(test, recommendedList);
                evaluatedMap["MAE"] = evaluateMAE(test, recommendedList);
                evaluatedMap["MSE"] = evaluateMSE(test, recommendedList);
                evaluatedMap["MPE"] = evaluateMPE(test, recommendedList, conf.getDouble("rec.measure.mpe", 0.01));
            }
        } else {
            recommendedList = ranking ? recommender->recommendRank() : recommender->recommendRating(test);
        }
        const std::vector<std::string>& rl = recommender->log();                              // grows over the folds: take the new lines
        lines.insert(lines.end(), rl.begin() + (std::ptrdiff_t)logSeen, rl.end());
        logSeen = rl.size();
        for (const auto& kv : evaluatedMap) {
            lines.push_back("Evaluator value:" + kv.first + " is " + java_double_to_string(kv.second));
            cv[kv.first].push_back(kv.second);
        }
    }
    lines.push_back("Average Evaluation Result of Cross Validation:");
    for (const auto& kv : cv) {
        double sum = 0.0;
        for (double v : kv.second) sum += v;
        const double avg = sum / (double)kv.second.size();
        evaluatedMap[kv.first] = avg;                                                         // metric() then reports the average
        lines.push_back("Evaluator value:" + kv.first + " is " + java_double_to_string(avg));
    }
    log = lines;
}

void RecommenderJob::runJob() {
    if (train.numRows == 0 && conf.has("data.input.path")) {                                 // RecommenderJob.java:121-128
        dataModel.reset(new TextDataModel(conf));
        dataModel->buildDataModel();
        if (dataModel->numFolds > 1) { runCrossValidation(); return; }
        train = dataModel->train; test = dataModel->test;
    }
    recommender = newRecommender(conf.get("rec.recommender.class"));
    recommender->train(conf, train, test);
    const bool ranking = conf.getBoolean("rec.recommender.isranking");
    if (conf.getBoolean("rec.eval.enable", true)) {                                          // :205-271
        if (ranking && recommender->rankingTopN() <= 64) recommendedList = recommender->recommendRankAndEvaluate(test, &evaluatedMap);
        else recommendedList = ranking ? recommender->recommendRank() : recommender->recommendRating(test);
        if (ranking && evaluatedMap.empty()) evaluateRanking(train, test, recommendedList, recommender->rankingTopN(), &evaluatedMap);   // topN > 64
        if (!ranking) {
            evaluatedMap["RMSE"] = evaluateRMSE(test, recommendedList);             // eval/Measure.java:100-107: RMSE, MSE, MAE, MPE
            evaluatedMap["MAE"] = evaluateMAE(test, recommendedList);
            evaluatedMap["MSE"] = evaluateMSE(test, recommendedList);
            evaluatedMap["MPE"] = evaluateMPE(test, recommendedList, conf.getDouble("rec.measure.mpe", 0.01));
        }
    } else {
        recommendedList = ranking ? recommender->recommendRank() : recommender->recommendRating(test);
    }
    log = recommender->log();
    if (dataModel) log.insert(log.begin(), dataModel->log.begin(), dataModel->log.end());
    if (conf.has("rec.eval.classes") && conf.getBoolean("rec.eval.enable", true)) {
        // RecommenderJob.java:219-231: only the designated evaluators, logged as "Evaluator info:<SimpleName> is <value>"
        static const std::map<std::string, std::pair<const char*, const char*>> known = {
            {"auc", {"AUC", "AUCEvaluator"}}, {"ap", {"AP", "AveragePrecisionEvaluator"}}, {"ndcg", {"NDCG", "NormalizedDCGEvaluator"}},
            {"precision", {"PRECISION", "PrecisionEvaluator"}}, {"recall", {"RECALL", "RecallEvaluator"}}, {"rr", {"RR", "ReciprocalRankEvaluator"}},
            {"novelty", {"Novelty", "NoveltyEvaluator"}}, {"entropy", {"Entropy", "EntropyEvaluator"}}, {"hitrate", {"HitRate", "HitRateEvaluator"}},
            {"arhr", {"ARHR", "AverageReciprocalHitRankEvaluator"}}, {"idcg", {"IDCG", "IdealDCGEvaluator"}},
            {"rmse", {"RMSE", "RMSEEvaluator"}}, {"mse", {"MSE", "MSEEvaluator"}}, {"mae", {"MAE", "MAEEvaluator"}}, {"mpe", {"MPE", "MPEEvaluator"}}};
        std::string spec = conf.get("rec.eval.classes", "");
        for (char& c : spec) { if (c == ',') c = ' '; c = (char)std::tolower((unsigned char)c); }
        std::istringstream in(spec);
        std::vector<std::string> keys;
        for (std::string k; in >> k;) keys.push_back(k);
        const bool wantHitRate = std::find(keys.begin(), keys.end(), "hitrate") != keys.end();
        if (ranking) evaluateRankingExtra(test, recommendedList, recommender->rankingTopN(), wantHitRate, &evaluatedMap);
        std::map<std::string, double> designated;
        for (const std::string& k : keys) {
            auto it = known.find(k);
            if (it == known.end()) throw LibrecException("ClassNotFoundException: rec.eval.classes=" + k + " (diversity needs a similarity matrix and is not on this path)");
            const std::string name = ranking && k != "rmse" && k != "mse" && k != "mae" && k != "mpe"
                                         ? std::string(it->second.first) + " top " + std::to_string(recommender->rankingTopN()) : std::string(it->second.first);
            auto v = evaluatedMap.find(name);
            if (v == evaluatedMap.end()) throw LibrecException(std::string(it->second.second) + " does not apply to this kind of recommender (rec.recommender.isranking)");
            designated[it->second.second] = v->second;
        }
        evaluatedMap = designated;
        for (const auto& kv : evaluatedMap) log.push_back("Evaluator info:" + kv.first + " is " + java_double_to_string(kv.second));
        return;
    }
    for (const auto& kv : evaluatedMap) log.push_back("Evaluator value:" + kv.first + " is " + java_double_to_string(kv.second));   // :257-260
}

std::string RecommenderJob::saveResult() {
    if (recommendedList.size() == 0) return "";
    std::string algo = conf.get("rec.recommender.class");                                    // DriverClassUtil.getDriverName: the short name
    const std::string outputPath = conf.get("dfs.result.dir", "result") + "/" + conf.get("data.input.path", "data") + "-" + algo + "-output/" + algo;
    std::string out;
    out.reserve((size_t)recommendedList.size() * 16);
    for (size_t c = 0; c < recommendedList.lists.size(); ++c) {
        for (const KeyValue& kv : recommendedList.lists[c]) {
            // AbstractRecommender.java:213-235: raw ids through the inverse id maps; without a data model the inner ids are the ids
            const std::string uid = dataModel ? dataModel->userIds[c] : std::to_string(c);
            const std::string iid = dataModel ? dataModel->itemIds[(size_t)kv.key] : std::to_string(kv.key);
            if (uid.find_first_not_of(" \t\r\n") == std::string::npos || iid.find_first_not_of(" \t\r\n") == std::string::npos) continue;   // StringUtils.isNotBlank
            out += uid; out += ','; out += iid; out += ','; out += java_double_to_string(kv.value); out += '\n';
        }
    }
    // util/FileUtil.java:314-326 creates the parent directories
    for (size_t pos = outputPath.find('/', 1); pos != std::string::npos; pos = outputPath.find('/', pos + 1)) {
        const std::string d = outputPath.substr(0, pos);
        if (!d.empty()) mkdir(d.c_str(), 0777);
    }
    FILE* fp = fopen(outputPath.c_str(), "wb");
    if (!fp) throw LibrecException("saveResult: cannot write " + outputPath);
    fwrite(out.data(), 1, out.size(), fp);
    fclose(fp);
    log.push_back("Result path is " + outputPath);
    return outputPath;
}

}  // namespace librec
