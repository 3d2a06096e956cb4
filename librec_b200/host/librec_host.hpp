// C++ mirror of the reference's plugin interface for the MF hot path (the Java toolchain is absent
// from this image, so the host side above the C ABI is written in C++ with the reference's own
// names, argument meaning, configuration keys, log lines and error behaviour).
//
//   net.librec.conf.Configuration                         -> librec::Configuration
//   net.librec.common.LibrecException                     -> librec::LibrecException
//   net.librec.math.algorithm.Randoms (java.util.Random)  -> librec::Randoms
//   net.librec.math.structure.DenseMatrix / VectorBasedDenseVector / SequentialAccessSparseMatrix
//   net.librec.recommender.item.RecommendedList / KeyValue
//   net.librec.recommender.{AbstractRecommender, MatrixRecommender, MatrixFactorizationRecommender}
//   net.librec.recommender.cuda.{BiasedMF,PMF,BPR}CudaRecommender   (the drop-in classes of INTEGRATION.md)
//   net.librec.eval.rating.{RMSE,MAE}Evaluator, net.librec.job.RecommenderJob (train + evaluate part)
// Paths in comments are relative to core/src/main/java/net/librec/ in the reference.
#pragma once
#include <cstdint>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/librec_b200.h"

namespace librec {

// common/LibrecException.java
struct LibrecException : public std::runtime_error {
    explicit LibrecException(const std::string& m) : std::runtime_error(m) {}
};

// java.lang.Double.toString / Float.toString (shortest repr; plain for 1e-3 <= |x| < 1e7, else d.dddE[-]n)
std::string java_double_to_string(double v);
std::string java_float_to_string(float v);

// conf/Configuration.java:182-417 (java.util.Properties semantics for the getters the path uses)
class Configuration {
public:
    void load_properties(const std::string& text);       // key=value lines, '#'/'!' comments
    void set(const std::string& k, const std::string& v) { props_[k] = v; }
    bool has(const std::string& k) const;
    std::string get(const std::string& k, const std::string& def = "") const;
    int getInt(const std::string& k, int def) const;                 // Configuration.java:199-207
    long long getLong(const std::string& k, long long def) const;
    float getFloat(const std::string& k, float def) const;           // Float.valueOf  (:232-239)
    double getDouble(const std::string& k, double def) const;        // Double.valueOf (:270-277)
    bool getBoolean(const std::string& k, bool def = false) const;   // Boolean.valueOf (:405-417)
private:
    std::map<std::string, std::string> props_;
};

// java.util.Random (JDK 8) behind math/algorithm/Randoms.java:31 -- ONE global generator
class Randoms {
public:
    static void seed(long long s);                        // Randoms.java:45-47
    static int uniform(int range);                        // Randoms.java:41-43 -> nextInt(bound)
    static double uniform();                              // Randoms.java:117-119 -> nextDouble
    static double gaussian(double mu, double sigma);      // Randoms.java:158-160 -> mu + sigma * nextGaussian
    // the generator's 48-bit state (Random.seed of Randoms.r), handed to and taken back from the reference-order BPR epochs on the
    // device; the cached Gaussian of nextGaussian is not part of it (BPR draws only nextInt)
    static uint64_t state();
    static void setState(uint64_t s);
};

// math/structure/DenseMatrix.java:20 (double[][] in Java; contiguous row-major here)
struct DenseMatrix {
    int rows = 0, cols = 0;
    std::vector<double> values;
    DenseMatrix() = default;
    DenseMatrix(int r, int c) : rows(r), cols(c), values((size_t)r * c, 0.0) {}
    double get(int r, int c) const { return values[(size_t)r * cols + c]; }            // :121
    void plus(int r, int c, double v) { values[(size_t)r * cols + c] += v; }           // :160
    const double* row(int r) const { return values.data() + (size_t)r * cols; }        // :136
    void init(double mean, double sigma);                                              // :95-97, row-major draws
};
// math/structure/VectorBasedDenseVector.java:14
struct VectorBasedDenseVector {
    std::vector<double> values;
    VectorBasedDenseVector() = default;
    explicit VectorBasedDenseVector(int n) : values((size_t)n, 0.0) {}
    double get(int i) const { return values[(size_t)i]; }
    void init(double mean, double sigma);                                              // DenseVector.java:26-28
};
// math/structure/SequentialAccessSparseMatrix.java:23 flattened (RowSequentialAccessSparseMatrix.java:19):
// row r = [rowptr[r], rowptr[r+1]) of (col ascending, val)
struct SequentialAccessSparseMatrix {
    int numRows = 0, numCols = 0;
    std::vector<int64_t> rowptr;
    std::vector<int32_t> col;
    std::vector<double> val;
    int rowSize() const { return numRows; }
    int columnSize() const { return numCols; }
    int64_t size() const { return (int64_t)col.size(); }
    double mean() const;                                   // RowSequentialAccessSparseMatrix.java:161-167
};

// recommender/item/KeyValue.java, RecommendedList.java:17
struct KeyValue { int key; double value; };
struct RecommendedList {
    std::vector<std::vector<KeyValue>> lists;
    int size() const { return (int)lists.size(); }
    void addList() { lists.emplace_back(); }                                           // :124-132
    void add(int ctx, int key, double value) { lists[(size_t)ctx].push_back({key, value}); }   // :134-151
};

// ---- recommenders ------------------------------------------------------------------------------
class AbstractRecommender {                                  // recommender/AbstractRecommender.java:39
public:
    virtual ~AbstractRecommender() = default;
    void train(const Configuration& conf, const SequentialAccessSparseMatrix& train, const SequentialAccessSparseMatrix& test);   // :143-150
    virtual RecommendedList recommendRank() = 0;
    virtual RecommendedList recommendRating(const SequentialAccessSparseMatrix& predictMatrix) = 0;
    virtual std::string simpleName() const = 0;
    const std::vector<std::string>& log() const { return log_; }
    double loss = 0.0, lastLoss = 0.0;
protected:
    virtual void setup();                                    // :110-128
    virtual void trainModel() = 0;                           // :135
    virtual void cleanup() {}
    bool isConverged(int iter);                              // :249-267
    void info(const std::string& line) { log_.push_back(line); }
    Configuration conf;
    const SequentialAccessSparseMatrix* trainMatrix = nullptr;
    const SequentialAccessSparseMatrix* testMatrix = nullptr;
    bool isRanking = false, earlyStop = false, verbose = true;
    int topN = 10;
    std::vector<std::string> log_;
};

class MatrixRecommender : public AbstractRecommender {       // recommender/MatrixRecommender.java:35
protected:
    void setup() override;                                   // :88-128
    virtual double predict(int userIdx, int itemIdx) = 0;    // :260
    double predict(int userIdx, int itemIdx, bool bound);    // :272-284
    int numUsers = 0, numItems = 0;
    int64_t numRates = 0;
    double maxRate = 0, minRate = 0, globalMean = 0;
    std::vector<double> ratingScale;
};

class MatrixFactorizationRecommender : public MatrixRecommender {   // recommender/MatrixFactorizationRecommender.java:12
protected:
    void setup() override;                                   // :67-94
    double predict(int userIdx, int itemIdx) override;       // :104-106
    void updateLRate(int iter);                              // :121-139
    float learnRate = 0.01f, maxLearnRate = 1000.0f, initMean = 0.0f, initStd = 0.001f, regUser = 0.01f, regItem = 0.01f, decay = 1.0f;
    bool isBoldDriver = false;
    int numFactors = 10, numIterations = 100;
    DenseMatrix userFactors, itemFactors, impUserFactors, impItemFactors;
};

// The drop-in: trainModel()/recommendRank()/recommendRating() forward to the C ABI (INTEGRATION.md section 2)
class MatrixFactorizationCudaRecommender : public MatrixFactorizationRecommender {
public:
    ~MatrixFactorizationCudaRecommender() override;
    RecommendedList recommendRank() override;                                               // MatrixRecommender.java:137-201
    RecommendedList recommendRank(const std::vector<int>& userIds);
    // recommendRank() for every user + the ranking evaluators of job/RecommenderJob.java:229-250 in one native call:
    // measures[] = AUC, AP, NDCG, PRECISION, RECALL, RR, Novelty, Entropy (eval/Measure.java names) at rec.recommender.ranking.topn
    int rankingTopN() const { return topN; }
    RecommendedList recommendRankAndEvaluate(const SequentialAccessSparseMatrix& test, std::map<std::string, double>* measures);
    RecommendedList recommendRating(const SequentialAccessSparseMatrix& predictMatrix) override;   // :211-248
    const DenseMatrix& getUserFactors() const { return userFactors; }
    const DenseMatrix& getItemFactors() const { return itemFactors; }
    const VectorBasedDenseVector& getUserBiases() const { return userBiases; }
    const VectorBasedDenseVector& getItemBiases() const { return itemBiases; }
    double getGlobalMean() const { return globalMean; }
protected:
    virtual int model() const = 0;
    void setup() override;
    void trainModel() override;
    void cleanup() override {}
    void check(int status) const;
    lrk_handle_t handle = nullptr;
    VectorBasedDenseVector userBiases, itemBiases;
    bool biased = false;
    double regBias = 0.0;
};
class BiasedMFCudaRecommender : public MatrixFactorizationCudaRecommender {     // cf/rating/BiasedMFRecommender.java:32
public:
    std::string simpleName() const override { return "BiasedMFCudaRecommender"; }
protected:
    int model() const override { return LRK_MODEL_BIASEDMF; }
    void setup() override;                                   // :54-64
    double predict(int userIdx, int itemIdx) override;       // :118-120
};
class PMFCudaRecommender : public MatrixFactorizationCudaRecommender {          // vanilla PMF, PMFSimilarityRecommender.java:59-90
public:
    std::string simpleName() const override { return "PMFCudaRecommender"; }
protected:
    int model() const override { return LRK_MODEL_PMF; }
};
class BPRCudaRecommender : public MatrixFactorizationCudaRecommender {          // cf/ranking/BPRRecommender.java:37
public:
    std::string simpleName() const override { return "BPRCudaRecommender"; }
protected:
    int model() const override { return LRK_MODEL_BPR; }
    // rec.cuda.order=reference: the device draws the samples from Randoms' own stream, continuing it where setup()'s factor init
    // left it, and hands the state back after training (the next kcv fold's init continues the same stream)
    void trainModel() override;
};

class RankSGDCudaRecommender : public MatrixFactorizationCudaRecommender {      // cf/ranking/RankSGDRecommender.java:37 (SURVEY 8f N3)
public:
    std::string simpleName() const override { return "RankSGDCudaRecommender"; }
protected:
    int model() const override { return LRK_MODEL_RANKSGD; }
};

// util/DriverClassUtil.java:79-88 : short name or fully-qualified class name -> recommender
std::unique_ptr<MatrixFactorizationCudaRecommender> newRecommender(const std::string& className);

// eval/rating/RMSEEvaluator.java:33-69, MAEEvaluator.java:34-70 : zip ground truth and predictions
double evaluateRMSE(const SequentialAccessSparseMatrix& test, const RecommendedList& recommended);
double evaluateMAE(const SequentialAccessSparseMatrix& test, const RecommendedList& recommended);
// eval/rating/MSEEvaluator.java:33-66, MPEEvaluator.java:33-73 (share of entries with |error| > rec.measure.mpe, default 0.01)
double evaluateMSE(const SequentialAccessSparseMatrix& test, const RecommendedList& recommended);
// the eight default ranking measures (eval/Measure.java:76-93) on the host; keys "<MEASURE> top <N>" like the job's log lines
void evaluateRankingExtra(const SequentialAccessSparseMatrix& test, const RecommendedList& recommended, int topN, bool wantHitRate,
                          std::map<std::string, double>* measures);   // HitRate (leave-one-out only), ARHR, IDCG
void evaluateRanking(const SequentialAccessSparseMatrix& train, const SequentialAccessSparseMatrix& test, const RecommendedList& recommended,
                     int topN, std::map<std::string, double>* measures);
double evaluateMPE(const SequentialAccessSparseMatrix& test, const RecommendedList& recommended, double mpe);

// data/model/TextDataModel.java + data/convertor/TextDataConvertor.java:136-200 + math/structure/DataFrame.java:237-261,370-379
// + data/splitter/RatioDataSplitter.java:136-156, straight into flat CSR arrays (SURVEY.md 8f, row N2): no per-line String[],
// no HashBasedTable<Integer,Integer,Double>, no per-row objects.  Semantics kept: fields split at every one of "\t;, " (empty
// interior fields survive, like Pattern.split), the first blank line ends a file, inner ids in first-seen order, on a duplicate
// (user,item) the EARLIEST line wins (the reference scans the frame backwards into a table), binThold >= 0 maps the rating to
// +1 / -1, rows sorted by item; the ratio splitter draws one Randoms.uniform() per entry in CSR order (< ratio -> train) and
// entries whose value is exactly 0.0 vanish from both sides (OrderedIntDoubleMapping.java:342-359).
struct TextDataModel {
    explicit TextDataModel(const Configuration& conf) : conf(conf) {}
    void buildDataModel();                           // AbstractDataModel.java:92-117: convert, then split
    void buildConvert();                             // reads dfs.data.dir + "/" + data.input.path (a file)
    // data.model.splitter = ratio (data.splitter.ratio = rating | user | item), kcv (data.splitter.cv.number), loocv
    // (data.splitter.loocv = user | item | userdate | itemdate), givenn (data.splitter.givenn = user | item | userdate |
    // itemdate, data.splitter.givenn.n), ratio also ratingdate | userdate | itemdate (UIRT input) and valid
    // (data.splitter.validset.ratio), testset (data.testset.path); ratio "userfixed" is not implemented (LibrecException)
    void buildSplitter();
    // AbstractDataModel.hasNextFold / nextFold over AbstractDataSplitter.nextFold (AbstractDataSplitter.java:104-128): one
    // fold for every splitter but kcv, which yields data.splitter.cv.number folds (fold k's test set = entries assigned k)
    bool hasNextFold();
    void nextFold() {}
    int foldsDone() const { return foldCursor; }
    Configuration conf;
    SequentialAccessSparseMatrix preference, train, test, valid;   // valid: data.splitter.ratio=valid only
    SequentialAccessSparseMatrix givenTest;          // data.model.splitter=testset: the matrix of data.testset.path
    std::vector<int64_t> datetime;                   // UIRT: Long.parseLong of the date column of the line that won, per stored entry
    std::vector<int32_t> assign;                     // kcv: fold id (1..K) per stored entry, CSR order
    int numFolds = 1, foldCursor = 0;
    std::vector<std::string> userIds, itemIds;       // inner id -> raw id (the BiMap inverses of DataFrame)
    std::vector<std::string> log;
};

// job/RecommenderJob.java:72-79,121-143,205-271 : seed -> [data model] -> instantiate -> train -> evaluate -> log lines -> save
struct RecommenderJob {
    explicit RecommenderJob(const Configuration& conf);
    void setData(const SequentialAccessSparseMatrix& train, const SequentialAccessSparseMatrix& test);
    void runJob();                                   // builds the TextDataModel first when no data was set and data.input.path is
    void runCrossValidation();                       // the fold loop of RecommenderJob.java:125-133 for data.model.splitter=kcv
    // job/RecommenderJob.java:281-306 + AbstractRecommender.java:213-235 (SURVEY.md 8f, row N4): "user,item,value\n" with raw ids,
    // values printed like String.valueOf(double); returns the path written ("" when there is nothing to write)
    std::string saveResult();
    Configuration conf;
    std::unique_ptr<TextDataModel> dataModel;
    SequentialAccessSparseMatrix train, test;
    std::unique_ptr<MatrixFactorizationCudaRecommender> recommender;
    std::map<std::string, double> evaluatedMap;     // "RMSE", "MAE", ...
    RecommendedList recommendedList;
    std::vector<std::string> log;
};

}  // namespace librec
