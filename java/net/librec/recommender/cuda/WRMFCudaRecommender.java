// NOT COMPILED HERE.  rec.recommender.class=net.librec.recommender.cuda.WRMFCudaRecommender
// Replaces the trainModel() of recommender/cf/ranking/WRMFRecommender.java:74-166 (alternating least squares, one Gauss-Jordan
// inverse per user and per item and iteration); rec.factor.number <= 112.  rec.cuda.devices=0,1,... trains on several GPUs of one
// box through one multi-device handle (each device solves a range of users and of items, the new rows are exchanged between the
// devices after each half-iteration), with the same bit-identical factors as one GPU.  setup() keeps the reference's
// weightMatrix() (:63-72) in Java -- Math.log / Math.pow are evaluated by the JVM exactly as before -- and the native side receives
// the weighted values.  The native iteration performs the reference's floating-point operations in the reference's order in fp64,
// so userFactors / itemFactors come back bit-identical to what WRMFRecommender would have computed; recommendRank is the native
// top-N (prediction = p_u . q_i, as MatrixFactorizationRecommender.predict).
package net.librec.recommender.cuda;

import it.unimi.dsi.fastutil.doubles.Double2DoubleOpenHashMap;

import net.librec.common.LibrecException;
import net.librec.math.structure.MatrixEntry;

public class WRMFCudaRecommender extends MatrixFactorizationCudaRecommender {
    protected float weightCoefficient;

    @Override int model() { return LibrecB200.MODEL_WRMF; }

    public double weight(double value) {                                   // WRMFRecommender.java:58-61
        return Math.log(1.0 + Math.pow(10, weightCoefficient) * value);
    }

    @Override
    protected void beforeStage() throws LibrecException {                  // WRMFRecommender.java:50-72
        weightCoefficient = conf.getFloat("rec.wrmf.weight.coefficient", 4.0f);
        Double2DoubleOpenHashMap ratingWeightMap = new Double2DoubleOpenHashMap();
        for (double rating : ratingScale) ratingWeightMap.putIfAbsent(rating, weight(rating));
        for (MatrixEntry matrixEntry : trainMatrix) matrixEntry.set(ratingWeightMap.get(matrixEntry.get()));
    }
}
