// NOT COMPILED HERE.  rec.recommender.class=net.librec.recommender.cuda.BPRCudaRecommender
package net.librec.recommender.cuda;

import java.lang.reflect.Field;
import java.nio.ByteBuffer;
import java.nio.ByteOrder;
import java.nio.charset.StandardCharsets;
import java.util.Random;
import java.util.concurrent.atomic.AtomicLong;

import net.librec.common.LibrecException;
import net.librec.math.algorithm.Randoms;

public class BPRCudaRecommender extends MatrixFactorizationCudaRecommender {
    private static final byte[] STATE = "jdk.random.state".getBytes(StandardCharsets.UTF_8);

    @Override int model() { return LibrecB200.MODEL_BPR; }

    private boolean referenceOrder() { return "reference".equals(conf.get("rec.cuda.order", "shuffled")); }

    // Randoms.r (math/algorithm/Randoms.java:31) and its java.util.Random.seed: JDK 9 and later need
    // --add-opens java.base/java.util=ALL-UNNAMED for the second (INTEGRATION.md)
    private static AtomicLong generatorSeed() throws LibrecException {
        try {
            Field r = Randoms.class.getDeclaredField("r");
            r.setAccessible(true);
            Field seed = Random.class.getDeclaredField("seed");
            seed.setAccessible(true);
            return (AtomicLong) seed.get(r.get(null));
        } catch (ReflectiveOperationException | RuntimeException e) {
            throw new LibrecException("rec.cuda.order=reference for BPR reads Randoms.r's state: " + e);
        }
    }

    /** rec.cuda.order=reference: the device draws BPRRecommender.java:54-67's samples from Randoms' own stream, continuing it
     *  where setup()'s factor init left it, and the state comes back after training (a kcv run's next fold continues it). */
    @Override
    protected void trainModel() throws LibrecException {
        if (!referenceOrder()) { super.trainModel(); return; }
        AtomicLong seed = generatorSeed();
        ByteBuffer s = ByteBuffer.allocateDirect(8).order(ByteOrder.nativeOrder());
        s.putDouble(0, (double) seed.get());                        // 48-bit state: exact as a double
        check(LibrecB200.setMatrix(handle, STATE, s));
        super.trainModel();
        check(LibrecB200.getMatrix(handle, STATE, s));
        seed.set((long) s.getDouble(0));
    }
}
