/*
 * GBMRegressorNative.scala — the reference's GBMRegressor with its train() body rewired onto the B200 hot path.
 *
 * What stays exactly as in the reference (regression/GBMRegressor.scala:237-476): Params, instrumentation, the
 * train/validation split, the init model (DummyRegressor / base learner), sub-spaces (HasSubBag.subspace), the base
 * learner fit (third party), commons-math3's BrentOptimizer with SearchInterval(0, 100, 1) / MaxEval(maxIter), the
 * early-stop bookkeeping and the returned GBMRegressionModel(weights, subspaces, models, init).
 * What moves to the GPU (one SeNative call each, include/se_abi.h): every per-row RDD closure —
 *   :342-353 huber delta (approxQuantile of |y - F|)      -> SeNative.quantile(ctx, 1, ...)   (exact order statistic)
 *   :368-385 pseudo-residuals (gradient / newton)          -> SeNative.gbmPseudoResiduals, fused into gbmUpdate afterwards
 *   :398-425 RDDLossFunction + GBMLossAggregator           -> SeNative.gbmLinesearchEval (one pass per Brent evaluation)
 *                                                             or SeNative.gbmRound (statistics + Brent + update in ONE launch)
 *   :434-442 F += weight * direction                       -> SeNative.gbmUpdate (fused with the next residuals + loss)
 *   :444-465 validation update + mean loss                 -> SeNative.gbmUpdateValidation
 * State (y, w, F, h, r and optionally the column-major feature matrix) lives in HBM for the whole fit; per round only
 * the pseudo-residuals (device -> host, the base learner's labels) and the direction (host -> device, or a tree
 * evaluated on device with SeNative.treePredict) move.
 *
 * NOT COMPILED in this repository's image (no JDK / scalac / sbt / Spark jars).  It lives in package
 * org.apache.spark.ml.regression because it uses the same private[ml] members as the reference.
 */
package org.apache.spark.ml.regression

import org.apache.commons.math3.optim.{MaxEval, MaxIter}
import org.apache.commons.math3.optim.nonlinear.scalar.GoalType
import org.apache.commons.math3.optim.univariate.{BrentOptimizer, SearchInterval, UnivariateObjectiveFunction}
import org.apache.commons.math3.analysis.UnivariateFunction
import org.apache.spark.ml.ensemble.{EnsemblePredictionModelType, Utils}
import org.apache.spark.ml.feature.Instance
import org.apache.spark.ml.linalg.Vector
import org.apache.spark.ml.param.{BooleanParam, IntParam, ParamMap}
import org.apache.spark.ml.se.SeNative
import org.apache.spark.ml.se.SeNative.{Loss, Slot, Upd}
import org.apache.spark.ml.util.Instrumentation.instrumented
import org.apache.spark.ml.util.MetadataUtils
import org.apache.spark.sql.Dataset
import org.apache.spark.sql.functions.{col, not}

class GBMRegressorNative(override val uid: String) extends GBMRegressor(uid) {

  /** GPU ordinal of the context this fit runs on (one context == one GPU == one row shard). */
  val device = new IntParam(this, "device", "CUDA device ordinal")
  /** Keep the column-major feature matrix in HBM and evaluate fitted trees on device (SeNative.treePredict). */
  val residentFeatures = new BooleanParam(this, "residentFeatures", "evaluate base models on device")
  /** squared loss: line search + update as ONE native call (se_gbm_round; Brent with commons-math semantics on device). */
  val nativeRound = new BooleanParam(this, "nativeRound", "statistics + Brent + update in one kernel launch")
  setDefault(device -> 0, residentFeatures -> false, nativeRound -> true)

  private def lossId(name: String): Int = name match {
    case "squared" => Loss.Squared; case "absolute" => Loss.Absolute
    case "huber" => Loss.Huber; case "quantile" => Loss.Quantile
  }

  override protected def train(dataset: Dataset[_]): GBMRegressionModel = instrumented { instr =>
    instr.logPipelineStage(this)
    instr.logDataset(dataset)
    val spark = dataset.sparkSession
    val withValidation = isDefined(validationIndicatorCol) && $(validationIndicatorCol).nonEmpty
    val (trainRows, validRows) =
      if (withValidation)
        (extractInstances(dataset.filter(not(col($(validationIndicatorCol))))).collect(),
          extractInstances(dataset.filter(col($(validationIndicatorCol)))).collect())
      else (extractInstances(dataset).collect(), Array.empty[Instance])
    val n = trainRows.length.toLong
    val nv = validRows.length.toLong
    val numFeatures = MetadataUtils.getNumFeatures(dataset, $(featuresCol))
    val hasWeights = trainRows.exists(_.weight != 1.0)

    val models = Array.ofDim[EnsemblePredictionModelType]($(numBaseLearners))
    val subspaces = Array.tabulate($(numBaseLearners))(i => subspace($(subspaceRatio), numFeatures, $(seed) + i))
    val weights = Array.ofDim[Double]($(numBaseLearners))
    val trainDF = spark.createDataFrame(spark.sparkContext.parallelize(trainRows))
    val init = initModel(trainDF)                                      // reference :287-303, unchanged (see below)
    var quantile = getLoss match {                                     // :305-308
      case "huber" => dataset.stat.approxQuantile("label", Array($(alpha)), $(tol))(0)
      case _ => $(alpha)
    }
    val newton = getUpdates == "newton" && getLoss == "squared"        // HasScalarHessian among the selectable losses :369
    val optimizer = new BrentOptimizer($(tol), $(tol))                 // :311

    val ctx = SeNative.ctxCreate($(device))
    try {
      SeNative.gbmConfigure(ctx, n, nv, 1, lossId(getLoss), quantile, hasWeights)
      SeNative.uploadF64(ctx, Slot.Y, trainRows.map(_.label), n, 0)
      if (hasWeights) SeNative.uploadF64(ctx, Slot.W, trainRows.map(_.weight), n, 0)
      SeNative.uploadF64(ctx, Slot.F, trainRows.map(r => init.predict(r.features)), n, 0)           // :313
      if (withValidation) {
        SeNative.uploadF64(ctx, Slot.VY, validRows.map(_.label), nv, 0)
        SeNative.uploadF64(ctx, Slot.VF, validRows.map(r => init.predict(r.features)), nv, 0)       // :324
      }
      if ($(residentFeatures)) {
        SeNative.slotAlloc2d(ctx, Slot.X, numFeatures, n)
        uploadFeatures(ctx, Slot.X, trainRows.map(_.features), numFeatures)
        if (withValidation) { SeNative.slotAlloc2d(ctx, Slot.VX, numFeatures, nv); uploadFeatures(ctx, Slot.VX, validRows.map(_.features), numFeatures) }
      }
      // RDD.sample(replacement, subsampleRatio, seed) uses the SAME seed every round (:357-359): one bag per fit.
      val bagCounts: Option[Array[Float]] =
        if ($(subsampleRatio) == 1.0 && !$(replacement)) None
        else Some(sparkBagCounts(trainRows.length, $(replacement), $(subsampleRatio), $(seed)))
      bagCounts.foreach { c => SeNative.gbmSetBag(ctx, true); SeNative.upload(ctx, Slot.BAG, c, n, 0) }
      var bestValidationError = if (withValidation) SeNative.gbmMeanLoss(ctx, 1) else 0.0           // :330-335

      val residuals = new Array[Float](trainRows.length)
      val newWeights = new Array[Float](trainRows.length)
      val sumHess = new Array[Double](1)
      SeNative.gbmPseudoResiduals(ctx, newton, sumHess)                // residuals of F0; later rounds: fused into the update
      var i = 0
      var v = 0
      while (i < $(numBaseLearners) && v < $(numRounds)) {             // :340
        if (getLoss == "huber") {                                      // :342-353
          quantile = SeNative.quantile(ctx, 1, 0, 0, $(alpha))
          SeNative.gbmSetLossParam(ctx, quantile)
          SeNative.gbmPseudoResiduals(ctx, false, sumHess)
        }
        val sub = subspaces(i)
        SeNative.download(ctx, Slot.R, residuals, n, 0)                // the base learner's labels (:368-385)
        if (newton) SeNative.download(ctx, Slot.WOUT, newWeights, n, 0)
        val pseudo = trainRows.indices.flatMap { k =>                  // the bag, with multiplicities
          val c = bagCounts.map(_(k).toInt).getOrElse(1)
          val inst = Instance(residuals(k), if (newton) newWeights(k) else trainRows(k).weight, slice(sub)(trainRows(k).features))
          Iterator.fill(c)(inst)
        }
        val df = spark.createDataFrame(spark.sparkContext.parallelize(pseudo))
          .withColumn("features", col("features"), Utils.getFeaturesMetadata(dataset, $(featuresCol), Some(sub)))
        val model = fitBaseLearner($(baseLearner), "label", "features", $(predictionCol), Some("weight"))(df)  // third party

        setDirection(ctx, model, sub, trainRows, Slot.H, Slot.X)       // :405: h = model.predict(slice(x))
        val solution =
          if (!$(optimizedWeights)) 1.0
          else if ($(nativeRound) && getLoss == "squared" && !newton) Double.NaN   // taken by gbmRound below
          else {
            // the reference's optimiser, untouched: every evaluation is one streaming pass on the GPU (:398-425)
            val objective = new UnivariateObjectiveFunction(new UnivariateFunction {
              override def value(x: Double): Double = SeNative.gbmLinesearchEval(ctx, Array(x), null)
            })
            optimizer.optimize(objective, new SearchInterval(0, 100, 1), GoalType.MINIMIZE,
              new MaxIter($(maxIter)), new MaxEval($(maxIter))).getPoint
          }
        val flags = if (newton) Upd.Newton | Upd.Loss else if (getLoss == "huber") Upd.Loss else Upd.Residual | Upd.Loss
        val weight =
          if (solution.isNaN) {
            // one cooperative launch: statistics -> Brent (commons-math semantics) -> F update + next residuals
            val r = SeNative.gbmRound(ctx, $(learningRate), true, $(tol), $(maxIter), flags)
            $(learningRate) * r(0)                                     // :427
          } else {
            val w = $(learningRate) * solution
            SeNative.gbmUpdate(ctx, Array(w), flags, sumHess)          // :434-442 (+ :368-385 for the next round)
            w
          }
        models(i) = model
        weights(i) = weight
        if (withValidation) {                                          // :444-465
          setDirection(ctx, model, sub, validRows, Slot.VH, Slot.VX)
          val validationError = SeNative.gbmUpdateValidation(ctx, Array(weight))
          if (bestValidationError - validationError < $(validationTol) * math.max(validationError, 0.01)) v += 1
          else if (validationError < bestValidationError) { bestValidationError = validationError; v = 0 }
        }
        i += 1
      }
      new GBMRegressionModel(weights.take(i - v), subspaces.take(i - v), models.take(i - v), init)  // :474
    } finally {
      SeNative.ctxDestroy(ctx)
    }
  }

  /** The reference's init-model selection (:287-303), factored out unchanged. */
  private def initModel(trainDF: org.apache.spark.sql.DataFrame): EnsemblePredictionModelType = getInitStrategy match {
    case "base" => fitBaseLearner($(baseLearner), "label", "features", $(predictionCol), Some("weight"))(trainDF)
    case "zero" => new DummyRegressor().setStrategy("constant").setConstant(0.0).fit(trainDF)
    case "constant" => (getLoss match {
      case "squared" => new DummyRegressor().setStrategy("mean")
      case "absolute" | "huber" => new DummyRegressor().setStrategy("median")
      case "quantile" => new DummyRegressor().setStrategy("quantile").setQuantile($(alpha))
    }).fit(trainDF)
  }

  /** Direction of this round into `slot`: a Spark decision tree is flattened and evaluated on device over the resident
   *  feature matrix; anything else is predicted on the host and uploaded (the reference's path). */
  private def setDirection(ctx: Long, model: EnsemblePredictionModelType, sub: Array[Int], rows: Array[Instance],
      slot: Int, xSlot: Int): Unit = model match {
    case tree: DecisionTreeRegressionModel if $(residentFeatures) =>
      val t = FlatTree(tree)  // pre-order arrays: feature (-1 = leaf), threshold, left, right, value
      SeNative.treePredict(ctx, if (xSlot == Slot.VX) 1 else 0, t.feature.length, t.feature, t.threshold, t.left, t.right,
        t.value, sub, sub.length, slot, 0)
    case _ =>
      SeNative.uploadF64(ctx, slot, rows.map(r => model.predict(slice(sub)(r.features))), rows.length.toLong, 0)
  }

  private def uploadFeatures(ctx: Long, slot: Int, rows: Array[Vector], d: Int): Unit = {
    val chunk = math.max(1, (1 << 22) / d)
    var done = 0
    while (done < rows.length) {
      val m = math.min(chunk, rows.length - done)
      val buf = new Array[Float](m * d)
      var r = 0
      while (r < m) { rows(done + r).foreachActive((j, x) => buf(r * d + j) = x.toFloat); r += 1 }
      SeNative.uploadRowmajor(ctx, slot, buf, m.toLong, d, done.toLong)   // transposed to column-major on the device
      done += m
    }
  }

  /** Multiplicities of RDD.sample(replacement, ratio, seed) over one partition, drawn with Spark's own samplers so the
   *  bag is the one the reference would draw (BernoulliSampler / PoissonSampler are Spark classes, used as is). */
  private def sparkBagCounts(n: Int, replacement: Boolean, ratio: Double, seed: Long): Array[Float] = {
    import org.apache.spark.util.random.{BernoulliSampler, PoissonSampler}
    val counts = new Array[Float](n)
    val sampler = if (replacement) new PoissonSampler[Int](ratio) else new BernoulliSampler[Int](ratio)
    sampler.setSeed(seed)   // partition 0; with several partitions RDD.sample seeds each with seed + index
    sampler.sample(Iterator.range(0, n)).foreach(k => counts(k) += 1f)
    counts
  }

  override def copy(extra: ParamMap): GBMRegressorNative = defaultCopy(extra)
}

/** Pre-order flattening of a Spark regression tree into the arrays se_tree_predict takes (continuous splits only). */
private[ml] case class FlatTree(feature: Array[Int], threshold: Array[Float], left: Array[Int], right: Array[Int], value: Array[Float])
private[ml] object FlatTree {
  import org.apache.spark.ml.tree.{ContinuousSplit, InternalNode, LeafNode, Node}
  def apply(model: DecisionTreeRegressionModel): FlatTree = {
    val f = scala.collection.mutable.ArrayBuffer[Int](); val t = scala.collection.mutable.ArrayBuffer[Float]()
    val l = scala.collection.mutable.ArrayBuffer[Int](); val r = scala.collection.mutable.ArrayBuffer[Int]()
    val v = scala.collection.mutable.ArrayBuffer[Float]()
    def visit(node: Node): Int = {
      val id = f.length
      f += -1; t += 0f; l += 0; r += 0; v += node.prediction.toFloat
      node match {
        case n: InternalNode =>
          val s = n.split.asInstanceOf[ContinuousSplit]  // categorical splits: fall back to the host path upstream
          f(id) = s.featureIndex
          // x <= threshold goes left on the JVM in fp64; the device compares fp32: round the threshold DOWN so that a
          // feature value that narrows onto it cannot change sides (se_abi.h se_tree_predict)
          val tf = s.threshold.toFloat
          t(id) = if (tf.toDouble > s.threshold) java.lang.Math.nextDown(tf) else tf   // the largest float <= threshold
          l(id) = visit(n.leftChild)
          r(id) = visit(n.rightChild)
        case _: LeafNode => ()
      }
      id
    }
    visit(model.rootNode)
    FlatTree(f.toArray, t.toArray, l.toArray, r.toArray, v.toArray)
  }
}
