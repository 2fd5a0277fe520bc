/*
 * BoostingRegressionModelNative.scala — the reference's BoostingRegressionModel (AdaBoost.R2) with transform() evaluated
 * per PARTITION on the B200 instead of per row on the JVM (regression/BoostingRegressor.scala:333-342:
 *     median: Utils.weightedMedian(models.map(_.predict(x)), weights)      (ensemble/Utils.scala:26-40)
 *     mean:   BLAS.dot(predictions, weights) / sumWeights).
 *
 * Routes, all through org.apache.spark.ml.se.SeNative (include/se_abi.h):
 *   every member is a DecisionTreeRegressionModel with continuous splits
 *       -> the partition's features go to HBM once (uploadRowmajor), the trees are flattened and concatenated in model
 *          order (FlatTree, GBMRegressorNative.scala), and
 *            median: SeNative.forestWeightedMedian selects the weighted median of the leaves in one pass over the uint8
 *                    rank matrix (se_forest_weighted_median: no [M][n] intermediate, the bits of the member route);
 *            mean:   SeNative.forestPredict sums weights(i) / Σ weights · tree_i(x) (Σ in fp64, model order);
 *          a RuntimeException (SE_ERR_STATE: more than 64 members, a forest beyond one chunk of the kernel's shared
 *          memory, a column with more than 255 thresholds) falls through to the member route;
 *   anything else
 *       -> each member predicts on the host into Slot.P ([M][n]) and SeNative.aggRun aggregates
 *          (SE_AGG_BOOSTING_REG_MEDIAN / SE_AGG_BOOSTING_REG_MEAN).
 * predict(features: Vector) for single rows stays the reference's.
 *
 * NOT COMPILED in this repository's image (no JDK / scalac / sbt / Spark jars).
 */
package org.apache.spark.ml.regression

import org.apache.spark.ml.ensemble.EnsemblePredictionModelType
import org.apache.spark.ml.linalg.Vector
import org.apache.spark.ml.param.ParamMap
import org.apache.spark.ml.se.SeNative
import org.apache.spark.ml.se.SeNative.{Agg, Slot}
import org.apache.spark.ml.tree.{ContinuousSplit, InternalNode, Node}
import org.apache.spark.sql.{DataFrame, Dataset, Row}

class BoostingRegressionModelNative(
    uid: String,
    weights: Array[Double],
    models: Array[EnsemblePredictionModelType],
    val device: Int = 0)
    extends BoostingRegressionModel(uid, weights, models) {

  private def continuousOnly(node: Node): Boolean = node match {
    case n: InternalNode => n.split.isInstanceOf[ContinuousSplit] && continuousOnly(n.leftChild) && continuousOnly(n.rightChild)
    case _ => true
  }

  private def median: Boolean = getVotingStrategy.toLowerCase == "median"

  private lazy val flatForest: Option[(Array[Int], FlatTree)] = {
    val trees = models.collect { case t: DecisionTreeRegressionModel if continuousOnly(t.rootNode) => t }
    if (trees.length != models.length || models.isEmpty) None
    else {
      val flats = trees.map(FlatTree(_))
      val offsets = flats.scanLeft(0)(_ + _.feature.length)
      Some((offsets, FlatTree(flats.flatMap(_.feature), flats.flatMap(_.threshold), flats.flatMap(_.left),
        flats.flatMap(_.right), flats.flatMap(_.value))))
    }
  }

  /** One pass over the resident rows into Slot.RAW; false when the forest is beyond the kernel (SE_ERR_STATE). */
  private def forestPartition(ctx: Long, rows: Array[Vector], offsets: Array[Int], forest: FlatTree): Boolean = {
    val n = rows.length
    val d = rows.head.size
    SeNative.slotAlloc2d(ctx, Slot.X, d.toLong, n.toLong)
    val chunk = math.max(1, (1 << 22) / d)
    var done = 0
    while (done < n) {
      val m = math.min(chunk, n - done)
      val buf = new Array[Float](m * d)
      var r = 0
      while (r < m) { rows(done + r).foreachActive((j, x) => buf(r * d + j) = x.toFloat); r += 1 }
      SeNative.uploadRowmajor(ctx, Slot.X, buf, m.toLong, d, done.toLong)
      done += m
    }
    SeNative.slotAlloc2d(ctx, Slot.RAW, 1L, n.toLong)
    try {
      if (median) {
        SeNative.forestWeightedMedian(ctx, 0, models.length, offsets, forest.feature, forest.threshold, forest.left,
          forest.right, forest.value, weights, Slot.RAW, 0)
      } else {
        var sumW = 0.0
        weights.foreach(a => sumW += a)  // fp64, model order
        SeNative.forestPredict(ctx, 0, models.length, offsets, forest.feature, forest.threshold, forest.left,
          forest.right, forest.value, weights.map(_ / sumW), 0.0, Slot.RAW, 0)
      }
      true
    } catch {
      case e: IllegalArgumentException => throw e  // SE_ERR_ARG: not a forest the reference could have built
      case _: RuntimeException => false           // SE_ERR_STATE: the member route below
    }
  }

  /** Predictions of one partition (rows in partition order). */
  private[regression] def predictPartition(rows: Array[Vector]): Array[Double] = {
    val n = rows.length
    if (n == 0) return Array.emptyDoubleArray
    val ctx = SeNative.ctxCreate(device)
    try {
      val viaForest = flatForest match {
        case Some((offsets, forest)) => forestPartition(ctx, rows, offsets, forest)
        case None => false
      }
      if (!viaForest) {
        SeNative.aggConfigure(ctx, if (median) Agg.BoostingRegMedian else Agg.BoostingRegMean, models.length, 0, 1, 0,
          n.toLong)
        var i = 0
        while (i < models.length) {
          val member = models(i)
          SeNative.uploadF64(ctx, Slot.P, rows.map(x => member.predict(x)), n.toLong, i.toLong * n)
          i += 1
        }
        SeNative.aggRun(ctx, weights, Array(0.0))
      }
      val out = new Array[Float](n)
      SeNative.download(ctx, Slot.RAW, out, n.toLong, 0L)
      out.map(_.toDouble)
    } finally SeNative.ctxDestroy(ctx)
  }

  override def transform(dataset: Dataset[_]): DataFrame = {
    transformSchema(dataset.schema, logging = true)
    val spark = dataset.sparkSession
    val featuresIdx = dataset.schema.fieldIndex($(featuresCol))
    val outSchema = dataset.schema.add($(predictionCol), org.apache.spark.sql.types.DoubleType)
    val model = this
    val rdd = dataset.toDF.rdd.mapPartitions { it =>
      val part = it.toArray
      val pred = model.predictPartition(part.map(_.getAs[Vector](featuresIdx)))
      part.iterator.zip(pred.iterator).map { case (row, p) => Row.fromSeq(row.toSeq :+ p) }
    }
    spark.createDataFrame(rdd, outSchema)
  }

  override def copy(extra: ParamMap): BoostingRegressionModelNative =
    copyValues(new BoostingRegressionModelNative(uid, weights, models, device), extra).setParent(parent)
}
