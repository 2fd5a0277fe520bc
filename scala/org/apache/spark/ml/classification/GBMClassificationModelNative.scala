/*
 * GBMClassificationModelNative.scala — the reference's GBMClassificationModel with transform() evaluated per PARTITION on
 * the B200 instead of per row on the JVM (classification/GBMClassifier.scala:567-589:
 *     res = init.predictRaw(x); for (i <- models; j <- 0 until dim) res(j) += models(i)(j).predict(slice(subspaces(i))(x)) * weights(i)(j)
 *     binary dim 1: (-res(0), res(0)); probability by the loss's raw2probability, prediction = argmax).
 *
 * Two routes, both through org.apache.spark.ml.se.SeNative (include/se_abi.h):
 *   every member is a DecisionTreeRegressionModel with continuous splits and init is a DummyClassificationModel
 *       -> the partition's features go to HBM once (uploadRowmajor), the M·dim trees are flattened and concatenated in
 *          the order models(i)(j) (FlatTree, GBMRegressorNative.scala) with their feature indices mapped through
 *          subspaces(i), and SeNative.forestClassify writes rawPrediction, probability and prediction in one pass over
 *          the uint8 rank matrix (se_forest_classify: no [M][dim][n] intermediate);
 *   anything else
 *       -> each member predicts on the host into Slot.P ([M][dim][n]) and SeNative.aggRun forms the same three outputs
 *          (SE_AGG_GBM_CLASSIFIER); a non-constant init is added to the raw sums on the host first.
 * predict(features: Vector) for single rows stays the reference's.
 *
 * NOT COMPILED in this repository's image (no JDK / scalac / sbt / Spark jars).
 */
package org.apache.spark.ml.classification

import org.apache.spark.ml.ensemble.{EnsembleClassificationModelType, EnsemblePredictionModelType}
import org.apache.spark.ml.linalg.{Vector, Vectors}
import org.apache.spark.ml.param.ParamMap
import org.apache.spark.ml.regression.{DecisionTreeRegressionModel, FlatTree}
import org.apache.spark.ml.se.SeNative
import org.apache.spark.ml.se.SeNative.{Agg, Loss, Slot}
import org.apache.spark.ml.tree.{ContinuousSplit, InternalNode, Node}
import org.apache.spark.sql.{DataFrame, Dataset, Row}

class GBMClassificationModelNative(
    uid: String,
    numClasses: Int,
    weights: Array[Array[Double]],
    subspaces: Array[Array[Int]],
    models: Array[Array[EnsemblePredictionModelType]],
    init: EnsembleClassificationModelType,
    dim: Int,
    val device: Int = 0)
    extends GBMClassificationModel(uid, numClasses, weights, subspaces, models, init, dim) {

  private def continuousOnly(node: Node): Boolean = node match {
    case n: InternalNode => n.split.isInstanceOf[ContinuousSplit] && continuousOnly(n.leftChild) && continuousOnly(n.rightChild)
    case _ => true
  }

  private def lossId: Int = getLoss.toLowerCase match {
    case "logloss" => Loss.LogLoss
    case "bernoulli" => Loss.Bernoulli
    case "exponential" => Loss.Exponential
  }

  private def outClasses: Int = if (dim == 1 && numClasses == 2) 2 else dim

  // tree t = models(t / dim)(t % dim), feature indices mapped through subspaces(t / dim) (HasSubBag.slice, :81-84)
  private lazy val flatForest: Option[(Array[Int], FlatTree)] = {
    val members = models.flatten
    val trees = members.collect { case t: DecisionTreeRegressionModel if continuousOnly(t.rootNode) => t }
    if (trees.length != members.length || members.isEmpty) None
    else {
      val flats = trees.zipWithIndex.map { case (t, k) =>
        val sub = subspaces(k / dim)
        val f = FlatTree(t)
        f.copy(feature = f.feature.map(j => if (j < 0) j else sub(j)))
      }
      val offsets = flats.scanLeft(0)(_ + _.feature.length)
      Some((offsets, FlatTree(flats.flatMap(_.feature), flats.flatMap(_.threshold), flats.flatMap(_.left),
        flats.flatMap(_.right), flats.flatMap(_.value))))
    }
  }

  /** (rawPrediction, probability, prediction) of one partition, rows in partition order. */
  private[classification] def transformPartition(rows: Array[Vector]): Array[(Vector, Vector, Double)] = {
    val n = rows.length
    if (n == 0) return Array.empty
    val C = outClasses
    val ctx = SeNative.ctxCreate(device)
    try {
      flatForest match {
        case Some((offsets, forest)) if init.isInstanceOf[DummyClassificationModel] =>
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
          // a DummyClassificationModel's raw prediction is a constant: it is the `init` of the class sums (:569)
          SeNative.forestClassify(ctx, 0, Agg.GbmClassifier, numClasses, dim, lossId, models.length * dim, offsets,
            forest.feature, forest.threshold, forest.left, forest.right, forest.value, 1, weights.flatten,
            init.predictRaw(rows.head).toArray.take(dim))
        case _ =>
          SeNative.aggConfigure(ctx, Agg.GbmClassifier, math.max(models.length, 1), numClasses, dim, lossId, n.toLong)
          var i = 0
          while (i < models.length) {
            val sub = subspaces(i)
            var j = 0
            while (j < dim) {
              val member = models(i)(j)
              SeNative.uploadF64(ctx, Slot.P, rows.map(x => member.predict(slice(sub)(x))), n.toLong, (i.toLong * dim + j) * n)
              j += 1
            }
            i += 1
          }
          if (models.isEmpty) SeNative.fill(ctx, Slot.P, 0f, dim.toLong * n, 0L)
          val w = if (models.isEmpty) Array.fill(dim)(0.0) else weights.flatten
          if (init.isInstanceOf[DummyClassificationModel]) {
            SeNative.aggRun(ctx, w, init.predictRaw(rows.head).toArray.take(dim))
          } else {
            // a row-dependent init: the member sums come from the device, init and the epilogue stay on the host
            SeNative.aggRun(ctx, w, Array.fill(dim)(0.0))
            val raw = new Array[Float](C * n)
            SeNative.download(ctx, Slot.RAW, raw, C.toLong * n, 0L)
            return rows.indices.map { r =>
              val initRaw = init.predictRaw(rows(r)).toArray
              val res = Array.tabulate(dim)(j => initRaw(j) + (if (C == 2 && dim == 1) raw(n + r) else raw(j * n + r)))
              val rawVec = if (dim == 1 && numClasses == 2) Vectors.dense(-res(0), res(0)) else Vectors.dense(res)
              (rawVec, raw2probability(rawVec), raw2prediction(rawVec))
            }.toArray
          }
      }
      val raw = new Array[Float](C * n)
      val prob = new Array[Float](C * n)
      val label = new Array[Float](n)
      SeNative.download(ctx, Slot.RAW, raw, C.toLong * n, 0L)
      SeNative.download(ctx, Slot.PROB, prob, C.toLong * n, 0L)
      SeNative.download(ctx, Slot.LABEL, label, n.toLong, 0L)
      Array.tabulate(n) { r =>
        (Vectors.dense(Array.tabulate(C)(c => raw(c * n + r).toDouble)),
          Vectors.dense(Array.tabulate(C)(c => prob(c * n + r).toDouble)), label(r).toDouble)
      }
    } finally SeNative.ctxDestroy(ctx)
  }

  override def transform(dataset: Dataset[_]): DataFrame = {
    transformSchema(dataset.schema, logging = true)
    val spark = dataset.sparkSession
    val featuresIdx = dataset.schema.fieldIndex($(featuresCol))
    val vec = new org.apache.spark.ml.linalg.VectorUDT
    val outSchema = dataset.schema.add($(rawPredictionCol), vec).add($(probabilityCol), vec)
      .add($(predictionCol), org.apache.spark.sql.types.DoubleType)
    val model = this
    val rdd = dataset.toDF.rdd.mapPartitions { it =>
      val part = it.toArray
      val out = model.transformPartition(part.map(_.getAs[Vector](featuresIdx)))
      part.iterator.zip(out.iterator).map { case (row, (raw, prob, label)) => Row.fromSeq(row.toSeq :+ raw :+ prob :+ label) }
    }
    spark.createDataFrame(rdd, outSchema)
  }

  override def copy(extra: ParamMap): GBMClassificationModelNative =
    copyValues(new GBMClassificationModelNative(uid, numClasses, weights, subspaces, models, init, dim, device), extra)
      .setParent(parent)
}
