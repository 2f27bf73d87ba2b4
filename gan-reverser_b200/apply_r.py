"""Host-side mirror of apply_r.lua's four analysis modes and helpers.  Same names and argument
meaning as the reference; the inner loops are single calls into libganrev_cuda.so.  Each function
returns the data the reference would have drawn; present.py (SURVEY.md section 8f, rank 2) turns
those results into the reference's JPEG grids (saveClusterImages, saveSimilaritySearchImages,
saveFixedFaces, saveAnomalies).
"""
import math
import os

import numpy as np

from . import nn_utils


def cosineSimilarity(v1, v2, ctx=None):
    """apply_r.lua:396-400."""
    from .models import default_context
    return (ctx or default_context()).cosine(v1, v2)


def unsup_kmeans(x, k, niter, init=None, rng=None, ctx=None):
    """unsup.kmeans(x, k, niter) as called at apply_r.lua:198.  unsup draws N(0,1) centroids and
    divides each row by its norm; that draw happens here (seeded numpy) unless `init` is given.
    Returns centroids [k x d], totalcounts [k]."""
    from .models import default_context
    ctx = ctx or default_context()
    x = np.ascontiguousarray(x, dtype=np.float32)
    if init is None:
        rng = rng if rng is not None else np.random.default_rng(6)
        init = rng.normal(size=(k, x.shape[1])).astype(np.float32)
        init /= np.linalg.norm(init, axis=1, keepdims=True).astype(np.float32)
    ctx.db_set(x)
    cen, tot, _ = ctx.kmeans(k, niter, init, want_labels=False)
    return cen, tot


def createClusterImages(nbClusters, nbIterations, nbMaxPerCluster, images, attributes, init=None, ctx=None):
    """apply_r.lua:197-260.  Returns dict(centroids, counts, img2cluster (0-based), cos,
    member_ids [k x m] (-1 padded), member_counts, average_faces [k x C x H x W])."""
    from .models import default_context
    ctx = ctx or default_context()
    attributes = np.ascontiguousarray(attributes, dtype=np.float32)
    images = np.ascontiguousarray(images, dtype=np.float32)
    centroids, counts = unsup_kmeans(attributes, nbClusters, nbIterations, init=init, ctx=ctx)   # :198
    img2cluster, cos = ctx.assign_cosine_min(centroids)                                          # :206-218
    ids, cnt, mean = ctx.cluster_members(nbClusters, nbMaxPerCluster, images)                   # :222-243
    return {"centroids": centroids, "counts": counts, "img2cluster": img2cluster, "cos": cos,
            "member_ids": ids, "member_counts": cnt, "average_faces": mean.reshape((nbClusters,) + images.shape[1:])}


def createSimilaritySearchImages(nbSimilarNeedles, nbShowMax, images, attributes, ctx=None):
    """apply_r.lua:265-318.  Needle i (1-based) is row i*100 (:268), i.e. 0-based row i*100-1.
    Returns {"attributes": (ids, scores), "pixelwise": (ids, scores)}, ids 0-based [needles x n]."""
    from .models import default_context
    ctx = ctx or default_context()
    attributes = np.ascontiguousarray(attributes, dtype=np.float32)
    images = np.ascontiguousarray(images, dtype=np.float32)
    N = attributes.shape[0]
    n = min(nbShowMax, N)                                        # :281
    needles = np.array([i * 100 - 1 for i in range(1, nbSimilarNeedles + 1)])
    out = {}
    ctx.db_set(attributes)                                       # similarityMeasureAttributes :303-305
    out["attributes"] = ctx.search_rows(needles, n)            # the needles are rows of the searched tensor
    flat = images.reshape(N, -1)                                 # similarityMeasurePixelwise :308-314
    ctx.db_set(flat)
    out["pixelwise"] = ctx.search_rows(needles, n)
    return out


def fixFaces(nbPairs, nbFixedImages, images, attributesFixer, model_G):
    """apply_r.lua:324-352: G over the fixer's recovered vectors (pairs, then the first N)."""
    pairs_fixed = nn_utils.forwardBatched(model_G, attributesFixer[:nbPairs])                    # :328-332
    fixed = nn_utils.forwardBatched(model_G, attributesFixer[:nbFixedImages])                   # :349
    return {"pairs": (np.asarray(images[:nbPairs]), pairs_fixed), "unfixed": np.asarray(images[:nbFixedImages]),
            "fixed": fixed}


def detectAnomalies(nbImagesCalculations, nbImagesShow, threshold, images, noise, attributesFixer, model_G):
    """apply_r.lua:355-390.  `noise` is unused, as in the reference.  Returns (flags [nbImagesShow],
    similarities = 1 - dist [nbImagesCalculations], anomalyBelow)."""
    ctx = model_G.ctx
    fixed = nn_utils.forwardBatched(model_G, attributesFixer[:nbImagesCalculations])             # :361-363
    l2 = ctx.l2(np.asarray(images[:nbImagesCalculations]), fixed)                                # :366
    if math.floor(nbImagesCalculations * threshold) < 1:
        raise ValueError("floor(nbImagesCalculations*threshold) must be >= 1 (Lua would index nil)")
    flags, thr = ctx.anomaly_flags(l2, nbImagesCalculations, nbImagesShow, threshold)            # :370-378
    return flags.astype(bool), 1.0 - l2, thr


def refineAttributes(images, attributes, model_G, nbIterations, lr=0.01, prior=0.0, zclamp=0.0, slot=1):
    """New work (the reference stops at R's single pass, apply_r.lua:152-153): starting from R's guess `attributes`, nbIterations
    Adam steps per image on ||G(z) - x||^2 + prior ||z||^2 through G's backward pass on the GPU; |z| <= zclamp after every step when
    zclamp > 0.  The refined vectors stay resident in ATTRS_slot (default: the fixer's), the distances for ctx.anomaly_flags(None, ..).
    Returns (refined [N x nd], fixed = G(refined) [N x C x H x W], l2 = torch.dist per image [N])."""
    return model_G.ctx.refine_l2(slot, np.asarray(images, np.float32), np.asarray(attributes, np.float32), iters=nbIterations,
                                 lr=lr, prior=prior, zclamp=zclamp)


def main(G=None, R=None, R_fixer=None, writeTo="r_results", seed=1, dimensions=(1, 32, 32), noiseDim=100,
         noiseMethod="normal", colorSpace="y", nbImages=10000, ctx=None, write=True, refine=0):
    """apply_r.lua main() (apply_r.lua:59-192) end to end.  `G` / `R` / `R_fixer` are paths of Torch7 `.net`
    checkpoints (read with t7.py, geometry from G's `opt` as at :62-79) or None for seeded random-init
    networks of `dimensions` / `noiseDim`.  Same constants as the reference: 16 variation steps, 10,000
    faces, 20 clusters x 15 iterations x 71 members, 5 needles x top-100, 52 pairs / 528 fixed faces, 1024
    anomaly distances at the 15 % quantile.  Returns a dict of everything computed; with `write`, also
    saves the reference's JPEG files under `writeTo` (present.py).  refine > 0 (new work) also refines the fixer's vectors of the
    first 1024 faces by that many Adam steps through G (refineAttributes) and writes fixed_refined.jpg / anomalies_refined.jpg
    from them; refine = 0 leaves every output as it was."""
    from . import models, present
    from .models import default_context
    ctx = ctx or default_context()
    rng = np.random.default_rng(seed)
    if G is not None:
        model_G, opt = models.load_G(G, ctx=ctx)                                                  # :62-69
        dimensions, noiseDim = model_G.dimensions, model_G.noiseDim
        noiseMethod = opt.get("noiseMethod", noiseMethod)
        colorSpace = opt.get("colorSpace", colorSpace)
    else:
        model_G = models.create_G(dimensions, noiseDim, seed=seed, ctx=ctx)
    if R is not None:
        model_R = models.load_R(R, dimensions, noiseDim, noiseMethod, fixer=False, ctx=ctx)       # :92-94
    else:
        model_R = models.create_R(dimensions, noiseDim, noiseMethod, fixer=False, seed=seed + 1, ctx=ctx)
    if R_fixer == "":
        model_R_fixer = model_R                                                                   # :97-98
    elif R_fixer is not None:
        model_R_fixer = models.load_R(R_fixer, dimensions, noiseDim, noiseMethod, fixer=True, ctx=ctx)
    else:
        model_R_fixer = models.create_R(dimensions, noiseDim, noiseMethod, fixer=True, seed=seed + 2, ctx=ctx)
    out = {"dimensions": tuple(dimensions), "noiseDim": noiseDim, "files": []}

    # vary single components of one noise vector (:111-136)
    nbSteps = 16
    steps = np.linspace(-1, 1, nbSteps) if noiseMethod == "uniform" else np.linspace(-3, 3, nbSteps)
    base = nn_utils.createNoiseInputs(1, noiseDim, noiseMethod, rng=rng)
    noise = np.repeat(base, noiseDim * nbSteps, axis=0)
    for i in range(noiseDim):
        noise[i * nbSteps:(i + 1) * nbSteps, i] = steps
    out["variations"] = nn_utils.forwardBatched(model_G, noise)
    out["variation_noise"] = noise

    noise = nn_utils.createNoiseInputs(nbImages, noiseDim, noiseMethod, rng=rng)                  # :143
    images = nn_utils.forwardBatched(model_G, noise)                                              # :144
    attributes = nn_utils.forwardBatched(model_R, images)                                         # :150
    attributesFixer = nn_utils.forwardBatched(model_R_fixer, images)                              # :151
    out.update(noise=noise, images=images, attributes=attributes, attributesFixer=attributesFixer)

    nbClusters, nbIterations, nbMaxPerCluster = 20, 15, 64 + 7                                    # :158-161
    init = rng.normal(size=(nbClusters, attributes.shape[1])).astype(np.float32)
    init /= np.linalg.norm(init, axis=1, keepdims=True)
    out["clusters"] = createClusterImages(nbClusters, nbIterations, nbMaxPerCluster, images, attributes, init=init, ctx=ctx)
    out["similar"] = createSimilaritySearchImages(5, 100, images, attributes, ctx=ctx)            # :169-171
    out["fixed"] = fixFaces(52, 512 + 16, images, attributesFixer, model_G)                       # :178-180
    flags, sims, thr = detectAnomalies(1024, 512 + 16, 0.15, images, noise, attributesFixer, model_G)   # :186-190
    out["anomalies"] = {"flags": flags, "similarities": sims, "anomalyBelow": thr}
    if refine > 0:
        nRef = max(1024, 512 + 16)
        refined, fixed_r, l2_r = refineAttributes(images[:nRef], attributesFixer[:nRef], model_G, refine)
        flags_r, thr_r = ctx.anomaly_flags(l2_r, 1024, 512 + 16, 0.15)
        out["refined"] = {"attributes": refined, "fixed": fixed_r[:512 + 16], "flags": flags_r.astype(bool),
                          "similarities": 1.0 - l2_r, "anomalyBelow": thr_r}
    if write:
        out["files"].append(present.save(os.path.join(writeTo, "variations.jpg"),
                                         present.toDisplayTensor(out["variations"], nrow=nbSteps, min=0, max=1.0)))
        out["files"] += present.saveClusterImages(out["clusters"], images, colorSpace, writeTo)
        out["files"] += present.saveSimilaritySearchImages(out["similar"], images, colorSpace, writeTo)
        out["files"] += present.saveFixedFaces(out["fixed"], colorSpace, writeTo)
        out["files"].append(present.saveAnomalies(images, flags, colorSpace, writeTo))
        if refine > 0:
            r = out["refined"]
            n = r["fixed"].shape[0]
            out["files"].append(present.save(os.path.join(writeTo, "fixed_refined.jpg"),
                                             present.toDisplayTensor(r["fixed"], nrow=int(math.floor(math.sqrt(n))), min=0, max=1.0)))
            out["files"].append(present.save(os.path.join(writeTo, "anomalies_refined.jpg"),
                                             present.anomalyGrid(np.asarray(images)[:len(r["flags"])], r["flags"], colorSpace)))
    return out
