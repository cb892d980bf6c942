"""Host-side callers and data formats either side of the device path (SURVEY.md 8b: "the replacement package must be
importable as np_bnn and satisfy the five scripts unchanged").

Everything here is file / table / bookkeeping code around the MCMC hot path: reading the tab-separated inputs
(`get_data`, reference np_bnn/BNN_files.py:10-99), train/test splits (`randomize_data`, :190-260), the prediction
driver (`predictBNN`, BNN_lib.py:404-501, whose forward passes run on the device through `get_posterior_cat_prob`),
accuracy / confusion / threshold summaries of an [N, K] probability table (BNN_lib.py:195-233, 309-348, 627-679), the
alternative proposal and Gibbs helpers (BNN_mcmc.py:27-150) and the count-data likelihoods (BNN_lik.py).  Semantics,
argument names, printed messages, file names and the order of random draws follow the reference so that a seeded
script produces the same splits and files; the code itself is written for this package.

The elementwise helpers of the reference (`relu_f`, `swish_f`, `SoftMax`, `SoftPlus` ...) double as the selector tokens
user code passes around (`output_act_fun=bn.SoftMax`).  Inside MCMC / prediction they select device code; called
directly on a host array (post-processing of a prediction table) they evaluate the reference's formula with numpy.
The contractions of the path (`MatrixMultiplicationD`, `RunHiddenLayer`) always run on the device.
"""
import copy
import csv
import glob
import os
import pickle
import random
import sys
from copy import deepcopy  # noqa: F401  (re-exported: the reference's star-imports expose it)

import numpy as np

small_number = 1e-10


# ------------------------------------------------------------------------------------------------------
# elementwise forms (BNN_lib.py:50-66, 166-182) -- selector tokens on the device path, numpy on host tables
# ------------------------------------------------------------------------------------------------------
def relu_f(z, _=0):
    z[z < 0] = 0
    return z


def leaky_relu_f(z, prm):
    z[z < 0] = z[z < 0] * prm
    return z


def swish_f(z, _=0):
    return z * (1.0 + np.exp(-z)) ** (-1)


def tanh_f(z, _=0):
    return 1.0 - 2.0 / (np.exp(2.0 * z) + 1.0)


def SoftMax(z):
    e = np.exp(z - np.max(z, axis=1, keepdims=True))
    return e / np.sum(e, axis=1, keepdims=True)


def SoftPlus(z):
    return np.logaddexp(0, z)


def RegressTransform(z):
    return z


def RegressTransformError(z, ind=None):
    if ind is None:
        ind = int(z.shape[1] / 2)
    z[:, ind:] = SoftPlus(z[:, ind:])
    return z


def _log_norm_pdf(x, mu, sd):
    r = (x - mu) / sd
    return -0.5 * r * r - np.log(sd) - 0.5 * np.log(2.0 * np.pi)


def calc_likelihood(prediction, labels, sample_id, class_weight=[], instance_weight=None, lik_temp=1, sig2=0):
    """BNN_lib.py:100-121 on a host prediction table (the sampler evaluates it inside the forward kernels)."""
    lp = np.log(prediction[sample_id, labels])
    if len(class_weight):
        lp = lp * class_weight[labels]
    if instance_weight is not None:
        lp = lp * instance_weight
    return lik_temp * np.sum(lp)


def calc_likelihood_regression(prediction, true_values, _, class_weight=[], instance_weight=None, lik_temp=1, sig2=1):
    if instance_weight is not None:
        sys.exit("Instance weights not available for regression")
    return lik_temp * np.sum(_log_norm_pdf(true_values, prediction, sig2))


def calc_likelihood_regression_error(prediction, true_values, _, class_weight=[], instance_weight=None, lik_temp=1, sig2=1):
    if instance_weight is not None:
        sys.exit("Instance weights not available for regression")
    ind = int(prediction.shape[1] / 2)
    return lik_temp * np.sum(_log_norm_pdf(true_values, prediction[:, :ind], prediction[:, ind:]))


# ------------------------------------------------------------------------------------------------------
# single contractions through the device (BNN_lib.py:145-193)
# ------------------------------------------------------------------------------------------------------
def _one_layer_on_device(x, w, act, alpha):
    """act(x @ w.T (+ bias column 0)) as a two-layer network [w, I] with identity output on the prediction kernels:
    the second layer multiplies by 1.0 and adds zeros, which is exact."""
    from .engine import Engine, NetShape
    from . import _lib as L
    x = np.ascontiguousarray(x, dtype=np.float64)
    w = np.ascontiguousarray(w, dtype=np.float64)
    eye = np.eye(w.shape[0])
    eng = Engine(NetShape.from_weights([w, eye], x.shape[1], act=act, lik=L.LIK_GAUSSIAN))
    try:
        al = None if alpha is None else np.array([[alpha, 0.0]])
        return eng.predict(x, [[w, eye]], alphas=al, mean=False, dense=True)["dense"][0]
    finally:
        eng.close()


def MatrixMultiplicationD(x1, x2):
    """x1 @ x2.T, or x1 @ x2.T[1:] + x2.T[0] when x2 has one more column than x1 (bias = column 0)."""
    return _one_layer_on_device(x1, x2, "genReLU", 1.0)      # slope-1 leaky ReLU = no activation


MatrixMultiplication = MatrixMultiplicationD


def RunHiddenLayer(z0, w01, actFun, layer_n, data_transform=None):
    if data_transform is not None:
        z0 = data_transform.transform(z0)
    if not actFun:
        return MatrixMultiplicationD(z0, w01)
    fun = actFun._function
    alpha = None
    if fun == "genReLU":
        alpha = float(np.atleast_1d(actFun._prm)[layer_n])
    return _one_layer_on_device(z0, w01, fun, alpha)


# ------------------------------------------------------------------------------------------------------
# summaries of prediction tables (BNN_lib.py:195-233, 309-348)
# ------------------------------------------------------------------------------------------------------
def CalcAccuracyRegression(y, lab):
    return np.mean((y[:, 0:lab.shape[1]] - lab) ** 2)


def CalcLabelAccuracyRegression(y, lab):
    return np.mean((y[:, 0:lab.shape[1]] - lab) ** 2, axis=0)


def CalcAccuracy(y, lab):
    """Argmax-equals-label rate of an [N, K] table; one rate per posterior sample for an [S, N, K] tensor."""
    y = np.asarray(y)
    if y.ndim == 3:
        return np.array([np.sum(i == lab) / len(i) for i in np.argmax(y, axis=2)])
    prediction = np.argmax(y, axis=1)
    return np.sum(prediction == lab) / len(prediction)


def CalcLabelAccuracy(y, lab):
    pred = np.argmax(y, axis=1)
    lab = np.asarray(lab)
    return np.array([np.sum(pred[lab == c] == c) / np.sum(lab == c) for c in np.unique(lab)])


def CalcLabelFreq(y):
    pred = np.argmax(y, axis=1)
    return np.bincount(pred, minlength=y.shape[1]) / len(pred)


def CalcConfusionMatrix(y, lab):
    """Rows = true class, columns = predicted class over the classes present in `lab`, with 'All' margins
    (pd.crosstab(..., margins=True, dropna=False), BNN_lib.py:220-225).  Predictions of a class absent from `lab` have
    no column (pd.Categorical turns them into missing values) but still count in the row totals and the grand total."""
    import pandas as pd
    lab = np.asarray(lab)
    cats = np.unique(lab)
    pred = np.argmax(y, axis=1)
    k = len(cats)
    m = np.zeros((k + 1, k + 1), dtype=int)
    for a, ca in enumerate(cats):
        for b, cb in enumerate(cats):
            m[a, b] = np.sum((lab == ca) & (pred == cb))
    m[:k, k] = [np.sum(lab == ca) for ca in cats]
    m[k, :k] = m[:k, :k].sum(axis=0)
    m[k, k] = len(lab)
    names = list(cats) + ["All"]
    return pd.DataFrame(m, index=pd.Index(names, name="True"), columns=pd.Index(names, name="Predicted"))


def SkipAccuracy(_, __):
    return 1.0


def SkipAccuracyVec(_, __):
    return np.ones(1)


def _supported(y, threshold):
    pred = np.argmax(y, axis=1)
    return pred, (y[np.arange(len(pred)), pred] > threshold)


def CalcTP(y, lab, threshold=0.95):
    pred, strong = _supported(y, threshold)
    return np.sum(strong[pred == lab]) / len(pred)


def CalcFP(y, lab, threshold=0.95):
    pred, strong = _supported(y, threshold)
    return np.sum(strong[pred != lab]) / len(pred)


def _bayes_factor(y, y_p):
    pred = np.argmax(y, axis=1)
    rows = np.arange(len(pred))
    post, prior = y[rows, pred], y_p[rows, pred]
    return pred, (post / (small_number + 1 - post)) / (prior / (small_number + 1 - prior))


def CalcTP_BF(y, y_p, lab, threshold=150):
    pred, bf = _bayes_factor(y, y_p)
    return np.sum((bf > threshold)[pred == lab]) / len(pred)


def CalcFP_BF(y, y_p, lab, threshold=150):
    pred, bf = _bayes_factor(y, y_p)
    return np.sum((bf > threshold)[pred != lab]) / len(pred)


def CalcAccAboveThreshold(y, lab, threshold=0.95):
    keep = np.where(np.max(y, axis=1) > threshold)
    pred = np.argmax(y, axis=1)[keep]
    print(np.sum(pred == np.asarray(lab)[keep]) / len(pred))


def RecurMeanVar(it, list_mu_var_old, list_curr_param, indx):
    """Running mean / variance of the entries touched by a proposal (BNN_lib.py:274-284)."""
    ix, iy = indx
    mu_old, var_old = list_mu_var_old
    mu, var = mu_old + 0, var_old + 0
    cur = list_curr_param[ix, iy]
    it = it + 1
    mu[ix, iy] = (it - 1) / it * mu_old[ix, iy] + 1 / it * cur
    var[ix, iy] = (it - 1) / it * var_old[ix, iy] + 1 / (it - 1) * (cur - mu[ix, iy]) ** 2
    return [mu, var]


def calcHPD(data, level):
    """Shortest interval holding `level` of the sample."""
    assert 0 < level < 1
    d = np.sort(np.asarray(list(data)))
    n_in = int(round(level * len(d)))
    if n_in < 2:
        sys.exit("\n\nToo little data to calculate marginal parameters.")
    widths = d[n_in - 1:] - d[:len(d) - n_in + 1]
    i = int(np.argmin(widths))
    return (d[i], d[i + n_in - 1])


# ------------------------------------------------------------------------------------------------------
# threshold utilities (BNN_lib.py:627-679)
# ------------------------------------------------------------------------------------------------------
def get_accuracy_threshold(probs, labels, threshold=0.75):
    keep = np.where(np.max(probs, axis=1) > threshold)[0]
    sup, lab = probs[keep, :], np.asarray(labels)[keep]
    pred = np.argmax(sup, axis=1)
    return {"predictions": pred, "accuracy": len(pred[pred == lab]) / len(pred),
            "retained_samples": len(pred) / len(labels), "confusion_matrix": CalcConfusionMatrix(sup, lab)}


def get_posterior_threshold(pkl_file, target_acc=0.9, post_summary_mode=1, output_file=None):
    """Smallest posterior-probability cut-off (0.01 ... 0.99) at which the test accuracy reaches target_acc.  Collective
    under a process group of several ranks (predictBNN); only rank 0 writes output_file."""
    from . import api
    bnn_obj, mcmc_obj, logger_obj = load_obj(pkl_file)
    res = predictBNN(bnn_obj._test_data, pickle_file=pkl_file, test_labels=bnn_obj._test_labels,
                     post_summary_mode=post_summary_mode, verbose=0)["post_prob_predictions"]
    rows = []
    for thr in np.linspace(0.01, 0.99, 99):
        try:
            sc = get_accuracy_threshold(res, bnn_obj._test_labels, threshold=thr)
            rows.append([thr, sc["accuracy"], sc["retained_samples"]])
        except Exception:           # no instance above the cut-off
            pass
    tbl = np.array(rows)
    if output_file is not None and api._is_rank0():
        import pandas as pd
        np.round(pd.DataFrame(tbl, columns=["Threshold", "Accuracy", "Retained_data"]), 3).to_csv(
            path_or_buf=output_file, sep="\t", index=False, header=True)
    try:
        i = np.min(np.where(np.round(tbl[:, 1], 2) >= target_acc))
    except ValueError:
        sys.exit("Target accuracy can not be reached. Please set threshold lower or try different post_summary_mode.")
    sel = tbl[i, :]
    print("Selected threshold: PP =", np.round(sel[0], 3), "yielding test accuracy ~ %s" % (target_acc))
    print("Retained instances above threshold:", np.round(sel[2], 3))
    return sel


def turn_low_pp_instances_to_nan(pred, high_pp_indices):
    out = np.full(pred.shape, np.nan)
    out[high_pp_indices] = pred[high_pp_indices]
    return out


# ------------------------------------------------------------------------------------------------------
# prediction driver (BNN_lib.py:404-501)
# ------------------------------------------------------------------------------------------------------
def predictBNN(predict_features, pickle_file, test_labels=[], instance_id=[], pickle_file_prior=0, target_acc=None,
               post_cutoff=None, threshold=0.95, bf=150, post_summary_mode=0, fname="", wd="", verbose=1):
    """Posterior prediction for `predict_features` from the samples stored in `pickle_file`; all posterior samples are
    scored in one device pass (api.get_posterior_cat_prob).  Writes <fname_><pkl>_pred_pr.npy, _pred_mean_pr.txt and
    (with labels) _accuracy.txt next to the pickle (or into `wd`).  Under a process group of several ranks the call is
    collective (every rank passes the same arguments and gets the same result) and only rank 0 writes the files."""
    from . import api
    bnn_obj, mcmc_obj, logger_obj = load_obj(pickle_file)
    post_samples = logger_obj._post_weight_samples
    actFun, output_act_fun = bnn_obj._act_fun, bnn_obj._output_act_fun
    out_name = os.path.basename(os.path.splitext(pickle_file)[0])
    outdir = wd if wd != "" else os.path.dirname(pickle_file)
    dense, post_prob = api.get_posterior_cat_prob(predict_features, post_samples, post_summary_mode=post_summary_mode,
                                                  actFun=actFun, output_act_fun=output_act_fun)
    if fname != "":
        fname = fname + "_"
    f_dense = os.path.join(outdir, fname + out_name + "_pred_pr.npy")
    f_mean = os.path.join(outdir, fname + out_name + "_pred_mean_pr.txt")
    writer = api._is_rank0()
    if len(test_labels) > 0:
        accuracy = CalcAccuracy(post_prob, test_labels)
        tp = CalcTP(post_prob, test_labels, threshold=threshold)
        fp = CalcFP(post_prob, test_labels, threshold=threshold)
        mean_accuracy = np.mean(accuracy)
        cm = CalcConfusionMatrix(post_prob, test_labels)
        cm_out = cm.values.astype(int)
        if verbose:
            print("Accuracy:", mean_accuracy)
            print("True positive rate:", np.mean(tp))
            print("False positive rate:", np.mean(fp))
            print("Confusion matrix:\n", cm)
        if writer:
            with open(os.path.join(outdir, fname + out_name + "_accuracy.txt"), "w") as outf:
                outf.writelines("Mean accuracy: %s (TP: %s; FP: %s)" % (mean_accuracy, tp, fp))
    else:
        mean_accuracy, cm_out = np.nan, np.nan
    if pickle_file_prior:
        prior_samples = load_obj(pickle_file_prior)
        _, prior_prob = api.get_posterior_cat_prob(predict_features, prior_samples, post_summary_mode=1, actFun=actFun,
                                                   output_act_fun=output_act_fun, return_dense=False)
        tp = CalcTP_BF(post_prob, prior_prob, test_labels, threshold=bf)
        fp = CalcFP_BF(post_prob, prior_prob, test_labels, threshold=bf)
        if verbose:
            print("True positive rate (BF):", np.mean(tp))
            print("False positive rate (BF):", np.mean(fp))
    if target_acc or post_cutoff:
        cut = get_posterior_threshold(pickle_file, target_acc, post_summary_mode) if target_acc else post_cutoff
        keep = np.where(np.max(post_prob, axis=1) > cut)[0]
        post_prob = turn_low_pp_instances_to_nan(post_prob, keep)
        dense = np.array([turn_low_pp_instances_to_nan(i, keep) for i in dense])
    if not writer:
        return {"post_prob_predictions": post_prob, "mean_accuracy": mean_accuracy, "confusion_matrix": cm_out}
    if len(instance_id):
        instance_id = np.asarray(instance_id)
        tbl = np.hstack((instance_id.reshape(len(instance_id), 1), np.round(post_prob, 4).astype(str)))
        np.savetxt(f_mean, tbl, fmt="%s", delimiter="\t")
    else:
        np.savetxt(f_mean, post_prob, fmt="%.3f")
    np.save(f_dense, dense)
    if verbose:
        print("Predictions saved in files:")
        print("   ", f_dense)
        print("   ", f_mean, "\n")
    return {"post_prob_predictions": post_prob, "mean_accuracy": mean_accuracy, "confusion_matrix": cm_out}


def get_weights_from_tensorflow_model(model_dir):
    try:
        import tensorflow as tf
    except Exception:
        sys.exit("The required Tensorflow library not found.")
    model = tf.keras.models.load_model(model_dir)
    nodes, weights, biases = [], [], []
    for layer in model.layers:
        nodes.append(np.array(layer.weights[0].shape)[1])
        weights.append(layer.weights[0].numpy().T)
        if len(layer.weights) == 2:
            biases.append(layer.weights[1].numpy())
    return [nodes[:-1], weights, biases]


# ------------------------------------------------------------------------------------------------------
# data files (BNN_files.py)
# ------------------------------------------------------------------------------------------------------
def load_obj(file_name):
    with open(file_name, "rb") as f:
        return pickle.load(f)


def turn_labels_to_numeric(labels, label_file, save_to_file=False):
    """Class names -> 0..K-1 in the sorted order of np.unique."""
    labels = np.asarray(labels)
    numeric = np.zeros(len(labels)).astype(int)
    for c, name in enumerate(np.unique(labels)):
        numeric[(labels == name).flatten()] = c
    if save_to_file:
        np.savetxt(label_file.replace(".txt", "_numerical.txt"), numeric, fmt="%i")
    return numeric


def randomize_data(tot_x, tot_labels, testsize=0.1, all_class_in_testset=1, inst_id=[], randomize=True, cv=-1, rs=None):
    """Train / test split (BNN_files.py:190-260).  Draw order on `rs`: one permutation (only when randomize and
    testsize), then -- with all_class_in_testset -- one rs.choice (with replacement) per class."""
    n = len(tot_labels)
    if randomize and testsize:
        order = rs.choice(range(n), n, replace=False)
    else:
        order = np.arange(n)
    if not randomize:
        all_class_in_testset = 0
    tot_x, tot_labels = tot_x[order], tot_labels[order]
    ids = inst_id[order] if len(inst_id) else []
    n_test = int(testsize * n)
    id_train, id_test = [], []
    if cv > -1 and testsize:
        a = n_test * cv
        test_idx = range(a, int(np.min([a + n_test, n])))
        x_test, lab_test = tot_x[test_idx, :], tot_labels[test_idx]
        x, lab = np.delete(tot_x, test_idx, axis=0), np.delete(tot_labels, test_idx, axis=0)
        if len(inst_id):
            id_test, id_train = ids[test_idx], np.delete(ids, test_idx)
        print("test set:", test_idx)
    elif all_class_in_testset and testsize:
        picked = []
        for c in np.unique(tot_labels):
            members = np.where(tot_labels == c)[0]
            picked += list(rs.choice(members, np.max([1, int(testsize * len(members))])))
        test_idx = np.array(picked)
        keep = np.ones(tot_labels.size, dtype=bool)
        keep[test_idx] = False
        train_idx = np.flatnonzero(keep)
        x_test, lab_test = tot_x[test_idx], tot_labels[test_idx]
        x, lab = tot_x[train_idx], tot_labels[train_idx]
        if len(inst_id):
            id_train, id_test = ids[train_idx], ids[test_idx]
    elif n_test == 0:
        x_test, lab_test, x, lab = [], [], tot_x, tot_labels
        if len(inst_id):
            id_train, id_test = ids, []
    else:
        x_test, lab_test = tot_x[-n_test:, :], tot_labels[-n_test:]
        x, lab = tot_x[:-n_test, :], tot_labels[:-n_test]
        if len(inst_id):
            id_test, id_train = ids[-n_test:], ids[:-n_test]
    return x, lab, x_test, lab_test, id_train, id_test


def get_data(f, l=None, testsize=0.1, batch_training=0, seed=1234, all_class_in_testset=1, instance_id=0, header=0,
             feature_indx=None, randomize_order=True, from_file=True, label_mode="classification", cv=-1):
    """Feature / label tables -> the data dictionary npBNN takes (BNN_files.py:10-99): keys data, labels, label_dict,
    test_data, test_labels, id_data, id_test_data, file_name, feature_names."""
    import pandas as pd
    rs = np.random.default_rng(seed)
    ids = []
    print("instance_id", instance_id)
    if from_file:
        fname = os.path.splitext(os.path.basename(f))[0]
        try:
            tot_x = np.load(f, allow_pickle=True)
        except Exception:
            if not instance_id:
                tot_x = np.loadtxt(f, skiprows=int(header))
            else:
                raw = np.genfromtxt(f, skip_header=header, dtype=str)
                tot_x, ids = raw[:, 1:].astype(float), raw[:, 0].astype(str)
        if header:
            with open(f) as fh:
                feature_names = np.array(next(fh).split()[1:])
        else:
            feature_names = np.array(["feature_%s" % i for i in range(tot_x.shape[1])])
    else:
        f = pd.DataFrame(f)
        fname = "bnn"
        if not instance_id:
            feature_names, tot_x = np.array(f.columns), f.values
        else:
            feature_names, tot_x, ids = np.array(f.columns[1:]), f.values[:, 1:], f.values[:, 0].astype(str)
    if feature_indx is not None:
        feature_indx = np.array(feature_indx)
        tot_x, feature_names = tot_x[:, feature_indx], feature_names[feature_indx]
    if l is None:
        return {"data": np.array(tot_x).astype(float), "labels": [], "label_dict": [], "test_data": [], "test_labels": [],
                "id_data": ids, "id_test_data": [], "file_name": fname, "feature_names": feature_names}
    try:
        l = pd.DataFrame(l)                       # labels handed over as a table; a path raises and is read below
        if instance_id:
            tot_labels = l.values[:, 1:]
        elif label_mode == "classification":
            tot_labels = l.values.astype(str).flatten()
        else:
            tot_labels = l.values
    except Exception:
        tot_labels = np.loadtxt(l, skiprows=int(header), dtype=str)
        if instance_id:
            tot_labels = tot_labels[:, 1:]
    if label_mode == "classification":
        numeric = turn_labels_to_numeric(tot_labels, l)
    else:
        numeric = tot_labels.reshape((tot_labels.shape[0], 1)) if len(tot_labels.shape) == 1 else tot_labels
    print("tot_labels_numeric", numeric.shape)
    x, labels, x_test, labels_test, id_x, id_test = randomize_data(
        tot_x, numeric, testsize=testsize, all_class_in_testset=all_class_in_testset, inst_id=ids,
        randomize=randomize_order, cv=cv, rs=rs)
    if batch_training:
        pick = rs.integers(0, len(labels), batch_training)
        x, labels = x[pick], labels[pick]
    if label_mode == "regression":
        labels = labels.astype(float)
        if testsize:
            labels_test = labels_test.astype(float)
    return {"data": np.array(x).astype(float), "labels": labels, "label_dict": np.unique(tot_labels),
            "test_data": np.array(x_test).astype(float), "test_labels": labels_test, "id_data": id_x,
            "id_test_data": id_test, "file_name": fname, "feature_names": feature_names}


def save_data(dat, lab, outname="data", test_dat=[], test_lab=[]):
    test_lab = np.array(test_lab)
    np.savetxt(outname + "_features.txt", dat, delimiter="\t")
    np.savetxt(outname + "_labeles.txt", lab.astype(int), delimiter="\t")       # file names as the reference writes them
    if len(test_dat) > 0:
        np.savetxt(outname + "_test_features.txt", test_dat, delimiter="\t")
        np.savetxt(outname + "_test_labeles.txt", test_lab.astype(int), delimiter="\t")


def log_header(bnn_obj, add_prms=None):
    """Column names of the .log file (BNN_files.py:136-174)."""
    head = ["it", "posterior", "likelihood", "prior"]
    if bnn_obj._estimation_mode == "classification":
        head += ["accuracy", "test_accuracy"] + ["acc_C%s" % i for i in range(bnn_obj._n_output_prm)]
    elif bnn_obj._estimation_mode == "custom":
        head += ["MSE", "test_MSE"]
    else:
        head += ["MSE", "test_MSE"] + ["MSE_prm%s" % i for i in range(bnn_obj._n_output_prm)]
    for i in range(bnn_obj._n_layers):
        head += ["mean_w%s" % i, "std_w%s" % i]
        if bnn_obj._hyper_p:
            head.append(("prior_std_w%s" if bnn_obj._hyper_p == 1 else "mean_prior_std_w%s") % i)
    if bnn_obj._freq_indicator:
        head.append("mean_ind")
    if add_prms:
        head += add_prms
    if bnn_obj._act_fun._trainable:
        head += ["alpha_%s" % i for i in range(bnn_obj._n_layers - 1)]
    if len(bnn_obj._error_prm):
        head += ["sig_%s" % i for i in range(len(bnn_obj._error_prm))]
    if bnn_obj._feature_indicators is not None:
        head += ["feature_ind_%s" % i for i in range(bnn_obj._n_features)]
    return head + ["acc_prob", "mcmc_id"]


def init_output_files(bnn_obj, filename="bnn", sample_from_prior=0, outpath="", add_prms=None, continue_logfile=False,
                      log_all_weights=0):
    """Creates <filename>_l<nodes>.log (+ _W.log) with their header rows; returns (log, weight log or None, pkl)."""
    outdir = os.path.dirname(filename)
    if len(outdir) > 0 and not os.path.exists(outdir):
        os.makedirs(outdir)
    stem = "%s_l%s" % (filename, "_".join(map(str, bnn_obj._n_nodes)))
    logfile = os.path.join(outpath, stem + ".log")
    w_file = os.path.join(outpath, stem + "_W.log") if log_all_weights else None
    if not continue_logfile:
        with open(logfile, "w", newline="") as fh:
            csv.writer(fh, delimiter="\t").writerow(log_header(bnn_obj, add_prms))
    if log_all_weights:
        with open(w_file, "w", newline="") as fh:
            csv.writer(fh, delimiter="\t").writerow(
                ["it"] + ["w_%s_%s" % (i, j) for i in range(bnn_obj._n_layers) for j in range(bnn_obj._w_layers[i].size)])
    return logfile, w_file, os.path.join(outpath, stem + ".pkl")


def merge_dict(d1, d2):
    from collections import defaultdict
    d = defaultdict(list)
    for a, b in list(d1.items()) + list(d2.items()):
        d[a].append(b)
    return d


def combine_pkls(files=None, dir=None, tag=""):
    """Writes combine_pkl<tag>.pkl holding the [bnn, mcmc, logger] of the first file (BNN_files.py:277-300; like the
    reference, the posterior samples of the other files are read but not merged)."""
    if dir is not None:
        files = glob.glob(os.path.join(dir, "*%s*.pkl" % tag))
        print("Combining %s files: \n" % len(files), files)
    out_file = os.path.join(os.path.dirname(files[0]), "combine_pkl%s.pkl" % tag)
    first = None
    for f in files:
        if f == out_file:
            continue
        objs = load_obj(f)
        if first is None:
            first = objs
    with open(out_file, "wb") as output:
        pickle.dump(list(first[:3]), output, pickle.HIGHEST_PROTOCOL)
    return out_file


def assign_indx(l):
    """Rank of first appearance: ['b','a','b'] -> [0, 1, 0]."""
    seen, out = {}, []
    for v in l:
        if v not in seen:
            seen[v] = len(seen)
        out.append(seen[v])
    return np.array(out)


def unique_unsorted(a_tmp):
    a = copy.deepcopy(a_tmp)
    return a_tmp[np.sort(np.unique(a, return_index=True)[1])]


# ------------------------------------------------------------------------------------------------------
# proposal / Gibbs helpers other than UpdateNormal (BNN_mcmc.py:27-150).  MCMC(update_function=...) accepts only
# UpdateNormal on the device; these serve user code that calls them directly on host matrices.
# ------------------------------------------------------------------------------------------------------
def _default_rs(rs):
    return rs if rs else np.random.default_rng(random.randint(1000, 9999))


def _reflect(z, Mb, mb):
    z[z > Mb] = Mb - (z[z > Mb] - Mb)
    z[z < mb] = mb + (mb - z[z < mb])
    return z


def UpdateNormal(i, d=0.01, n=1, Mb=100, mb=-100, rs=0):
    """The sampler's proposal (BNN_mcmc.py:57-69).  Inside MCMC it is the selector of the device kernel k_mh_update;
    called directly it perturbs a host matrix (duplicate indices: last increment wins, single reflection)."""
    i, rs = np.array(i), _default_rs(rs)
    ix, iy = rs.integers(0, i.shape[0], n), rs.integers(0, i.shape[1], n)
    z = np.zeros(i.shape) + i
    z[ix, iy] = z[ix, iy] + rs.normal(0, d[ix, iy], n)
    return _reflect(z, Mb, mb), (ix, iy), 0


def UpdateFixedNormal(i, d=1, n=1, Mb=100, mb=-100, rs=0):
    rs = _default_rs(rs)
    ix, iy = rs.integers(0, i.shape[0], n), rs.integers(0, i.shape[1], n)
    cur, new = i[ix, iy], rs.normal(0, d[ix, iy], n)
    hastings = np.sum(_log_norm_pdf(cur, 0, d[ix, iy]) - _log_norm_pdf(new, 0, d[ix, iy]))
    z = np.zeros(i.shape) + i
    z[ix, iy] = new
    return _reflect(z, Mb, mb), (ix, iy), hastings


def UpdateNormal1D(i, d=0.01, n=1, Mb=100, mb=-100, rs=0):
    i, rs = np.array(i), _default_rs(rs)
    ix = rs.integers(0, len(i), n)
    z = np.zeros(i.shape) + i
    z[ix] = z[ix] + rs.normal(0, d, n)
    return _reflect(z, Mb, mb), ix, 0


def UpdateNormalNormalized(i, d=0.01, n=1, Mb=100, mb=-100, rs=0):
    i, rs = np.array(i), _default_rs(rs)
    ix, iy = rs.integers(0, i.shape[0], n), rs.integers(0, i.shape[1], n)
    z = np.zeros(i.shape) + i
    z[ix, iy] = z[ix, iy] + rs.normal(0, d[ix, iy], n)
    return z / np.sum(z), (ix, iy), 0


def UpdateUniform(i, d=0.1, n=1, Mb=100, mb=-100):
    i = np.array(i)
    ix, iy = np.random.randint(0, i.shape[0], n), np.random.randint(0, i.shape[1], n)
    z = np.zeros(i.shape) + i
    z[ix, iy] = z[ix, iy] + np.random.uniform(-d[ix, iy], d[ix, iy], n)
    return _reflect(z, Mb, mb), (ix, iy), 0


def UpdateBinomial(ind, update_f, shape_out):
    return np.abs(ind - np.random.binomial(1, np.random.random() * update_f, shape_out))


def multiplier_proposal_vector(q, d=1.05, f=1, rs=0):
    rs = _default_rs(rs)
    ff = rs.binomial(1, f, q.shape)
    m = np.exp(2 * np.log(d) * (rs.random(q.shape) - .5))
    m[ff == 0] = 1.
    return q * m, 0, np.sum(np.log(m))


def multiplier_proposal(i, d=1.05):
    m = np.exp(2 * np.log(d) * (np.random.random() - .5))
    return (i + 0) * m, 0, np.log(m)


def GibbsSampleNormStdGammaVector(x, a=2, b=0.1, mu=0):
    tau = np.random.gamma(a + len(x) / 2., scale=1. / (b + np.sum((x - mu) ** 2) / 2.))
    return 1 / np.sqrt(tau)


def GibbsSampleNormStdGamma2D(x, a=1, b=0.1, mu=0):
    tau = np.random.gamma(a + x.shape[0] / 2., scale=1. / (b + np.sum((x - mu) ** 2, axis=0) / 2.))
    return 1 / np.sqrt(tau)


def GibbsSampleNormStdGammaONE(x, a=1.5, b=0.1, mu=0):
    tau = np.random.gamma(a + 1 / 2., scale=1. / (b + ((x - mu) ** 2) / 2.))
    return 1 / np.sqrt(tau)


def GibbsSampleGammaRateExp(sd, a, alpha_0=1., beta_0=1.):
    tau = 1. / (sd ** 2)
    return np.random.gamma(alpha_0 + len(tau) * a, scale=1. / (beta_0 + np.sum(tau)))


# ------------------------------------------------------------------------------------------------------
# count-data likelihoods of BNN_lik.py: host functions for estimation_mode="custom" users.  Inside MCMC / MC3
# (likelihood_f=, accuracy_f=) the four count likelihoods and their accuracy functions are identity tokens that select
# the device epilogue (BNN_LIK_POISSON / NEGBIN / NEGBIN10); gamma_likelihood is not on the device path
# ------------------------------------------------------------------------------------------------------
def _nbinom_logpmf(k, n, p):
    from scipy.special import gammaln, xlog1py, xlogy
    return gammaln(k + n) - gammaln(k + 1) - gammaln(n) + xlogy(n, p) + xlog1py(k, -p)


def poi_likelihood(prediction, true_values, sample_id=None, class_weight=None, instance_weight=None, lik_temp=1, sig2=0):
    from scipy.special import gammaln, xlogy
    rate, k = np.exp(prediction[:, 0]), true_values[:, 0]
    return np.sum(xlogy(k, rate) - gammaln(k + 1) - rate)


def negbin_likelihood(prediction, true_values, sample_id=None, class_weight=None, instance_weight=None, lik_temp=1, sig2=0):
    mean, p = np.exp(prediction[:, 0]), 1 / (1 + np.exp(-prediction[:, 1]))
    return np.sum(_nbinom_logpmf(true_values[:, 0], p * mean / (1 - p), p))


def negbin_likelihood2d(prediction, true_values, sample_id=None, class_weight=None, instance_weight=None, lik_temp=1, sig2=0):
    o = true_values.shape[1]
    mean, p = np.exp(prediction[:, :o]), 1 / (1 + np.exp(-prediction[:, o:]))
    return np.sum(_nbinom_logpmf(true_values, p * mean / (1 - p), p))


def negbin_likelihood_base10(prediction, true_values, sample_id=None, class_weight=None, instance_weight=None, lik_temp=1,
                             sig2=0):
    mean, p = 10 ** (prediction[:, 0]), 1 / (1 + 10 ** (-prediction[:, 1]))
    return np.sum(_nbinom_logpmf(true_values[:, 0], p * mean / (1 - p), p))


def gamma_likelihood(prediction, true_values, sample_id=None, class_weight=None, instance_weight=None, lik_temp=1, sig2=0):
    import scipy.stats
    # scipy's positional (a, loc): the reference passes exp(prediction[:, 1]) as the LOCATION (BNN_lik.py:83)
    return np.sum(scipy.stats.gamma.logpdf(true_values, np.exp(prediction[:, 0]), np.exp(prediction[:, 1])))


def negbin_acc(y, lab):
    return np.mean((np.exp(y[:, 0]) - lab[:, 0]) ** 2)


def negbin_acc_base10(y, lab):
    return np.mean((10 ** (y[:, 0]) - lab[:, 0]) ** 2)


def negbin2d_acc(y, lab):
    return np.mean((np.exp(y[:, :lab.shape[1]]) - lab[:, :lab.shape[1]]) ** 2)


def poi_acc(y, lab):
    return np.mean((np.exp(y[:, 0]) - lab[:, 0]) ** 2)


def gamma_acc(y, lab):
    acc = np.mean((np.exp(y[:, 0]) - lab.flatten()) ** 2)     # the reference computes and drops it (returns None)


def get_feature_summary(data, focal_features):
    """[3, n_focal]: integer-like flag (binary / ordinal), min, max of each focal feature (BNN_pdp.py:14-28)."""
    out = np.zeros((3, len(focal_features)))
    for i, f in enumerate(focal_features):
        values = np.unique(data[:, f])
        out[1, i], out[2, i] = np.nanmin(values), np.nanmax(values)
        out[0, i] = np.all(np.isin(values, np.arange(out[1, i], out[2, i] + 1)))
    return out
