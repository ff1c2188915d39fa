"""Argument validators used by the drop-in gaussianmixture / hiddenmarkovnormal API.

Only the validators on the LearnModel paths are provided; each has the contract of the
reference function of the same name in bayesml/_check.py (cited per function): return the (possibly
float-cast) value or raise `exception_class(<name> + message)`.
"""
import numpy as np


def _is_int(v):
    return np.issubdtype(type(v), np.integer)


def _is_float(v):
    return np.issubdtype(type(v), np.floating)


def _is_array_of(v, kind):
    return type(v) is np.ndarray and np.issubdtype(v.dtype, kind)


def pos_int(val, val_name, exception_class):
    """Positive integer scalar (reference _check.py:28-32)."""
    if _is_int(val) and val > 0:
        return val
    raise exception_class(val_name + " must be int. Its value must be positive (not including 0).")


def pos_floats(val, val_name, exception_class):
    """Positive scalar, or ndarray of positive numbers; integers are cast to float (reference _check.py:175-185)."""
    if _is_float(val) and val > 0.0:
        return val
    if _is_int(val) and val > 0:
        return float(val)
    if _is_array_of(val, np.integer) and np.all(val > 0):
        return val.astype(float)
    if _is_array_of(val, np.floating) and np.all(val > 0.0):
        return val
    raise exception_class(val_name + " must be float or a numpy.ndarray. Its values must be positive (not including 0)")


def float_vec(val, val_name, exception_class):
    """1-dimensional numeric ndarray (reference _check.py:187-193)."""
    if type(val) is np.ndarray and val.ndim == 1:
        if np.issubdtype(val.dtype, np.integer):
            return val.astype(float)
        if np.issubdtype(val.dtype, np.floating):
            return val
    raise exception_class(val_name + " must be a 1-dimensional numpy.ndarray.")


def float_vec_sum_1(val, val_name, exception_class):
    """1-dimensional numeric ndarray whose elements sum to 1 within sqrt(eps) (reference _check.py:219-225)."""
    if type(val) is np.ndarray and val.ndim == 1 and abs(val.sum() - 1.0) <= np.sqrt(np.finfo(np.float64).eps):
        if np.issubdtype(val.dtype, np.integer):
            return val.astype(float)
        if np.issubdtype(val.dtype, np.floating):
            return val
    raise exception_class(val_name + " must be a 1-dimensional numpy.ndarray, and the sum of its elements must equal to 1.")


def float_vecs_sum_1(val, val_name, exception_class):
    """Numeric ndarray with ndim >= 1 whose sums along the last axis are each 1 within sqrt(eps) (the stacked form of
    float_vec_sum_1)."""
    if type(val) is np.ndarray and val.ndim >= 1 and np.all(np.abs(val.sum(axis=-1) - 1.0) <= np.sqrt(np.finfo(np.float64).eps)):
        if np.issubdtype(val.dtype, np.integer):
            return val.astype(float)
        if np.issubdtype(val.dtype, np.floating):
            return val
    raise exception_class(val_name + " must be a numpy.ndarray whose ndim >= 1, and the sum along the last dimension must equal to 1.")


def float_vecs(val, val_name, exception_class):
    """Numeric ndarray with ndim >= 1 (reference _check.py:203-209)."""
    if type(val) is np.ndarray and val.ndim >= 1:
        if np.issubdtype(val.dtype, np.integer):
            return val.astype(float)
        if np.issubdtype(val.dtype, np.floating):
            return val
    raise exception_class(val_name + " must be a numpy.ndarray whose ndim >= 1.")


def pos_def_sym_mats(val, val_name, exception_class):
    """Stack of symmetric positive-definite matrices, checked by Cholesky (reference _check.py:139-154)."""
    ok = type(val) is np.ndarray and val.ndim >= 2 and val.shape[-1] == val.shape[-2]
    if ok and np.allclose(val, np.swapaxes(val, -1, -2)):
        try:
            np.linalg.cholesky(val)
            return val
        except np.linalg.LinAlgError:
            raise exception_class(
                val_name + " must be a positive definite symmetric 2-dimensional numpy.ndarray.") from None
    raise exception_class(val_name + " must be a symmetric 2-dimensional numpy.ndarray.")


def floats(val, val_name, exception_class):
    """Real scalar, or numeric ndarray; integers are cast to float (reference _check.py:163-173)."""
    if _is_float(val):
        return val
    if _is_int(val):
        return float(val)
    if _is_array_of(val, np.integer):
        return val.astype(float)
    if _is_array_of(val, np.floating):
        return val
    raise exception_class(val_name + " must be float or a numpy.ndarray.")


def shape_consistency(val, val_name, correct, correct_name, exception_class):
    """`val` (a dimension) must equal `correct` (reference _check.py:268-272)."""
    if val != correct:
        raise exception_class(f"{val_name} must coincide with {correct_name}: "
                              f"{val_name} = {val}, {correct_name} = {correct}")


def pos_float(val, val_name, exception_class):
    """Positive real scalar; integers are cast to float (reference _check.py:19-26)."""
    if _is_float(val) and val > 0.0:
        return val
    if _is_int(val) and val > 0:
        return float(val)
    raise exception_class(val_name + " must be positive (not including 0.0).")


def pos_def_sym_mat(val, val_name, exception_class):
    """One symmetric positive-definite matrix, checked by Cholesky (reference _check.py:121-138)."""
    ok = type(val) is np.ndarray and val.ndim == 2 and val.shape[0] == val.shape[1]
    if ok and np.allclose(val, val.T):
        try:
            np.linalg.cholesky(val)
            return val
        except np.linalg.LinAlgError:
            raise exception_class(
                val_name + " must be a positive definite symmetric 2-dimensional numpy.ndarray.") from None
    raise exception_class(val_name + " must be a symmetric 2-dimensional numpy.ndarray.")
