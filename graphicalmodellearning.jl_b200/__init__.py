"""gml_b200: B200-native replacement of the learn() hot path of GraphicalModelLearning.jl."""
from .api import (B200, B200Exact, B200Gibbs, B200SwendsenWang, B200Tempering, Gibbs, GMLSampler, Session, NLP, RISE, RISEA, RPLE, FactorGraph, GMLFormulation,
                  GMLMethod, data_info, empirical_moments, fit_likelihood, learn, learn_matrix, learn_packed, log_likelihood, log_partition, logRISE, matrix_to_dict, moments, multiRISE, multirise_keys,
                  pack_histogram, regularizer_lambda, sample, sample_device, sample_terms_device)
from ._lib import GMLB200Error, LIB_PATH, Stats, Opts

__all__ = ["B200", "B200Exact", "B200Gibbs", "B200SwendsenWang", "B200Tempering", "Gibbs", "GMLSampler", "Session", "NLP", "RISE", "RISEA", "RPLE", "FactorGraph",
           "GMLFormulation", "GMLMethod", "data_info", "empirical_moments", "fit_likelihood", "learn", "learn_matrix", "learn_packed", "log_likelihood", "log_partition", "logRISE", "matrix_to_dict", "moments",
           "multiRISE", "multirise_keys", "pack_histogram", "regularizer_lambda", "sample", "sample_device",
           "sample_terms_device", "GMLB200Error", "LIB_PATH", "Stats", "Opts"]
