// korali_host.cpp — the host shim above the C ABI (include/kcma.h): a pybind11 module that mirrors Korali's own
// Python surface for ONE path — korali.Engine / korali.Experiment with "Solver": {"Type": "Optimizer/CMAES"} — so
// the reference's CMA-ES scripts run unchanged with `import korali_b200 as korali`.
//
// What is mirrored (reference file:line):
//   * KoraliJson cursor semantics of __getitem__/__setitem__      source/auxiliar/koraliJson.cpp:13-50, jsonInterface.cpp:42-64
//   * pybind11 class surface (Engine.run, Experiment.loadState)    source/engine.cpp:201-254
//   * Engine::run -> Experiment::initialize/run generation loop    source/engine.cpp:147-166, experiment.cpp.base:39-118,165-206
//   * generated CMAES/Optimizer/Solver setConfiguration: every known key is consumed, wrong types and left-over keys are
//     errors (" + Unrecognized settings for Korali module: CMAES: ...")   CMAES.cpp:1018-1782, source_builders.py:164-169
//   * getConfiguration result keys                                   CMAES.cpp:1784-1881
//   * finalize: e["Results"]["Best Sample"]                          CMAES.cpp.base:994-1010
//   * errors are std::runtime_error -> Python RuntimeError           logger.cpp:83-99
// What is NOT here: every other Korali module, conduit, problem type and solver (out of scope, SURVEY.md 2.1).
// The JSON tree is held as Python objects (dict / list / float / ...): the reference's knlohmann fork is not vendored.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/kcma.h"
#include "../../include/kdea.h"
#include "../../include/kmocma.h"
#include "../../include/ktmcmc.h"

namespace py = pybind11;

namespace {

[[noreturn]] void korali_error(const char* fmt, ...) {
  char buf[2048];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  throw std::runtime_error(std::string("\n[Korali] Error: ") + buf);
}

bool is_number(const py::handle& o) { return (py::isinstance<py::float_>(o) || py::isinstance<py::int_>(o)) && !py::isinstance<py::bool_>(o); }

// isElemental (jsonInterface.cpp:42-64): numbers, strings and arrays made only of those
bool is_elemental(const py::handle& o) {
  if (is_number(o)) return true;
  if (py::isinstance<py::str>(o)) return true;
  if (py::isinstance<py::list>(o)) {
    for (auto item : py::reinterpret_borrow<py::list>(o)) {
      bool ok = false;
      if (py::isinstance<py::list>(item)) ok = is_elemental(item);
      if (is_number(item) || py::isinstance<py::str>(item)) ok = true;
      if (!ok) return false;
    }
    return true;
  }
  return false;
}

// py2json: tuples become lists, numpy scalars become floats, callables are kept as they are (the reference stores an
// index into _functionVector, py2json.hpp:54-59; here the callable itself is the JSON leaf).
py::object normalise(const py::handle& v) {
  if (py::isinstance<py::dict>(v)) {
    py::dict d;
    for (auto kv : py::reinterpret_borrow<py::dict>(v)) d[kv.first] = normalise(kv.second);
    return d;
  }
  if (py::isinstance<py::list>(v) || py::isinstance<py::tuple>(v)) {
    py::list l;
    for (auto item : v) l.append(normalise(item));
    return l;
  }
  if (py::hasattr(v, "tolist") && !py::isinstance<py::str>(v)) return normalise(v.attr("tolist")());
  return py::reinterpret_borrow<py::object>(v);
}

// ---- a JSON tree with Korali's cursor -----------------------------------------------------------------------
class KoraliJson {
 public:
  py::dict _js;
  KoraliJson() { reset(); }
  virtual ~KoraliJson() = default;

  void reset() { _cur = _js; _parent = py::none(); _pkey = py::none(); }

  void traverse(const py::object& key) {
    if (!py::isinstance<py::str>(key) && !py::isinstance<py::int_>(key)) return;
    const bool is_str = py::isinstance<py::str>(key);
    // a null node becomes an object or an array depending on the first key used on it (nlohmann operator[])
    if (_cur.is_none()) {
      py::object fresh = is_str ? py::object(py::dict()) : py::object(py::list());
      if (!_parent.is_none()) _parent[_pkey] = fresh;
      _cur = fresh;
    }
    if (is_str) {
      if (!py::isinstance<py::dict>(_cur)) { reset(); korali_error("cannot use a string key on a JSON node that is not an object\n"); }
      py::dict d = py::reinterpret_borrow<py::dict>(_cur);
      if (!d.contains(key)) d[key] = py::none();
      _parent = d; _pkey = key; _cur = d[key];
    } else {
      if (!py::isinstance<py::list>(_cur)) { reset(); korali_error("cannot use an integer key on a JSON node that is not an array\n"); }
      py::list l = py::reinterpret_borrow<py::list>(_cur);
      const size_t i = key.cast<size_t>();
      while (py::len(l) <= i) l.append(py::none());
      _parent = l; _pkey = key; _cur = l[i];
    }
  }

  void setItem(const py::object key, const py::object val) {
    traverse(key);
    if (!_parent.is_none()) _parent[_pkey] = normalise(val);
    reset();
  }

  py::object getItem(const py::object key) {
    traverse(key);
    if (is_elemental(_cur)) {
      py::object tmp = _cur;
      reset();
      // whole-valued doubles come back as int (py2json.hpp:100-111)
      if (py::isinstance<py::float_>(tmp)) {
        const double d = tmp.cast<double>();
        if (std::isfinite(d) && d == std::floor(d) && std::fabs(d) < 9e15) return py::int_((long long)d);
      }
      return tmp;
    }
    return py::cast(this, py::return_value_policy::reference);
  }

 private:
  py::object _cur, _parent, _pkey;
};

// ---- helpers to read a settings object strictly ---------------------------------------------------------------
struct Settings {
  py::dict d;
  std::string module;
  Settings(py::dict dd, std::string m) : d(std::move(dd)), module(std::move(m)) {}
  bool has(const char* k) const { return d.contains(k); }
  py::object take(const char* k) {
    py::object v = d[k];
    PyDict_DelItemString(d.ptr(), k);
    return v;
  }
  double num(const char* k, double dflt) {
    if (!has(k)) return dflt;
    py::object v = take(k);
    if (!is_number(v)) korali_error(" + Object: [ %s ] \n + Key:    ['%s']\n + Reason: wrong type, a number was expected\n", module.c_str(), k);
    return v.cast<double>();
  }
  uint64_t uint(const char* k, uint64_t dflt) {
    if (!has(k)) return dflt;
    py::object v = take(k);
    if (!is_number(v)) korali_error(" + Object: [ %s ] \n + Key:    ['%s']\n + Reason: wrong type, an unsigned integer was expected\n", module.c_str(), k);
    const double x = v.cast<double>();
    if (std::isinf(x)) return x > 0 ? 0 : 0;  // size_t(Infinity) is 0 in the reference's release build (SURVEY Q2)
    if (x < 0) korali_error(" + Object: [ %s ] \n + Key:    ['%s']\n + Reason: negative value for an unsigned setting\n", module.c_str(), k);
    return (uint64_t)x;
  }
  int boolean(const char* k, int dflt) {
    if (!has(k)) return dflt;
    py::object v = take(k);
    if (py::isinstance<py::bool_>(v)) return v.cast<bool>() ? 1 : 0;
    if (is_number(v)) return v.cast<double>() != 0.0;
    korali_error(" + Object: [ %s ] \n + Key:    ['%s']\n + Reason: wrong type, a boolean was expected\n", module.c_str(), k);
  }
  std::string str(const char* k, const std::string& dflt) {
    if (!has(k)) return dflt;
    py::object v = take(k);
    if (!py::isinstance<py::str>(v)) korali_error(" + Object: [ %s ] \n + Key:    ['%s']\n + Reason: wrong type, a string was expected\n", module.c_str(), k);
    return v.cast<std::string>();
  }
  void finish() {
    if (py::len(d) == 0) return;
    std::string left = py::str(d).cast<std::string>();
    korali_error(" + Unrecognized settings for Korali module: %s: \n%s\n", module.c_str(), left.c_str());
  }
};

std::string canon(std::string s) {  // module types are compared case-insensitively with spaces stripped (module.cpp:103)
  std::string o;
  for (char c : s) if (c != ' ') o += (char)std::tolower((unsigned char)c);
  return o;
}

enum Verbosity { SILENT = 0, MINIMAL = 1, NORMAL = 2, DETAILED = 3 };

class Experiment;

// ---- the solver plug-in interface of this shim (the virtuals of Solver / Module that Experiment::initialize / run call,
// module.hpp:51-99, solver.hpp.base:65-85); selected by e["Solver"]["Type"] like Module::getModule (module.cpp:103-150)
class SolverBase {
 public:
  std::vector<double> lower, upper;
  std::vector<std::string> termination_criteria;
  std::string pending_error;
  virtual ~SolverBase() {}
  virtual const char* name() const = 0;
  virtual void setConfiguration(py::dict solver, py::list variables, py::dict problem, uint64_t seed) = 0;
  virtual void initialize(const std::vector<int>& device_ids) = 0;
  virtual void restore(uint64_t generation) = 0;
  virtual bool checkTermination() = 0;
  virtual void runGeneration() = 0;
  virtual void getConfiguration(py::dict js) = 0;
  virtual double scalar(const char* key) = 0;
  virtual std::vector<double> array(const char* key) = 0;
  virtual void printGeneration(const std::function<void(int, const char*)>& log) = 0;   // printGenerationAfter
  virtual std::string takeWarnings() { return ""; }
  virtual bool needsPython() const { return true; }   // a generation calls back into Python (models, constraints): the GIL stays held
  // finalize(): fills e["Results"] and prints the closing lines (CMAES.cpp.base:994-1010); false = the default single-objective form
  virtual bool finalize(py::dict results, const std::function<void(int, const char*)>& log) { (void)results; (void)log; return false; }
  virtual std::vector<std::pair<std::string, std::string>> sideCars() { return {}; }      // (key, file suffix) of N x N arrays saved as .npy
  virtual size_t variableCount() const = 0;
  void splitReasons(const char* reason) {
    termination_criteria.clear();
    std::string r(reason), item;
    for (char c : r) {
      if (c == ';') { if (!item.empty()) termination_criteria.push_back(item); item.clear(); }
      else item += c;
    }
  }
};

// One persistent host thread per additional device: with k["Conduit"]["Devices"] = G the population is sharded over G handles
// of this process, and the G calls of a generation must be in flight together (they meet in the NCCL collectives).
class RankPool {
 public:
  explicit RankPool(int n) : n_(n), rc_(n, 0) {
    for (int r = 1; r < n; r++) th_.emplace_back([this, r] { loop(r); });
  }
  ~RankPool() {
    { std::lock_guard<std::mutex> lk(m_); stop_ = true; epoch_++; }
    cv_.notify_all();
    for (auto& t : th_) t.join();
  }
  // fn(r) for every rank r (rank 0 on the caller's thread); returns the first failing rank + 1, or 0
  int run(const std::function<int(int)>& fn) {
    { std::lock_guard<std::mutex> lk(m_); fn_ = &fn; pending_ = n_ - 1; epoch_++; }
    cv_.notify_all();
    rc_[0] = fn(0);
    { std::unique_lock<std::mutex> lk(m_); done_.wait(lk, [&] { return pending_ == 0; }); }
    for (int r = 0; r < n_; r++) if (rc_[r]) return r + 1;
    return 0;
  }
 private:
  void loop(int r) {
    uint64_t seen = 0;
    for (;;) {
      std::unique_lock<std::mutex> lk(m_);
      cv_.wait(lk, [&] { return epoch_ != seen; });
      seen = epoch_;
      if (stop_) return;
      const std::function<int(int)>* f = fn_;
      lk.unlock();
      const int rc = (*f)(r);
      lk.lock();
      rc_[r] = rc;
      if (--pending_ == 0) done_.notify_one();
    }
  }
  int n_;
  std::vector<int> rc_;
  std::vector<std::thread> th_;
  std::mutex m_;
  std::condition_variable cv_, done_;
  const std::function<int(int)>* fn_ = nullptr;
  uint64_t epoch_ = 0;
  int pending_ = 0;
  bool stop_ = false;
};

// ---- the solver plug-in: Optimizer/CMAES on libkcma ----------------------------------------------------------
class CMAES : public SolverBase {
 public:
  kcma_t* h = nullptr;                  // rank 0 (the replicated state is read from it)
  std::vector<kcma_t*> hs;              // all ranks, one per device
  std::unique_ptr<RankPool> pool;
  kcma_cfg cfg;
  std::string mu_type = "Logarithmic";
  std::vector<double> init_val, init_sd, min_sd, gran;
  std::vector<std::string> names;
  py::object objective;                 // Python callable, or a string naming a built-in device objective
  std::vector<py::object> constraints;  // Python callables
  // termination criteria as given
  double tc_max_generations = 1e10, tc_max_model_evaluations = 1e9, tc_max_value = INFINITY, tc_min_value_diff = -INFINITY;
  double tc_max_infeasible = 0, tc_max_condition = INFINITY, tc_min_sd = -INFINITY, tc_max_sd = INFINITY;
  int devices = 1;

  const char* name() const override { return "Optimizer/CMAES"; }
  size_t variableCount() const override { return cfg.n; }
  std::string takeWarnings() override { const char* w = kcma_take_warnings(h); return w ? w : ""; }
  std::vector<std::pair<std::string, std::string>> sideCars() override {
    if ((uint64_t)cfg.n * cfg.n <= (1u << 22)) return {};
    return {{"Covariance Matrix", "C"}, {"Covariance Eigenvector Matrix", "B"}};
  }
  void printGeneration(const std::function<void(int, const char*)>& log) override {   // CMAES::printGenerationAfter :952-992
    char b[256];
    snprintf(b, sizeof(b), "Sigma:                        %+6.3e\n", scalar("Sigma")); log(NORMAL, b);
    snprintf(b, sizeof(b), "Current Function Value: Max = %+6.3e - Best = %+6.3e\n", scalar("Current Best Value"), scalar("Best Ever Value")); log(NORMAL, b);
    snprintf(b, sizeof(b), "Diagonal Covariance:    Min = %+6.3e -  Max = %+6.3e\n", scalar("Minimum Diagonal Covariance Matrix Element"),
             scalar("Maximum Diagonal Covariance Matrix Element")); log(NORMAL, b);
    snprintf(b, sizeof(b), "Covariance Eigenvalues: Min = %+6.3e -  Max = %+6.3e\n", scalar("Minimum Covariance Eigenvalue"), scalar("Maximum Covariance Eigenvalue"));
    log(NORMAL, b);
    snprintf(b, sizeof(b), "Number of Infeasible Samples: %zu\n", (size_t)scalar("Infeasible Sample Count")); log(DETAILED, b);
  }

  ~CMAES() {
    pool.reset();
    for (kcma_t* x : hs) if (x) kcma_destroy(x);
  }
  void each(const std::function<int(kcma_t*)>& fn) {
    for (kcma_t* x : hs) if (fn(x)) korali_error("%s", kcma_last_error(x));
  }

  void check(int rc) {
    if (rc) korali_error("%s", kcma_last_error(h));
  }

  double scalar(const char* key) override { double v = NAN; check(kcma_get_scalar(h, key, &v)); return v; }
  std::vector<double> array(const char* key) override {
    size_t n = 0;
    check(kcma_get_array(h, key, nullptr, 0, &n));
    std::vector<double> v(n);
    if (n) check(kcma_get_array(h, key, v.data(), n, &n));
    return v;
  }

  // generated CMAES::setConfiguration + Optimizer:: + Solver:: (strict)
  void setConfiguration(py::dict solver, py::list variables, py::dict problem, uint64_t seed) override {
    kcma_cfg_defaults(&cfg);
    Settings s(solver, "CMAES");
    s.take("Type");
    cfg.population_size = s.uint("Population Size", 0);
    cfg.mu_value = s.uint("Mu Value", 0);
    mu_type = s.str("Mu Type", "Logarithmic");
    if (mu_type == "Linear") cfg.mu_type = KCMA_MU_LINEAR;
    else if (mu_type == "Equal") cfg.mu_type = KCMA_MU_EQUAL;
    else if (mu_type == "Logarithmic") cfg.mu_type = KCMA_MU_LOGARITHMIC;
    else if (mu_type == "Proportional") cfg.mu_type = KCMA_MU_PROPORTIONAL;
    else korali_error("Invalid setting of Mu Type (%s) (Linear, Equal, Logarithmic, or Proportional accepted).", mu_type.c_str());
    cfg.initial_sigma_cumulation_factor = s.num("Initial Sigma Cumulation Factor", -1.0);
    cfg.initial_damp_factor = s.num("Initial Damp Factor", -1.0);
    cfg.use_gradient_information = s.boolean("Use Gradient Information", 0);
    cfg.gradient_step_size = (double)(float)s.num("Gradient Step Size", 0.01);   // a float in the reference (SURVEY Q9): dumps 0.009999999776...
    cfg.is_sigma_bounded = s.boolean("Is Sigma Bounded", 0);
    cfg.initial_cumulative_covariance = s.num("Initial Cumulative Covariance", -1.0);
    cfg.diagonal_covariance = s.boolean("Diagonal Covariance", 0);
    cfg.mirrored_sampling = s.boolean("Mirrored Sampling", 0);
    cfg.viability_population_size = s.uint("Viability Population Size", 2);
    cfg.viability_mu_value = s.uint("Viability Mu Value", 0);
    cfg.max_covariance_matrix_corrections = s.uint("Max Covariance Matrix Corrections", 1000000);
    cfg.target_success_rate = s.num("Target Success Rate", 0.1818);
    cfg.covariance_matrix_adaption_strength = s.num("Covariance Matrix Adaption Strength", 0.1);
    cfg.normal_vector_learning_rate = s.num("Normal Vector Learning Rate", -1.0);
    cfg.global_success_learning_rate = s.num("Global Success Learning Rate", 0.2);
    if (s.has("Termination Criteria")) {
      py::object tco = s.take("Termination Criteria");
      if (!py::isinstance<py::dict>(tco)) korali_error(" + Object: [ CMAES ] \n + Key:    ['Termination Criteria']\n + Reason: not an object\n");
      py::dict tcd;
      for (auto kv : py::reinterpret_borrow<py::dict>(tco)) tcd[kv.first] = kv.second;
      Settings tc(tcd, "CMAES['Termination Criteria']");
      tc_max_infeasible = (double)tc.uint("Max Infeasible Resamplings", 0);
      tc_max_condition = tc.num("Max Condition Covariance Matrix", INFINITY);
      tc_min_sd = tc.num("Min Standard Deviation", -INFINITY);
      tc_max_sd = tc.num("Max Standard Deviation", INFINITY);
      tc_max_value = tc.num("Max Value", INFINITY);
      tc_min_value_diff = tc.num("Min Value Difference Threshold", -INFINITY);
      tc_max_model_evaluations = tc.num("Max Model Evaluations", 1e9);
      tc_max_generations = tc.num("Max Generations", 1e10);
      tc.finish();
    }
    cfg.max_infeasible_resamplings = (uint64_t)tc_max_infeasible;
    // generators are part of the module defaults (CMAES.config:510-519). A saved state carries the Normal Generator's own
    // "Random Seed" (distribution.cpp.base:36-37): resuming with it continues the counter-based Philox stream exactly.
    for (const char* g : {"Normal Generator", "Uniform Generator"}) {
      if (!s.has(g)) continue;
      py::object go = s.take(g);
      if (std::string(g) == "Normal Generator" && py::isinstance<py::dict>(go)) {
        py::dict gd = py::reinterpret_borrow<py::dict>(go);
        if (gd.contains("Random Seed") && is_number(gd["Random Seed"]) && gd["Random Seed"].cast<double>() > 0) seed = (uint64_t)gd["Random Seed"].cast<double>();
      }
    }
    // "Internal Settings" (CMAES.config:137-483, optimizer.config, solver.config): present when a saved state is loaded;
    // consumed here like the generated code does and restored after kcma_create (restore()).
    static const char* kInternal[] = {
        "Is Viability Regime", "Value Vector", "Gradients", "Current Population Size", "Current Mu Value", "Mu Weights", "Effective Mu",
        "Sigma Cumulation Factor", "Damp Factor", "Cumulative Covariance", "Chi Square Number", "Covariance Eigenvalue Evaluation Frequency",
        "Sigma", "Trace", "Sample Population", "Finished Sample Count", "Current Best Variables", "Previous Best Value",
        "Previous Best Ever Value", "Sorting Index", "Covariance Matrix", "Auxiliar Covariance Matrix", "Covariance Eigenvector Matrix",
        "Auxiliar Covariance Eigenvector Matrix", "Axis Lengths", "Auxiliar Axis Lengths", "BDZ Matrix", "Auxiliar BDZ Matrix", "Current Mean",
        "Previous Mean", "Mean Update", "Evolution Path", "Conjugate Evolution Path", "Conjugate Evolution Path L2 Norm",
        "Infeasible Sample Count", "Maximum Diagonal Covariance Matrix Element", "Minimum Diagonal Covariance Matrix Element",
        "Maximum Covariance Eigenvalue", "Minimum Covariance Eigenvalue", "Is Eigensystem Updated", "Viability Indicator", "Has Constraints",
        "Covariance Matrix Adaption Factor", "Best Valid Sample", "Global Success Rate", "Viability Function Value", "Resampled Parameter Count",
        "Covariance Matrix Adaptation Count", "Viability Boundaries", "Viability Improvement", "Max Constraint Violation Count",
        "Sample Constraint Violation Counts", "Constraint Evaluations", "Normal Constraint Approximation", "Best Constraint Evaluations",
        "Has Discrete Variables", "Discrete Mutations", "Number Of Discrete Mutations", "Number Masking Matrix Entries", "Masking Matrix",
        "Masking Matrix Sigma", "Chi Square Number Discrete Mutations", "Current Min Standard Deviation", "Current Max Standard Deviation",
        "Constraint Evaluation Count", "Current Best Value", "Best Ever Value", "Best Ever Variables", "Variable Count", "Model Evaluation Count"};
    saved_internal = py::dict();
    for (const char* k : kInternal)
      if (s.has(k)) saved_internal[k] = s.take(k);
    // Result files written by older builds of the reference (the fixture tests/python/plot/cmaes/gen*.json is one) carry a few keys
    // that CMAES.config has since renamed or dropped; they are accepted so that such checkpoints load: 'Is Diagonal' is today's
    // 'Diagonal Covariance', the others are internal state without a successor.
    if (s.has("Is Diagonal")) { const int v = s.boolean("Is Diagonal", 0); if (v) cfg.diagonal_covariance = 1; }
    for (const char* k : {"Are Constraints Defined", "Best Sample Index", "Previous Value Vector"})
      if (s.has(k)) s.take(k);
    // variables (optimizer.config:45-82, CMAES.config Variable Defaults: Granularity 0.0)
    const size_t n = py::len(variables);
    if (n == 0) korali_error("Optimization Evaluation problems require at least one variable.\n");
    lower.assign(n, -INFINITY); upper.assign(n, INFINITY); init_val.assign(n, NAN); init_sd.assign(n, NAN); min_sd.assign(n, 0.0);
    gran.assign(n, 0.0);
    names.assign(n, "");
    for (size_t i = 0; i < n; i++) {
      if (!py::isinstance<py::dict>(variables[i])) korali_error("Variable %zu is not an object\n", i);
      py::dict vcopy;
      for (auto kv : py::reinterpret_borrow<py::dict>(variables[i])) vcopy[kv.first] = kv.second;
      Settings v(vcopy, "Variable");
      names[i] = v.str("Name", "");
      lower[i] = v.num("Lower Bound", -INFINITY);
      upper[i] = v.num("Upper Bound", INFINITY);
      init_val[i] = v.num("Initial Value", NAN);
      v.num("Initial Mean", NAN);
      init_sd[i] = v.num("Initial Standard Deviation", NAN);
      min_sd[i] = v.num("Minimum Standard Deviation Update", 0.0);
      if (v.has("Values")) v.take("Values");
      gran[i] = v.num("Granularity", 0.0);
      if (gran[i] < 0.0) korali_error("Negative granularity for variable '%s'.\n", names[i].c_str());   // CMAES.cpp.base:48
      v.finish();
    }
    cfg.n = n;
    cfg.lower_bound = lower.data(); cfg.upper_bound = upper.data(); cfg.initial_value = init_val.data();
    cfg.initial_stddev = init_sd.data(); cfg.min_stddev_update = min_sd.data(); cfg.granularity = gran.data();
    cfg.seed = seed;
    // problem (optimization.config)
    py::dict pcopy;
    for (auto kv : problem) pcopy[kv.first] = kv.second;
    Settings p(pcopy, "Optimization");
    const std::string ptype = canon(p.str("Type", ""));
    if (ptype != "optimization") korali_error("Only Problem Type 'Optimization' is served by the B200 CMA-ES path (got '%s')\n", ptype.c_str());
    if (!p.has("Objective Function")) korali_error(" + Object: [ Optimization ] \n + Key:    ['Objective Function']\n + Reason: mandatory setting missing\n");
    objective = p.take("Objective Function");
    p.uint("Num Objectives", 1);
    p.boolean("Has Discrete Variables", 0);
    constraints.clear();
    if (p.has("Constraints")) {
      py::object c = p.take("Constraints");
      if (!py::isinstance<py::list>(c)) korali_error(" + Object: [ Optimization ] \n + Key:    ['Constraints']\n + Reason: not an array\n");
      for (auto f : py::reinterpret_borrow<py::list>(c)) constraints.push_back(py::reinterpret_borrow<py::object>(f));
    }
    p.finish();
    cfg.n_constraints = constraints.size();
    cfg.constraint_family = constraints.empty() ? KCMA_CON_NONE : KCMA_CON_EXTERNAL;
    if (py::isinstance<py::str>(objective)) {
      const std::string o = canon(objective.cast<std::string>());
      if (o == "negsphere" || o == "sphere") cfg.objective = KCMA_OBJ_NEG_SPHERE;
      else if (o == "negrosenbrock" || o == "rosenbrock") cfg.objective = KCMA_OBJ_NEG_ROSENBROCK;
      else if (o == "negackley" || o == "ackley") cfg.objective = KCMA_OBJ_NEG_ACKLEY;
      else if (o == "negellipsoid" || o == "ellipsoid") cfg.objective = KCMA_OBJ_NEG_ELLIPSOID;
      else if (o == "negsumsq") cfg.objective = KCMA_OBJ_NEG_SUMSQ;
      else if (o == "negspheresin2") cfg.objective = KCMA_OBJ_NEG_SPHERE_SIN2;
      else korali_error("Unknown device objective '%s' (Sphere, Rosenbrock, Ackley, Ellipsoid, NegSumSq, NegSphereSin2)\n", o.c_str());
      cfg.keep_population = constraints.empty() ? 0 : 1;
    } else if (PyCallable_Check(objective.ptr())) {
      cfg.objective = KCMA_OBJ_EXTERNAL;
      cfg.keep_population = 1;
      // korali_b200.batched(fn) / korali_b200.batched_device(fn): the model takes the whole population in one call
      batched = py::hasattr(objective, "_korali_batched") ? objective.attr("_korali_batched").cast<std::string>() : std::string();
      if (!batched.empty() && batched != "numpy" && batched != "device") korali_error("Unknown batched model flavour '%s'\n", batched.c_str());
      if (!batched.empty() && cfg.use_gradient_information) korali_error("Batched models do not return gradients: use a per-sample model with 'Use Gradient Information'\n");
    } else {
      korali_error(" + Object: [ Optimization ] \n + Key:    ['Objective Function']\n + Reason: neither a callable nor the name of a device objective\n");
    }
    s.finish();
  }

  py::dict saved_internal;
  std::string batched;   // "", "numpy" or "device"

  // korali_b200.batched(fn): ONE call per generation with X as a (rows x N) NumPy view of the host copy of the population
  static void host_objective_batched(void* user, const double* x, uint64_t rows, uint64_t n, double* f_out) {
    CMAES* self = (CMAES*)user;
    try {
      py::array_t<double> X({(py::ssize_t)rows, (py::ssize_t)n}, {(py::ssize_t)(n * sizeof(double)), (py::ssize_t)sizeof(double)}, x, py::none());
      py::array_t<double, py::array::c_style | py::array::forcecast> F(self->objective(X));
      if ((uint64_t)F.size() != rows) korali_error("The batched model returned %zu values for %zu samples\n", (size_t)F.size(), (size_t)rows);
      const double* f = F.data();
      for (uint64_t i = 0; i < rows; i++) f_out[i] = f[i];
    } catch (const std::exception& e) {
      self->pending_error = e.what();
      for (uint64_t i = 0; i < rows; i++) f_out[i] = NAN;
    }
  }
  // korali_b200.batched_device(fn): the wrapper receives raw device pointers and builds zero-copy tensor views itself
  static void device_objective(void* user, const double* x_dev, uint64_t rows, uint64_t n, uint64_t ldx, double* f_dev, void* stream) {
    CMAES* self = (CMAES*)user;
    try {
      self->objective((uintptr_t)x_dev, rows, n, ldx, (uintptr_t)f_dev, (uintptr_t)stream);
    } catch (const std::exception& e) {
      self->pending_error = e.what();
    }
  }

  static void host_objective(void* user, const double* x, uint64_t rows, uint64_t n, double* f_out) {
    CMAES* self = (CMAES*)user;
    try {
      for (uint64_t i = 0; i < rows; i++) {
        py::dict sample;
        py::list params;
        for (uint64_t d = 0; d < n; d++) params.append(x[i * n + d]);
        sample["Parameters"] = params;
        sample["Sample Id"] = i;
        sample["Module"] = "Problem";
        sample["Operation"] = "Evaluate";
        self->objective(sample);
        if (!sample.contains("F(x)")) korali_error("The model did not set 'F(x)' for sample %zu\n", (size_t)i);
        f_out[i] = sample["F(x)"].cast<double>();
      }
    } catch (const std::exception& e) {
      self->pending_error = e.what();
      for (uint64_t i = 0; i < rows; i++) f_out[i] = NAN;
    }
  }
  // operation "Evaluate With Gradients" (CMAES.cpp.base:199-200, 226-228): the model sets "F(x)" and "Gradient"
  static void host_objective_grad(void* user, const double* x, uint64_t rows, uint64_t n, double* f_out, double* grad_out) {
    CMAES* self = (CMAES*)user;
    try {
      for (uint64_t i = 0; i < rows; i++) {
        py::dict sample;
        py::list params;
        for (uint64_t d = 0; d < n; d++) params.append(x[i * n + d]);
        sample["Parameters"] = params;
        sample["Sample Id"] = i;
        sample["Module"] = "Problem";
        sample["Operation"] = "Evaluate With Gradients";
        self->objective(sample);
        if (!sample.contains("F(x)")) korali_error("The model did not set 'F(x)' for sample %zu\n", (size_t)i);
        if (!sample.contains("Gradient")) korali_error("The model did not set 'Gradient' for sample %zu ('Use Gradient Information' is on)\n", (size_t)i);
        f_out[i] = sample["F(x)"].cast<double>();
        py::sequence grad = sample["Gradient"].cast<py::sequence>();
        if ((uint64_t)py::len(grad) != n) korali_error("'Gradient' of sample %zu has %zu entries, expected %zu\n", (size_t)i, (size_t)py::len(grad), (size_t)n);
        for (uint64_t d = 0; d < n; d++) grad_out[i * n + d] = grad[d].cast<double>();
      }
    } catch (const std::exception& e) {
      self->pending_error = e.what();
      for (uint64_t i = 0; i < rows; i++) f_out[i] = NAN;
      for (uint64_t i = 0; i < rows * n; i++) grad_out[i] = 0.0;
    }
  }
  static void host_constraints(void* user, const double* x, uint64_t rows, uint64_t n, double* g_out, uint64_t nc) {
    CMAES* self = (CMAES*)user;
    try {
      for (uint64_t i = 0; i < rows; i++) {
        py::list params;
        for (uint64_t d = 0; d < n; d++) params.append(x[i * n + d]);
        for (uint64_t c = 0; c < nc; c++) {
          py::dict sample;
          sample["Parameters"] = params;
          sample["Sample Id"] = 0;
          sample["Module"] = "Problem";
          sample["Operation"] = "Evaluate Constraints";
          self->constraints[c](sample);
          g_out[c * rows + i] = sample["F(x)"].cast<double>();
        }
      }
    } catch (const std::exception& e) {
      self->pending_error = e.what();
      for (uint64_t i = 0; i < rows * nc; i++) g_out[i] = NAN;
    }
  }

  void initialize(const std::vector<int>& device_ids) override {
    const int G = (int)device_ids.size();
    if (G > 1 && (cfg.objective == KCMA_OBJ_EXTERNAL || !constraints.empty()))
      korali_error("k['Conduit']['Devices'] > 1 shards the population over several GPUs of this process: it needs a device objective "
                   "(e['Problem']['Objective Function'] = 'Ellipsoid' ...) and no constraints; Python models run on one device\n");
    for (int r = 0; r < G; r++) {
      cfg.device = device_ids[r]; cfg.rank = r; cfg.nranks = G;
      kcma_t* x = nullptr;
      if (kcma_create(&cfg, &x)) korali_error("%s", kcma_last_error(nullptr));
      hs.push_back(x);
    }
    h = hs[0];
    if (G > 1) {
      if (kcma_comm_init_all(hs.data(), G)) korali_error("%s", kcma_last_error(h));
      pool = std::make_unique<RankPool>(G);
    }
    if (cfg.objective == KCMA_OBJ_EXTERNAL) {
      if (cfg.use_gradient_information) check(kcma_set_host_objective_grad(h, &CMAES::host_objective_grad, this));
      else if (batched == "device") check(kcma_set_device_objective(h, &CMAES::device_objective, this));
      else if (batched == "numpy") check(kcma_set_host_objective(h, &CMAES::host_objective_batched, this));
      else check(kcma_set_host_objective(h, &CMAES::host_objective, this));
    }
    if (!constraints.empty()) check(kcma_set_host_constraints(h, &CMAES::host_constraints, this));
    each([&](kcma_t* x) {
      return kcma_set_scalar(x, "Termination Criteria/Max Condition Covariance Matrix", tc_max_condition) ||
             kcma_set_scalar(x, "Termination Criteria/Min Standard Deviation", tc_min_sd) ||
             kcma_set_scalar(x, "Termination Criteria/Max Standard Deviation", tc_max_sd) ||
             kcma_set_scalar(x, "Termination Criteria/Max Value", tc_max_value) ||
             kcma_set_scalar(x, "Termination Criteria/Min Value Difference Threshold", tc_min_value_diff) ||
             kcma_set_scalar(x, "Termination Criteria/Max Model Evaluations", tc_max_model_evaluations) ||
             kcma_set_scalar(x, "Termination Criteria/Max Generations", tc_max_generations);
    });
  }

  // restore "Internal Settings" of a loaded state (CMAES.cpp:1042-1560): resume continues from the saved generation
  void restore(uint64_t generation) override {
    if (generation == 0) return;
    auto arr = [&](const char* k) {
      if (!saved_internal.contains(k)) return;
      std::vector<double> v = py::cast<std::vector<double>>(saved_internal[k]);
      each([&](kcma_t* x) { return kcma_set_array(x, k, v.data(), v.size()); });
    };
    auto sca = [&](const char* k) {
      if (!saved_internal.contains(k)) return;
      const double v = saved_internal[k].cast<double>();
      each([&](kcma_t* x) { return kcma_set_scalar(x, k, v); });
    };
    // the regime first: it fixes the population size / mu the arrays below are sized by, and re-derives the weights
    if (!constraints.empty()) sca("Is Viability Regime");
    for (const char* k : {"Covariance Matrix", "Current Mean", "Previous Mean", "Evolution Path", "Conjugate Evolution Path",
                          "Best Ever Variables", "Current Best Variables", "Axis Lengths", "Covariance Eigenvector Matrix", "Mean Update"})
      arr(k);
    if (saved_internal.contains("Mu Weights") && mu_type == "Proportional") arr("Mu Weights");   // data-dependent weights (:584-600)
    if (!constraints.empty()) {
      for (const char* k : {"Viability Boundaries", "Best Constraint Evaluations"}) arr(k);
      if (saved_internal.contains("Normal Constraint Approximation")) {   // saved as a C x N array of arrays
        std::vector<double> flat;
        for (auto row : saved_internal["Normal Constraint Approximation"]) for (auto x : row) flat.push_back(x.cast<double>());
        if (!flat.empty()) each([&](kcma_t* x) { return kcma_set_array(x, "Normal Constraint Approximation", flat.data(), flat.size()); });
      }
      for (const char* k : {"Global Success Rate", "Resampled Parameter Count", "Covariance Matrix Adaptation Count",
                            "Max Constraint Violation Count", "Constraint Evaluation Count", "Best Valid Sample"})
        sca(k);
    }
    for (const char* k : {"Sigma", "Best Ever Value", "Current Best Value", "Previous Best Value", "Previous Best Ever Value",
                          "Conjugate Evolution Path L2 Norm", "Infeasible Sample Count", "Model Evaluation Count",
                          "Maximum Covariance Eigenvalue", "Minimum Covariance Eigenvalue", "Current Min Standard Deviation",
                          "Current Max Standard Deviation", "Maximum Diagonal Covariance Matrix Element",
                          "Minimum Diagonal Covariance Matrix Element"})
      sca(k);
    each([&](kcma_t* x) { return kcma_set_scalar(x, "Current Generation", (double)generation); });
  }

  bool checkTermination() override {
    int fin = 0;
    const char* reason = "";
    check(kcma_check_termination(h, &fin, &reason));
    if (fin) splitReasons(reason);
    return fin != 0;
  }

  void runGeneration() override {
    pending_error.clear();
    if (pool) {   // one call per device, in flight together
      const int failed = pool->run([this](int r) { return kcma_run_generation(hs[r]); });
      if (failed) korali_error("%s", kcma_last_error(hs[failed - 1]));
      return;
    }
    int rc;
    if (!needsPython()) { py::gil_scoped_release nogil; rc = kcma_run_generation(h); }   // other experiments' threads run meanwhile
    else rc = kcma_run_generation(h);
    if (!pending_error.empty()) { std::string e = pending_error; pending_error.clear(); throw std::runtime_error(e); }
    check(rc);
  }
  bool needsPython() const override { return cfg.objective == KCMA_OBJ_EXTERNAL || !constraints.empty(); }

  // generated getConfiguration (CMAES.cpp:1784-1881): settings + internal state under Korali's key names.
  // Size policy: lambda x N arrays are exported only when small (SURVEY 5.4: they cannot be serialised at scale).
  void getConfiguration(py::dict js) override {
    js["Type"] = "Optimizer/CMAES";
    js["Population Size"] = cfg.population_size;
    js["Mu Value"] = cfg.mu_value;
    js["Mu Type"] = mu_type;
    js["Initial Sigma Cumulation Factor"] = cfg.initial_sigma_cumulation_factor;
    js["Initial Damp Factor"] = cfg.initial_damp_factor;
    js["Use Gradient Information"] = cfg.use_gradient_information;
    js["Gradient Step Size"] = cfg.gradient_step_size;
    js["Is Sigma Bounded"] = cfg.is_sigma_bounded;
    js["Initial Cumulative Covariance"] = cfg.initial_cumulative_covariance;
    js["Diagonal Covariance"] = cfg.diagonal_covariance;
    js["Mirrored Sampling"] = cfg.mirrored_sampling;
    js["Viability Population Size"] = cfg.viability_population_size;
    js["Viability Mu Value"] = cfg.viability_mu_value;
    js["Max Covariance Matrix Corrections"] = cfg.max_covariance_matrix_corrections;
    js["Target Success Rate"] = cfg.target_success_rate;
    js["Covariance Matrix Adaption Strength"] = cfg.covariance_matrix_adaption_strength;
    js["Normal Vector Learning Rate"] = cfg.normal_vector_learning_rate;
    js["Global Success Learning Rate"] = cfg.global_success_learning_rate;
    py::dict tc;
    tc["Max Infeasible Resamplings"] = tc_max_infeasible;
    tc["Max Condition Covariance Matrix"] = tc_max_condition;
    tc["Min Standard Deviation"] = tc_min_sd;
    tc["Max Standard Deviation"] = tc_max_sd;
    tc["Max Value"] = tc_max_value;
    tc["Min Value Difference Threshold"] = tc_min_value_diff;
    tc["Max Model Evaluations"] = tc_max_model_evaluations;
    tc["Max Generations"] = tc_max_generations;
    js["Termination Criteria"] = tc;
    py::dict ng, ug;
    ng["Type"] = "Univariate/Normal"; ng["Mean"] = 0.0; ng["Standard Deviation"] = 1.0; ng["Random Seed"] = cfg.seed;
    ug["Type"] = "Univariate/Uniform"; ug["Minimum"] = 0.0; ug["Maximum"] = 1.0; ug["Random Seed"] = cfg.seed + 1;
    js["Normal Generator"] = ng; js["Uniform Generator"] = ug;
    for (const char* k : {"Sigma", "Trace", "Effective Mu", "Sigma Cumulation Factor", "Damp Factor", "Cumulative Covariance", "Chi Square Number",
                          "Conjugate Evolution Path L2 Norm", "Best Ever Value", "Previous Best Ever Value", "Current Best Value",
                          "Maximum Diagonal Covariance Matrix Element", "Minimum Diagonal Covariance Matrix Element",
                          "Maximum Covariance Eigenvalue", "Minimum Covariance Eigenvalue", "Current Min Standard Deviation",
                          "Current Max Standard Deviation", "Global Success Rate"})
      js[k] = scalar(k);
    js["Previous Best Value"] = 0.0;  // the base-class copy the reference serialises (SURVEY Q1)
    for (const char* k : {"Model Evaluation Count", "Variable Count", "Current Population Size", "Current Mu Value", "Infeasible Sample Count",
                          "Is Viability Regime", "Has Constraints"})
      js[k] = (long long)scalar(k);
    if (!constraints.empty())
      for (const char* k : {"Resampled Parameter Count", "Covariance Matrix Adaptation Count", "Max Constraint Violation Count",
                            "Constraint Evaluation Count", "Best Valid Sample"})
        js[k] = (long long)scalar(k);
    for (const char* k : {"Current Mean", "Previous Mean", "Mean Update", "Evolution Path", "Conjugate Evolution Path", "Axis Lengths",
                          "Best Ever Variables", "Current Best Variables", "Mu Weights"})
      js[k] = array(k);
    const uint64_t n = cfg.n, lam = (uint64_t)scalar("Current Population Size");
    if (n * n <= (1u << 22)) {
      js["Covariance Matrix"] = array("Covariance Matrix");
      js["Covariance Eigenvector Matrix"] = array("Covariance Eigenvector Matrix");
    }
    if (lam <= (1u << 20)) {
      js["Value Vector"] = array("Value Vector");
      size_t cnt = 0;
      std::vector<uint64_t> idx(lam);
      if (scalar("Current Generation") > 0 && !kcma_get_index_array(h, "Sorting Index", idx.data(), lam, &cnt)) js["Sorting Index"] = idx;
    }
    if (cfg.keep_population && lam * n <= (1u << 22)) {
      std::vector<double> flat = array("Sample Population");
      py::list pop;
      for (uint64_t i = 0; i * n < flat.size(); i++) pop.append(std::vector<double>(flat.begin() + i * n, flat.begin() + (i + 1) * n));
      js["Sample Population"] = pop;
    }
    if (!constraints.empty()) {
      js["Viability Boundaries"] = array("Viability Boundaries");
      js["Best Constraint Evaluations"] = array("Best Constraint Evaluations");
      std::vector<double> flat = array("Normal Constraint Approximation");
      py::list rows;
      for (size_t c = 0; c * n < flat.size(); c++) rows.append(std::vector<double>(flat.begin() + c * n, flat.begin() + (c + 1) * n));
      js["Normal Constraint Approximation"] = rows;
    }
  }
};

// ---- the solver plug-in: Optimizer/DEA on libkcma (include/kdea.h) -------------------------------------------------
class DEA : public SolverBase {
 public:
  kdea_t* h = nullptr;
  kdea_cfg cfg;
  std::string mutation_rule = "Fixed", parent_rule = "Random", accept_rule = "Greedy", batched;
  py::object objective;
  double tc_max_generations = 1e10, tc_max_model_evaluations = 1e9, tc_max_value = INFINITY, tc_min_value_diff = -INFINITY;
  double tc_max_infeasible = 1e7, tc_min_value = -INFINITY, tc_min_step = -INFINITY;
  py::dict saved_internal;

  ~DEA() override { if (h) kdea_destroy(h); }
  const char* name() const override { return "Optimizer/DEA"; }
  size_t variableCount() const override { return cfg.n; }
  void check(int rc) { if (rc) korali_error("%s", kdea_last_error(h)); }
  double scalar(const char* key) override { double v = NAN; check(kdea_get_scalar(h, key, &v)); return v; }
  std::vector<double> array(const char* key) override {
    size_t n = 0;
    check(kdea_get_array(h, key, nullptr, 0, &n));
    std::vector<double> v(n);
    if (n) check(kdea_get_array(h, key, v.data(), n, &n));
    return v;
  }

  // generated DEA::setConfiguration (DEA.config) + Optimizer:: + Solver:: (strict)
  void setConfiguration(py::dict solver, py::list variables, py::dict problem, uint64_t seed) override {
    kdea_cfg_defaults(&cfg);
    uint64_t uniform_seed = 0;
    Settings s(solver, "DEA");
    s.take("Type");
    cfg.population_size = s.uint("Population Size", 200);
    cfg.crossover_rate = s.num("Crossover Rate", 0.9);
    cfg.mutation_rate = s.num("Mutation Rate", 0.5);
    mutation_rule = s.str("Mutation Rule", "Fixed");
    parent_rule = s.str("Parent Selection Rule", "Random");
    accept_rule = s.str("Accept Rule", "Greedy");
    cfg.fix_infeasible = s.boolean("Fix Infeasible", 1);
    if (mutation_rule == "Fixed") cfg.mutation_rule = KDEA_MUTATION_FIXED;
    else if (mutation_rule == "Self Adaptive") korali_error("Mutation Rule 'Self Adaptive' is not built on the B200 path (DEA.cpp.base:136-156)\n");
    else korali_error("Invalid setting of Mutation Rule (%s) (Fixed or Self Adaptive accepted).\n", mutation_rule.c_str());
    if (parent_rule == "Random") cfg.parent_selection_rule = KDEA_PARENT_RANDOM;
    else if (parent_rule == "Best") cfg.parent_selection_rule = KDEA_PARENT_BEST;
    else korali_error("Invalid setting of Parent Selection Rule (%s) (Random or Best accepted).\n", parent_rule.c_str());
    if (accept_rule == "Best") cfg.accept_rule = KDEA_ACCEPT_BEST;
    else if (accept_rule == "Greedy") cfg.accept_rule = KDEA_ACCEPT_GREEDY;
    else if (accept_rule == "Improved") cfg.accept_rule = KDEA_ACCEPT_IMPROVED;
    else if (accept_rule == "Iterative") cfg.accept_rule = KDEA_ACCEPT_ITERATIVE;
    else korali_error("Accept Rule (%s) not recognized.\n", accept_rule.c_str());
    if (s.has("Termination Criteria")) {
      py::object tco = s.take("Termination Criteria");
      if (!py::isinstance<py::dict>(tco)) korali_error(" + Object: [ DEA ] \n + Key:    ['Termination Criteria']\n + Reason: not an object\n");
      py::dict tcd;
      for (auto kv : py::reinterpret_borrow<py::dict>(tco)) tcd[kv.first] = kv.second;
      Settings tc(tcd, "DEA['Termination Criteria']");
      tc_max_infeasible = tc.num("Max Infeasible Resamplings", 1e7);
      tc_min_value = tc.num("Min Value", -INFINITY);
      tc_min_step = tc.num("Min Step Size", -INFINITY);
      tc_max_value = tc.num("Max Value", INFINITY);
      tc_min_value_diff = tc.num("Min Value Difference Threshold", -INFINITY);
      tc_max_model_evaluations = tc.num("Max Model Evaluations", 1e9);
      tc_max_generations = tc.num("Max Generations", 1e10);
      tc.finish();
    }
    for (const char* g : {"Normal Generator", "Uniform Generator"}) {
      if (!s.has(g)) continue;
      py::object go = s.take(g);
      if (std::string(g) == "Uniform Generator" && py::isinstance<py::dict>(go)) {
        py::dict gd = py::reinterpret_borrow<py::dict>(go);
        if (gd.contains("Random Seed") && is_number(gd["Random Seed"]) && gd["Random Seed"].cast<double>() > 0) uniform_seed = (uint64_t)gd["Random Seed"].cast<double>();
      }
    }
    static const char* kInternal[] = {"Value Vector", "Previous Value Vector", "Sample Population", "Candidate Population", "Best Sample Index",
                                      "Best Ever Value", "Previous Best Ever Value", "Current Best Value", "Previous Best Value", "Current Mean",
                                      "Previous Mean", "Best Ever Variables", "Current Best Variables", "Max Distances", "Infeasible Sample Count",
                                      "Current Minimum Step Size", "Variable Count", "Model Evaluation Count"};
    saved_internal = py::dict();
    for (const char* k : kInternal)
      if (s.has(k)) saved_internal[k] = s.take(k);
    const size_t n = py::len(variables);
    if (n == 0) korali_error("Optimization Evaluation problems require at least one variable.\n");
    lower.assign(n, -INFINITY); upper.assign(n, INFINITY);
    for (size_t i = 0; i < n; i++) {
      if (!py::isinstance<py::dict>(variables[i])) korali_error("Variable %zu is not an object\n", i);
      py::dict vcopy;
      for (auto kv : py::reinterpret_borrow<py::dict>(variables[i])) vcopy[kv.first] = kv.second;
      Settings v(vcopy, "Variable");
      v.str("Name", "");
      lower[i] = v.num("Lower Bound", -INFINITY);
      upper[i] = v.num("Upper Bound", INFINITY);
      for (const char* k : {"Initial Value", "Initial Mean", "Initial Standard Deviation", "Minimum Standard Deviation Update", "Granularity"}) v.num(k, NAN);
      if (v.has("Values")) v.take("Values");
      v.finish();
    }
    cfg.n = n; cfg.lower_bound = lower.data(); cfg.upper_bound = upper.data();
    cfg.seed = uniform_seed ? uniform_seed : seed + 1;   // Uniform Generator = S + 1 (distribution.cpp.base:36-37: Normal S, Uniform S + 1); a saved state carries its own
    py::dict pcopy;
    for (auto kv : problem) pcopy[kv.first] = kv.second;
    Settings p(pcopy, "Optimization");
    const std::string ptype = canon(p.str("Type", ""));
    if (ptype != "optimization") korali_error("Only Problem Type 'Optimization' is served by the B200 path (got '%s')\n", ptype.c_str());
    if (!p.has("Objective Function")) korali_error(" + Object: [ Optimization ] \n + Key:    ['Objective Function']\n + Reason: mandatory setting missing\n");
    objective = p.take("Objective Function");
    p.uint("Num Objectives", 1);
    p.boolean("Has Discrete Variables", 0);
    if (p.has("Constraints")) {
      py::object c = p.take("Constraints");
      if (py::isinstance<py::list>(c) && py::len(c) > 0) korali_error("Optimizer/DEA does not take constraints\n");
    }
    p.finish();
    if (py::isinstance<py::str>(objective)) {
      const std::string o = canon(objective.cast<std::string>());
      if (o == "negsphere" || o == "sphere") cfg.objective = KCMA_OBJ_NEG_SPHERE;
      else if (o == "negrosenbrock" || o == "rosenbrock") cfg.objective = KCMA_OBJ_NEG_ROSENBROCK;
      else if (o == "negackley" || o == "ackley") cfg.objective = KCMA_OBJ_NEG_ACKLEY;
      else if (o == "negellipsoid" || o == "ellipsoid") cfg.objective = KCMA_OBJ_NEG_ELLIPSOID;
      else if (o == "negsumsq") cfg.objective = KCMA_OBJ_NEG_SUMSQ;
      else if (o == "negspheresin2") cfg.objective = KCMA_OBJ_NEG_SPHERE_SIN2;
      else korali_error("Unknown device objective '%s' (Sphere, Rosenbrock, Ackley, Ellipsoid, NegSumSq, NegSphereSin2)\n", o.c_str());
    } else if (PyCallable_Check(objective.ptr())) {
      cfg.objective = KCMA_OBJ_EXTERNAL;
      batched = py::hasattr(objective, "_korali_batched") ? objective.attr("_korali_batched").cast<std::string>() : std::string();
      if (batched == "device") korali_error("Optimizer/DEA takes per-sample models and korali.batched(fn) models (not device-tensor models)\n");
    } else {
      korali_error(" + Object: [ Optimization ] \n + Key:    ['Objective Function']\n + Reason: neither a callable nor the name of a device objective\n");
    }
    s.finish();
  }

  static void host_objective(void* user, const double* x, uint64_t rows, uint64_t n, double* f_out) {
    DEA* self = (DEA*)user;
    try {
      if (self->batched == "numpy") {
        py::array_t<double> X({(py::ssize_t)rows, (py::ssize_t)n}, {(py::ssize_t)(n * sizeof(double)), (py::ssize_t)sizeof(double)}, x, py::none());
        py::array_t<double, py::array::c_style | py::array::forcecast> F(self->objective(X));
        if ((uint64_t)F.size() != rows) korali_error("The batched model returned %zu values for %zu samples\n", (size_t)F.size(), (size_t)rows);
        for (uint64_t i = 0; i < rows; i++) f_out[i] = F.data()[i];
        return;
      }
      for (uint64_t i = 0; i < rows; i++) {
        py::dict sample;
        py::list params;
        for (uint64_t d = 0; d < n; d++) params.append(x[i * n + d]);
        sample["Parameters"] = params;
        sample["Sample Id"] = i;
        sample["Module"] = "Problem";
        sample["Operation"] = "Evaluate";
        self->objective(sample);
        if (!sample.contains("F(x)")) korali_error("The model did not set 'F(x)' for sample %zu\n", (size_t)i);
        f_out[i] = sample["F(x)"].cast<double>();
      }
    } catch (const std::exception& e) {
      self->pending_error = e.what();
      for (uint64_t i = 0; i < rows; i++) f_out[i] = NAN;
    }
  }

  void initialize(const std::vector<int>& device_ids) override {
    if (device_ids.size() > 1) korali_error("Optimizer/DEA runs on one device (k['Conduit']['Devices'] > 1 is built for Optimizer/CMAES)\n");
    cfg.device = device_ids[0];
    if (kdea_create(&cfg, &h)) korali_error("%s", kdea_last_error(nullptr));
    if (cfg.objective == KCMA_OBJ_EXTERNAL) check(kdea_set_host_objective(h, &DEA::host_objective, this));
    check(kdea_set_scalar(h, "Termination Criteria/Max Infeasible Resamplings", tc_max_infeasible));
    check(kdea_set_scalar(h, "Termination Criteria/Min Value", tc_min_value));
    check(kdea_set_scalar(h, "Termination Criteria/Min Step Size", tc_min_step));
    check(kdea_set_scalar(h, "Termination Criteria/Max Value", tc_max_value));
    check(kdea_set_scalar(h, "Termination Criteria/Min Value Difference Threshold", tc_min_value_diff));
    check(kdea_set_scalar(h, "Termination Criteria/Max Model Evaluations", tc_max_model_evaluations));
    check(kdea_set_scalar(h, "Termination Criteria/Max Generations", tc_max_generations));
  }

  void restore(uint64_t generation) override {
    if (generation == 0) return;
    auto flat = [&](py::handle o) {
      std::vector<double> v;
      for (auto row : o) {
        if (py::isinstance<py::list>(row) || py::isinstance<py::tuple>(row)) for (auto x : row) v.push_back(x.cast<double>());
        else v.push_back(row.cast<double>());
      }
      return v;
    };
    for (const char* k : {"Sample Population", "Candidate Population", "Value Vector", "Previous Value Vector", "Current Mean", "Previous Mean",
                          "Best Ever Variables", "Current Best Variables", "Max Distances"})
      if (saved_internal.contains(k)) { std::vector<double> v = flat(saved_internal[k]); check(kdea_set_array(h, k, v.data(), v.size())); }
    for (const char* k : {"Best Ever Value", "Previous Best Ever Value", "Current Best Value", "Previous Best Value", "Best Sample Index",
                          "Infeasible Sample Count", "Model Evaluation Count"})
      if (saved_internal.contains(k)) check(kdea_set_scalar(h, k, saved_internal[k].cast<double>()));
    check(kdea_set_scalar(h, "Current Generation", (double)generation));
  }

  bool checkTermination() override {
    int fin = 0;
    const char* reason = "";
    check(kdea_check_termination(h, &fin, &reason));
    if (fin) splitReasons(reason);
    return fin != 0;
  }

  void runGeneration() override {
    pending_error.clear();
    int rc;
    if (!needsPython()) { py::gil_scoped_release nogil; rc = kdea_run_generation(h); }
    else rc = kdea_run_generation(h);
    if (!pending_error.empty()) { std::string e = pending_error; pending_error.clear(); throw std::runtime_error(e); }
    check(rc);
  }
  bool needsPython() const override { return cfg.objective == KCMA_OBJ_EXTERNAL; }

  void printGeneration(const std::function<void(int, const char*)>& log) override {   // DEA::printGenerationAfter :290-299
    char b[256];
    snprintf(b, sizeof(b), "Current Function Value: Max = %+6.3e - Best = %+6.3e\n", scalar("Current Best Value"), scalar("Best Ever Value")); log(NORMAL, b);
    snprintf(b, sizeof(b), "Number of Infeasible Samples: %zu\n", (size_t)scalar("Infeasible Sample Count")); log(DETAILED, b);
  }

  // generated getConfiguration: settings + internal state under Korali's key names (DEA.config)
  void getConfiguration(py::dict js) override {
    js["Type"] = "Optimizer/DEA";
    js["Population Size"] = cfg.population_size;
    js["Crossover Rate"] = cfg.crossover_rate;
    js["Mutation Rate"] = cfg.mutation_rate;
    js["Mutation Rule"] = mutation_rule;
    js["Parent Selection Rule"] = parent_rule;
    js["Accept Rule"] = accept_rule;
    js["Fix Infeasible"] = cfg.fix_infeasible;
    py::dict tc;
    tc["Max Infeasible Resamplings"] = tc_max_infeasible; tc["Min Value"] = tc_min_value; tc["Min Step Size"] = tc_min_step;
    tc["Max Value"] = tc_max_value; tc["Min Value Difference Threshold"] = tc_min_value_diff;
    tc["Max Model Evaluations"] = tc_max_model_evaluations; tc["Max Generations"] = tc_max_generations;
    js["Termination Criteria"] = tc;
    py::dict ng, ug;
    ng["Type"] = "Univariate/Normal"; ng["Mean"] = 0.0; ng["Standard Deviation"] = 1.0; ng["Random Seed"] = cfg.seed - 1;
    ug["Type"] = "Univariate/Uniform"; ug["Minimum"] = 0.0; ug["Maximum"] = 1.0; ug["Random Seed"] = cfg.seed;
    js["Normal Generator"] = ng; js["Uniform Generator"] = ug;
    for (const char* k : {"Best Ever Value", "Previous Best Ever Value", "Current Best Value", "Previous Best Value", "Current Minimum Step Size"})
      js[k] = scalar(k);
    for (const char* k : {"Best Sample Index", "Infeasible Sample Count", "Model Evaluation Count", "Variable Count"}) js[k] = (long long)scalar(k);
    for (const char* k : {"Current Mean", "Previous Mean", "Best Ever Variables", "Current Best Variables", "Max Distances", "Value Vector",
                          "Previous Value Vector"})
      js[k] = array(k);
    const uint64_t n = cfg.n, lam = cfg.population_size;
    if (lam * n <= (1u << 22))
      for (const char* k : {"Sample Population", "Candidate Population"}) {
        std::vector<double> flat = array(k);
        py::list pop;
        for (uint64_t i = 0; i * n < flat.size(); i++) pop.append(std::vector<double>(flat.begin() + i * n, flat.begin() + (i + 1) * n));
        js[k] = pop;
      }
  }
};

// ---- Experiment ------------------------------------------------------------------------------------------------
// ---- the solver plug-in: Optimizer/MOCMAES on libkcma (include/kmocma.h) ----------------------------------------------
class MOCMAES : public SolverBase {
 public:
  kmocma_t* h = nullptr;
  kmocma_cfg cfg;
  std::vector<double> init_val, init_sd;
  std::string batched;
  py::object objective;
  double tc_max_generations = 1e10, tc_max_model_evaluations = 1e9, tc_max_value = INFINITY, tc_min_value_diff = -INFINITY;
  double tc_min_max_value_diff = -INFINITY, tc_min_var_diff = -INFINITY, tc_min_sd = -INFINITY, tc_max_sd = INFINITY;

  ~MOCMAES() override { if (h) kmocma_destroy(h); }
  const char* name() const override { return "Optimizer/MOCMAES"; }
  size_t variableCount() const override { return cfg.n; }
  void check(int rc) { if (rc) korali_error("%s", kmocma_last_error(h)); }
  double scalar(const char* key) override {
    if (!strcmp(key, "Best Ever Value")) return NAN;    // the base-class scalars are disabled by MOCMAES (:64-66)
    double v = NAN; check(kmocma_get_scalar(h, key, &v)); return v;
  }
  std::vector<double> array(const char* key) override {
    size_t n = 0;
    check(kmocma_get_array(h, key, nullptr, 0, &n));
    std::vector<double> v(n);
    if (n) check(kmocma_get_array(h, key, v.data(), n, &n));
    return v;
  }

  // generated MOCMAES::setConfiguration (MOCMAES.config) + Optimizer:: + Solver:: (strict)
  void setConfiguration(py::dict solver, py::list variables, py::dict problem, uint64_t seed) override {
    kmocma_cfg_defaults(&cfg);
    Settings s(solver, "MOCMAES");
    s.take("Type");
    cfg.population_size = s.uint("Population Size", 0);
    cfg.mu_value = s.uint("Mu Value", 0);
    cfg.evolution_path_adaption_strength = s.num("Evolution Path Adaption Strength", -1.0);
    cfg.covariance_learning_rate = s.num("Covariance Learning Rate", -1.0);
    cfg.target_success_rate = s.num("Target Success Rate", 0.175);
    cfg.threshold_probability = s.num("Threshold Probability", 0.44);
    cfg.success_learning_rate = s.num("Success Learning Rate", 0.08);
    if (s.has("Termination Criteria")) {
      py::object tco = s.take("Termination Criteria");
      if (!py::isinstance<py::dict>(tco)) korali_error(" + Object: [ MOCMAES ] \n + Key:    ['Termination Criteria']\n + Reason: not an object\n");
      py::dict tcd;
      for (auto kv : py::reinterpret_borrow<py::dict>(tco)) tcd[kv.first] = kv.second;
      Settings tc(tcd, "MOCMAES['Termination Criteria']");
      tc_min_max_value_diff = tc.num("Min Max Value Difference Threshold", -INFINITY);   // parsed, but the criterion reads the base threshold
      tc_min_var_diff = tc.num("Min Variable Difference Threshold", -INFINITY);
      tc_min_sd = tc.num("Min Standard Deviation", -INFINITY);
      tc_max_sd = tc.num("Max Standard Deviation", INFINITY);
      tc_max_value = tc.num("Max Value", INFINITY);
      tc_min_value_diff = tc.num("Min Value Difference Threshold", -INFINITY);
      tc_max_model_evaluations = tc.num("Max Model Evaluations", 1e9);
      tc_max_generations = tc.num("Max Generations", 1e10);
      tc.finish();
    }
    for (const char* g : {"Multinormal Generator", "Uniform Generator", "Normal Generator"}) if (s.has(g)) s.take(g);
    const size_t n = py::len(variables);
    if (n == 0) korali_error("Optimization Evaluation problems require at least one variable.\n");
    lower.assign(n, -INFINITY); upper.assign(n, INFINITY); init_val.assign(n, NAN); init_sd.assign(n, NAN);
    for (size_t i = 0; i < n; i++) {
      if (!py::isinstance<py::dict>(variables[i])) korali_error("Variable %zu is not an object\n", i);
      py::dict vcopy;
      for (auto kv : py::reinterpret_borrow<py::dict>(variables[i])) vcopy[kv.first] = kv.second;
      Settings v(vcopy, "Variable");
      v.str("Name", "");
      lower[i] = v.num("Lower Bound", -INFINITY);
      upper[i] = v.num("Upper Bound", INFINITY);
      init_val[i] = v.num("Initial Value", NAN);
      init_sd[i] = v.num("Initial Standard Deviation", NAN);
      for (const char* k : {"Initial Mean", "Minimum Standard Deviation Update", "Granularity"}) v.num(k, NAN);
      if (v.has("Values")) v.take("Values");
      v.finish();
    }
    cfg.n = n; cfg.lower_bound = lower.data(); cfg.upper_bound = upper.data(); cfg.initial_value = init_val.data(); cfg.initial_stddev = init_sd.data();
    cfg.seed = seed;
    py::dict pcopy;
    for (auto kv : problem) pcopy[kv.first] = kv.second;
    Settings p(pcopy, "Optimization");
    const std::string ptype = canon(p.str("Type", ""));
    if (ptype != "optimization") korali_error("Korali problem incompatible with MO-CMAES, must be of type 'Optimization'.\n");
    if (!p.has("Objective Function")) korali_error(" + Object: [ Optimization ] \n + Key:    ['Objective Function']\n + Reason: mandatory setting missing\n");
    objective = p.take("Objective Function");
    cfg.num_objectives = p.uint("Num Objectives", 1);
    p.boolean("Has Discrete Variables", 0);
    if (p.has("Constraints")) {
      py::object c = p.take("Constraints");
      if (py::isinstance<py::list>(c) && py::len(c) > 0) korali_error("Optimizer/MOCMAES does not take constraints\n");
    }
    p.finish();
    if (py::isinstance<py::str>(objective)) {
      const std::string o = canon(objective.cast<std::string>());
      if (o == "negrosenbrockandsphere" || o == "rosenbrockandsphere") cfg.objective = KMOCMA_OBJ_NEG_ROSENBROCK_AND_SPHERE;
      else if (o == "negrosenbrockandtwospheres" || o == "rosenbrockandtwospheres") cfg.objective = KMOCMA_OBJ_NEG_ROSENBROCK_AND_TWO_SPHERES;
      else korali_error("Unknown multi-objective device model '%s' (RosenbrockAndSphere, RosenbrockAndTwoSpheres)\n", o.c_str());
    } else if (PyCallable_Check(objective.ptr())) {
      cfg.objective = KMOCMA_OBJ_EXTERNAL;
      batched = py::hasattr(objective, "_korali_batched") ? objective.attr("_korali_batched").cast<std::string>() : std::string();
      if (batched == "device") korali_error("Optimizer/MOCMAES takes per-sample models and korali.batched(fn) models (not device-tensor models)\n");
    } else {
      korali_error(" + Object: [ Optimization ] \n + Key:    ['Objective Function']\n + Reason: neither a callable nor the name of a device model\n");
    }
    s.finish();
  }

  // operation "Evaluate Multiple": sample["F(x)"] is a list of Num Objectives values (optimization.cpp.base)
  static void host_objective(void* user, const double* x, uint64_t rows, uint64_t n, double* f_out, uint64_t K) {
    MOCMAES* self = (MOCMAES*)user;
    try {
      if (self->batched == "numpy") {
        py::array_t<double> X({(py::ssize_t)rows, (py::ssize_t)n}, {(py::ssize_t)(n * sizeof(double)), (py::ssize_t)sizeof(double)}, x, py::none());
        py::array_t<double, py::array::c_style | py::array::forcecast> F(self->objective(X));
        if ((uint64_t)F.size() != rows * K) korali_error("The batched model returned %zu values for %zu samples x %zu objectives\n", (size_t)F.size(), (size_t)rows, (size_t)K);
        for (uint64_t i = 0; i < rows * K; i++) f_out[i] = F.data()[i];
        return;
      }
      for (uint64_t i = 0; i < rows; i++) {
        py::dict sample;
        py::list params;
        for (uint64_t d = 0; d < n; d++) params.append(x[i * n + d]);
        sample["Parameters"] = params;
        sample["Sample Id"] = i;
        sample["Module"] = "Problem";
        sample["Operation"] = "Evaluate Multiple";
        self->objective(sample);
        if (!sample.contains("F(x)")) korali_error("The model did not set 'F(x)' for sample %zu\n", (size_t)i);
        py::object fx = sample["F(x)"];
        if (!(py::isinstance<py::list>(fx) || py::isinstance<py::tuple>(fx)) || (uint64_t)py::len(fx) != K)
          korali_error("Multi-objective model: 'F(x)' of sample %zu must be a list of %zu values ('Num Objectives')\n", (size_t)i, (size_t)K);
        uint64_t k = 0;
        for (auto v : fx) f_out[i * K + k++] = v.cast<double>();
      }
    } catch (const std::exception& e) {
      self->pending_error = e.what();
      for (uint64_t i = 0; i < rows * K; i++) f_out[i] = NAN;
    }
  }

  void initialize(const std::vector<int>& device_ids) override {
    if (device_ids.size() > 1) korali_error("Optimizer/MOCMAES runs on one device (k['Conduit']['Devices'] > 1 is built for Optimizer/CMAES)\n");
    cfg.device = device_ids[0];
    if (kmocma_create(&cfg, &h)) korali_error("%s", kmocma_last_error(nullptr));
    if (cfg.objective == KMOCMA_OBJ_EXTERNAL) check(kmocma_set_host_objective(h, &MOCMAES::host_objective, this));
    check(kmocma_set_scalar(h, "Termination Criteria/Min Value Difference Threshold", tc_min_value_diff));
    check(kmocma_set_scalar(h, "Termination Criteria/Min Variable Difference Threshold", tc_min_var_diff));
    check(kmocma_set_scalar(h, "Termination Criteria/Min Standard Deviation", tc_min_sd));
    check(kmocma_set_scalar(h, "Termination Criteria/Max Standard Deviation", tc_max_sd));
    check(kmocma_set_scalar(h, "Termination Criteria/Max Model Evaluations", tc_max_model_evaluations));
    check(kmocma_set_scalar(h, "Termination Criteria/Max Generations", tc_max_generations));
  }

  void restore(uint64_t generation) override {
    if (generation != 0) korali_error("Resuming an Optimizer/MOCMAES run from a result file is not built on the B200 path\n");
  }

  bool checkTermination() override {
    int fin = 0;
    const char* reason = "";
    check(kmocma_check_termination(h, &fin, &reason));
    if (fin) splitReasons(reason);
    return fin != 0;
  }

  void runGeneration() override {
    pending_error.clear();
    int rc;
    if (!needsPython()) { py::gil_scoped_release nogil; rc = kmocma_run_generation(h); }
    else rc = kmocma_run_generation(h);
    if (!pending_error.empty()) { std::string e = pending_error; pending_error.clear(); throw std::runtime_error(e); }
    check(rc);
  }
  bool needsPython() const override { return cfg.objective == KMOCMA_OBJ_EXTERNAL; }

  py::list rowsOf(const std::vector<double>& flat, size_t width) {
    py::list out;
    for (size_t i = 0; width && (i + 1) * width <= flat.size(); i++) out.append(std::vector<double>(flat.begin() + i * width, flat.begin() + (i + 1) * width));
    return out;
  }

  void printGeneration(const std::function<void(int, const char*)>& log) override {   // MOCMAES::printGenerationAfter :524-537
    char b[256];
    std::vector<double> cb = array("Current Best Values"), be = array("Best Ever Values"), mn = array("Current Min Standard Deviations"),
                        mx = array("Current Max Standard Deviations");
    log(NORMAL, "Current Function Values = (Max, Best):\n");
    for (size_t k = 0; k < cb.size(); k++) { snprintf(b, sizeof(b), "                              = (%+6.3e, %+6.3e)\n", cb[k], be[k]); log(NORMAL, b); }
    snprintf(b, sizeof(b), "Standard Devs:            Min = %+6.3e - Max = %+6.3e\n", *std::min_element(mn.begin(), mn.end()), *std::max_element(mx.begin(), mx.end())); log(NORMAL, b);
    snprintf(b, sizeof(b), "Non Dominated Samples:   Current = %zu - Overall = %zu\n", (size_t)scalar("Current Non Dominated Sample Count"), (size_t)scalar("Sample Collection Size")); log(NORMAL, b);
    snprintf(b, sizeof(b), "Number of Infeasible Samples: %zu\n", (size_t)scalar("Infeasible Sample Count")); log(DETAILED, b);
  }

  // MOCMAES::finalize :539-552
  bool finalize(py::dict results, const std::function<void(int, const char*)>& log) override {
    py::dict pareto;
    pareto["F(x)"] = rowsOf(array("Sample Value Collection"), cfg.num_objectives);
    pareto["Parameters"] = rowsOf(array("Sample Collection"), cfg.n);
    results["Pareto Optimal Samples"] = pareto;
    log(MINIMAL, "--------------------------------------------------------------------\n");
    log(MINIMAL, "Optimizer/MOCMAES finished correctly.\n");
    return true;
  }

  // generated getConfiguration: settings + the internal state under Korali's key names (MOCMAES.config "Internal Settings")
  void getConfiguration(py::dict js) override {
    js["Type"] = "Optimizer/MOCMAES";
    js["Population Size"] = (uint64_t)scalar("Population Size");
    js["Mu Value"] = (uint64_t)scalar("Mu Value");
    js["Evolution Path Adaption Strength"] = scalar("Evolution Path Adaption Strength");
    js["Covariance Learning Rate"] = scalar("Covariance Learning Rate");
    js["Target Success Rate"] = cfg.target_success_rate;
    js["Threshold Probability"] = cfg.threshold_probability;
    js["Success Learning Rate"] = cfg.success_learning_rate;
    py::dict tc;
    tc["Min Max Value Difference Threshold"] = tc_min_max_value_diff; tc["Min Variable Difference Threshold"] = tc_min_var_diff;
    tc["Min Standard Deviation"] = tc_min_sd; tc["Max Standard Deviation"] = tc_max_sd; tc["Max Value"] = tc_max_value;
    tc["Min Value Difference Threshold"] = tc_min_value_diff; tc["Max Model Evaluations"] = tc_max_model_evaluations;
    tc["Max Generations"] = tc_max_generations;
    js["Termination Criteria"] = tc;
    const size_t n = cfg.n, K = cfg.num_objectives;
    js["Num Objectives"] = K;
    js["Current Non Dominated Sample Count"] = (uint64_t)scalar("Current Non Dominated Sample Count");
    js["Infeasible Sample Count"] = (uint64_t)scalar("Infeasible Sample Count");
    js["Model Evaluation Count"] = (uint64_t)scalar("Model Evaluation Count");
    for (const char* k : {"Current Values", "Previous Values"}) js[k] = rowsOf(array(k), K);
    for (const char* k : {"Parent Sample Population", "Current Sample Population", "Previous Sample Population", "Parent Evolution Paths",
                          "Current Evolution Paths", "Best Ever Variables Vector", "Current Best Variables Vector", "Sample Collection"})
      js[k] = rowsOf(array(k), n);
    js["Sample Value Collection"] = rowsOf(array("Sample Value Collection"), K);
    for (const char* k : {"Parent Covariance Matrix", "Current Covariance Matrix"}) js[k] = rowsOf(array(k), n * n);
    for (const char* k : {"Parent Sigma", "Current Sigma", "Parent Success Probabilities", "Current Success Probabilities", "Best Ever Values",
                          "Current Best Values", "Current Best Value Differences", "Current Best Variable Differences",
                          "Current Min Standard Deviations", "Current Max Standard Deviations"})
      js[k] = array(k);
    std::vector<double> pi = array("Parent Index");
    js["Parent Index"] = std::vector<uint64_t>(pi.begin(), pi.end());
  }
};

// ---- the solver plug-in: Sampler/TMCMC on libkcma (include/ktmcmc.h) for Bayesian/Custom problems ---------------------------------
class TMCMC : public SolverBase {
 public:
  ktmcmc_t* h = nullptr;
  ktmcmc_cfg cfg;
  py::object distributions = py::none();   // the experiment's top-level "Distributions" (the priors)
  std::vector<int32_t> prior_type;
  std::vector<double> prior_a, prior_b;
  std::vector<uint64_t> burn_in;
  std::vector<std::string> prior_name;
  std::string batched;
  py::object model;
  double tc_target = 1.0, tc_max_generations = 1e10, tc_max_model_evaluations = 1e9;

  ~TMCMC() override { if (h) ktmcmc_destroy(h); }
  const char* name() const override { return "Sampler/TMCMC"; }
  size_t variableCount() const override { return cfg.n; }
  void check(int rc) { if (rc) korali_error("%s", ktmcmc_last_error(h)); }
  double scalar(const char* key) override { double v = NAN; check(ktmcmc_get_scalar(h, key, &v)); return v; }
  std::vector<double> array(const char* key) override {
    size_t n = 0;
    check(ktmcmc_get_array(h, key, nullptr, 0, &n));
    std::vector<double> v(n);
    if (n) check(ktmcmc_get_array(h, key, v.data(), n, &n));
    return v;
  }

  // generated TMCMC::setConfiguration (TMCMC.config) + Sampler:: + Solver:: (strict); priors from e["Distributions"]
  void setConfiguration(py::dict solver, py::list variables, py::dict problem, uint64_t seed) override {
    ktmcmc_cfg_defaults(&cfg);
    Settings s(solver, "TMCMC");
    s.take("Type");
    const std::string version = s.str("Version", "TMCMC");
    if (canon(version) == "mtmcmc") korali_error("Sampler/TMCMC: 'Version' mTMCMC is not built on the B200 path (only 'TMCMC')\n");
    if (canon(version) != "tmcmc") korali_error(" + Object: [ TMCMC ] \n + Key:    ['Version']\n + Reason: unknown version '%s' (TMCMC)\n", version.c_str());
    cfg.population_size = s.uint("Population Size", 0);
    cfg.max_chain_length = s.uint("Max Chain Length", 1);
    cfg.default_burn_in = s.uint("Default Burn In", 0);
    if (s.has("Per Generation Burn In")) {
      py::object b = s.take("Per Generation Burn In");
      if (!py::isinstance<py::list>(b)) korali_error(" + Object: [ TMCMC ] \n + Key:    ['Per Generation Burn In']\n + Reason: an array was expected\n");
      for (auto x : b) {
        if (!is_number(x) || x.cast<double>() < 0) korali_error(" + Object: [ TMCMC ] \n + Key:    ['Per Generation Burn In']\n + Reason: unsigned integers were expected\n");
        burn_in.push_back((uint64_t)x.cast<double>());
      }
    }
    cfg.target_cov = s.num("Target Coefficient Of Variation", 1.0);
    cfg.covariance_scaling = s.num("Covariance Scaling", 0.04);
    cfg.min_annealing_update = s.num("Min Annealing Exponent Update", 1e-5);
    cfg.max_annealing_update = s.num("Max Annealing Exponent Update", 1.0);
    if (s.has("Termination Criteria")) {
      py::object tco = s.take("Termination Criteria");
      if (!py::isinstance<py::dict>(tco)) korali_error(" + Object: [ TMCMC ] \n + Key:    ['Termination Criteria']\n + Reason: not an object\n");
      py::dict tcd;
      for (auto kv : py::reinterpret_borrow<py::dict>(tco)) tcd[kv.first] = kv.second;
      Settings tc(tcd, "TMCMC['Termination Criteria']");
      tc_target = tc.num("Target Annealing Exponent", 1.0);
      tc_max_generations = tc.num("Max Generations", 1e10);
      tc_max_model_evaluations = tc.num("Max Model Evaluations", 1e9);
      tc.finish();
    }
    for (const char* g : {"Multinormal Generator", "Uniform Generator", "Normal Generator"}) if (s.has(g)) s.take(g);
    // the state a result file carries (getConfiguration); a run from such a file stops in restore()
    for (const char* k : {"Annealing Exponent", "Previous Annealing Exponent", "Coefficient Of Variation", "LogEvidence", "Max Loglikelihood",
                          "Proposals Acceptance Rate", "Selection Acceptance Rate", "Chain Count", "Model Evaluation Count", "Current Generation",
                          "Covariance Matrix", "Mean Theta", "Sample Database", "Sample LogLikelihood Database", "Sample LogPrior Database"})
      if (s.has(k)) s.take(k);
    s.finish();
    if (cfg.population_size < 2) korali_error("Sampler/TMCMC: 'Population Size' must be set to at least 2\n");
    // problem (bayesian/custom.config)
    py::dict pcopy;
    for (auto kv : problem) pcopy[kv.first] = kv.second;
    Settings p(pcopy, "Bayesian/Custom");
    const std::string ptype = canon(p.str("Type", ""));
    if (ptype != "bayesian/custom") korali_error("Sampler/TMCMC: only Problem Type 'Bayesian/Custom' is served (got '%s')\n", ptype.c_str());
    if (!p.has("Likelihood Model")) korali_error(" + Object: [ Bayesian/Custom ] \n + Key:    ['Likelihood Model']\n + Reason: mandatory setting missing\n");
    model = p.take("Likelihood Model");
    p.finish();
    if (py::isinstance<py::str>(model)) {
      const std::string o = canon(model.cast<std::string>());
      if (o == "negsphere" || o == "sphere") cfg.loglik = KCMA_OBJ_NEG_SPHERE;
      else if (o == "negrosenbrock" || o == "rosenbrock") cfg.loglik = KCMA_OBJ_NEG_ROSENBROCK;
      else if (o == "negackley" || o == "ackley") cfg.loglik = KCMA_OBJ_NEG_ACKLEY;
      else if (o == "negellipsoid" || o == "ellipsoid") cfg.loglik = KCMA_OBJ_NEG_ELLIPSOID;
      else if (o == "negsumsq") cfg.loglik = KCMA_OBJ_NEG_SUMSQ;
      else if (o == "negspheresin2") cfg.loglik = KCMA_OBJ_NEG_SPHERE_SIN2;
      else korali_error("Unknown device likelihood model '%s' (Sphere, Rosenbrock, Ackley, Ellipsoid, NegSumSq, NegSphereSin2)\n", o.c_str());
    } else if (PyCallable_Check(model.ptr())) {
      cfg.loglik = KCMA_OBJ_EXTERNAL;
      batched = py::hasattr(model, "_korali_batched") ? model.attr("_korali_batched").cast<std::string>() : std::string();
      if (!batched.empty() && batched != "numpy" && batched != "device") korali_error("Unknown batched model flavour '%s'\n", batched.c_str());
    } else {
      korali_error(" + Object: [ Bayesian/Custom ] \n + Key:    ['Likelihood Model']\n + Reason: neither a callable nor the name of a device model\n");
    }
    // priors: e["Distributions"][k] = {"Name", "Type", parameters}
    std::vector<std::string> dname, dtype;
    std::vector<double> da, db;
    if (!distributions.is_none()) {
      if (!py::isinstance<py::list>(distributions)) korali_error(" + Object: [ Experiment ] \n + Key:    ['Distributions']\n + Reason: an array was expected\n");
      for (auto item : distributions) {
        if (!py::isinstance<py::dict>(item)) korali_error("Distributions: every entry must be an object\n");
        py::dict dcopy;
        for (auto kv : py::reinterpret_borrow<py::dict>(item)) dcopy[kv.first] = kv.second;
        Settings d(dcopy, "Distribution");
        const std::string nm = d.str("Name", ""), ty = d.str("Type", "");
        const std::string ct = canon(ty);
        double a = NAN, b = NAN;
        if (ct == "univariate/uniform") { a = d.num("Minimum", NAN); b = d.num("Maximum", NAN); dtype.push_back("uniform"); }
        else if (ct == "univariate/normal") { a = d.num("Mean", NAN); b = d.num("Standard Deviation", NAN); dtype.push_back("normal"); }
        else korali_error("Sampler/TMCMC: prior distribution type '%s' of '%s' is not built (Univariate/Uniform, Univariate/Normal)\n", ty.c_str(), nm.c_str());
        if (d.has("Random Seed")) d.take("Random Seed");
        d.finish();
        if (!std::isfinite(a) || !std::isfinite(b)) korali_error("Distribution '%s' (%s): its parameters must be set to finite numbers\n", nm.c_str(), ty.c_str());
        dname.push_back(nm); da.push_back(a); db.push_back(b);
      }
    }
    const size_t n = py::len(variables);
    if (n == 0) korali_error("Bayesian problems require at least one variable.\n");
    lower.assign(n, -INFINITY); upper.assign(n, INFINITY);
    prior_type.assign(n, 0); prior_a.assign(n, 0.0); prior_b.assign(n, 0.0); prior_name.assign(n, "");
    for (size_t i = 0; i < n; i++) {
      if (!py::isinstance<py::dict>(variables[i])) korali_error("Variable %zu is not an object\n", i);
      py::dict vcopy;
      for (auto kv : py::reinterpret_borrow<py::dict>(variables[i])) vcopy[kv.first] = kv.second;
      Settings v(vcopy, "Variable");
      const std::string vname = v.str("Name", "");
      if (!v.has("Prior Distribution")) korali_error("Variable %zu ('%s') has no 'Prior Distribution'\n", i, vname.c_str());
      const std::string pd = v.str("Prior Distribution", "");
      v.num("Lower Bound", -INFINITY); v.num("Upper Bound", INFINITY);   // written back by getConfiguration
      v.finish();
      size_t k = 0;
      while (k < dname.size() && dname[k] != pd) k++;
      if (k == dname.size()) korali_error("Variable %zu ('%s'): prior distribution '%s' is not defined in e['Distributions']\n", i, vname.c_str(), pd.c_str());
      prior_name[i] = pd;
      prior_type[i] = dtype[k] == "uniform" ? KTMCMC_PRIOR_UNIFORM : KTMCMC_PRIOR_NORMAL;
      prior_a[i] = da[k]; prior_b[i] = db[k];
      if (prior_type[i] == KTMCMC_PRIOR_UNIFORM) { lower[i] = da[k]; upper[i] = db[k]; }
    }
    cfg.n = n; cfg.seed = seed;
    cfg.prior_type = prior_type.data(); cfg.prior_a = prior_a.data(); cfg.prior_b = prior_b.data();
    cfg.per_generation_burn_in = burn_in.empty() ? nullptr : burn_in.data(); cfg.burn_in_count = burn_in.size();
  }

  // Bayesian/Custom "Evaluate": the model sets sample["logLikelihood"]
  static void host_loglik(void* user, const double* x, uint64_t rows, uint64_t n, double* l_out) {
    TMCMC* self = (TMCMC*)user;
    try {
      if (self->batched == "numpy") {
        py::array_t<double> X({(py::ssize_t)rows, (py::ssize_t)n}, {(py::ssize_t)(n * sizeof(double)), (py::ssize_t)sizeof(double)}, x, py::none());
        py::array_t<double, py::array::c_style | py::array::forcecast> F(self->model(X));
        if ((uint64_t)F.size() != rows) korali_error("The batched model returned %zu values for %zu samples\n", (size_t)F.size(), (size_t)rows);
        for (uint64_t i = 0; i < rows; i++) l_out[i] = F.data()[i];
        return;
      }
      for (uint64_t i = 0; i < rows; i++) {
        py::dict sample;
        py::list params;
        for (uint64_t d = 0; d < n; d++) params.append(x[i * n + d]);
        sample["Parameters"] = params;
        sample["Sample Id"] = i;
        sample["Module"] = "Problem";
        sample["Operation"] = "Evaluate";
        self->model(sample);
        if (!sample.contains("logLikelihood")) korali_error("The model did not set 'logLikelihood' for sample %zu\n", (size_t)i);
        l_out[i] = sample["logLikelihood"].cast<double>();
      }
    } catch (const std::exception& e) {
      self->pending_error = e.what();
      for (uint64_t i = 0; i < rows; i++) l_out[i] = 0.0;
    }
  }
  static void device_loglik(void* user, const double* x_dev, uint64_t rows, uint64_t n, uint64_t ldx, double* f_dev, void* stream) {
    TMCMC* self = (TMCMC*)user;
    try {
      self->model((uintptr_t)x_dev, rows, n, ldx, (uintptr_t)f_dev, (uintptr_t)stream);
    } catch (const std::exception& e) {
      self->pending_error = e.what();
    }
  }

  void initialize(const std::vector<int>& device_ids) override {
    if (device_ids.size() > 1) korali_error("Sampler/TMCMC runs on one device (k['Conduit']['Devices'] > 1 is built for Optimizer/CMAES)\n");
    cfg.device = device_ids[0];
    if (ktmcmc_create(&cfg, &h)) korali_error("%s", ktmcmc_last_error(nullptr));
    if (cfg.loglik == KCMA_OBJ_EXTERNAL) {
      if (batched == "device") check(ktmcmc_set_device_loglik(h, &TMCMC::device_loglik, this));
      else check(ktmcmc_set_host_loglik(h, &TMCMC::host_loglik, this));
    }
    check(ktmcmc_set_scalar(h, "Termination Criteria/Target Annealing Exponent", tc_target));
    check(ktmcmc_set_scalar(h, "Termination Criteria/Max Generations", tc_max_generations));
    check(ktmcmc_set_scalar(h, "Termination Criteria/Max Model Evaluations", tc_max_model_evaluations));
  }

  void restore(uint64_t generation) override {
    if (generation != 0) korali_error("Resuming a Sampler/TMCMC run from a result file is not built on the B200 path\n");
  }

  bool checkTermination() override {
    int fin = 0;
    const char* reason = "";
    check(ktmcmc_check_termination(h, &fin, &reason));
    if (fin) splitReasons(reason);
    return fin != 0;
  }

  void runGeneration() override {
    pending_error.clear();
    int rc;
    if (!needsPython()) { py::gil_scoped_release nogil; rc = ktmcmc_run_generation(h); }
    else rc = ktmcmc_run_generation(h);
    if (!pending_error.empty()) { std::string e = pending_error; pending_error.clear(); throw std::runtime_error(e); }
    check(rc);
  }
  bool needsPython() const override { return cfg.loglik == KCMA_OBJ_EXTERNAL; }

  py::list rowsOf(const std::vector<double>& flat, size_t width) {
    py::list out;
    for (size_t i = 0; width && (i + 1) * width <= flat.size(); i++) out.append(std::vector<double>(flat.begin() + i * width, flat.begin() + (i + 1) * width));
    return out;
  }

  void printGeneration(const std::function<void(int, const char*)>& log) override {   // TMCMC::printGenerationAfter
    char b[256];
    snprintf(b, sizeof(b), "Acceptance Rate (proposals / selections): (%.2f%% / %.2f%%)\n", 100. * scalar("Proposals Acceptance Rate"),
             100. * scalar("Selection Acceptance Rate"));
    log(NORMAL, b);
    snprintf(b, sizeof(b), "Coefficient of Variation: %.2f%%\n", 100. * scalar("Coefficient Of Variation")); log(NORMAL, b);
    snprintf(b, sizeof(b), "Annealing Exponent:  %.3e.\n", scalar("Annealing Exponent")); log(NORMAL, b);
    snprintf(b, sizeof(b), "Log Evidence: %.3e\n", scalar("LogEvidence")); log(DETAILED, b);
  }

  bool finalize(py::dict results, const std::function<void(int, const char*)>& log) override {
    results["Posterior Sample Database"] = rowsOf(array("Sample Database"), cfg.n);
    results["Posterior Sample LogLikelihood Database"] = array("Sample LogLikelihood Database");
    results["Posterior Sample LogPrior Database"] = array("Sample LogPrior Database");
    results["Log Evidence"] = scalar("LogEvidence");
    char b[128];
    log(MINIMAL, "--------------------------------------------------------------------\n");
    snprintf(b, sizeof(b), "Log Evidence: %.4e\n", scalar("LogEvidence")); log(MINIMAL, b);
    log(MINIMAL, "Sampler/TMCMC finished correctly.\n");
    return true;
  }

  void getConfiguration(py::dict js) override {
    js["Type"] = "Sampler/TMCMC";
    js["Version"] = "TMCMC";
    js["Population Size"] = cfg.population_size;
    js["Max Chain Length"] = cfg.max_chain_length;
    js["Default Burn In"] = cfg.default_burn_in;
    js["Per Generation Burn In"] = burn_in;
    js["Target Coefficient Of Variation"] = cfg.target_cov;
    js["Covariance Scaling"] = cfg.covariance_scaling;
    js["Min Annealing Exponent Update"] = cfg.min_annealing_update;
    js["Max Annealing Exponent Update"] = cfg.max_annealing_update;
    py::dict tc;
    tc["Target Annealing Exponent"] = tc_target; tc["Max Generations"] = tc_max_generations; tc["Max Model Evaluations"] = tc_max_model_evaluations;
    js["Termination Criteria"] = tc;
    for (const char* k : {"Annealing Exponent", "Previous Annealing Exponent", "Coefficient Of Variation", "LogEvidence", "Max Loglikelihood",
                          "Proposals Acceptance Rate", "Selection Acceptance Rate"})
      js[k] = scalar(k);
    for (const char* k : {"Chain Count", "Model Evaluation Count", "Current Generation"}) js[k] = (uint64_t)scalar(k);
    const size_t n = cfg.n;
    js["Covariance Matrix"] = rowsOf(array("Covariance Matrix"), n);
    js["Mean Theta"] = array("Mean Theta");
    js["Sample Database"] = rowsOf(array("Sample Database"), n);
    js["Sample LogLikelihood Database"] = array("Sample LogLikelihood Database");
    js["Sample LogPrior Database"] = array("Sample LogPrior Database");
  }
};

class Experiment : public KoraliJson {
 public:
  std::unique_ptr<SolverBase> solver;
  uint64_t current_generation = 0;
  uint64_t random_seed = 0;
  Verbosity verbosity = NORMAL;
  uint64_t console_frequency = 1;
  bool file_enabled = true;
  std::string file_path = "_korali_result";
  uint64_t file_frequency = 1;
  bool is_finished = false;

  void loadState(const std::string& path) {
    py::object json = py::module_::import("json");
    py::object fh = py::module_::import("builtins").attr("open")(path, "r");
    py::object loaded = json.attr("load")(fh);
    fh.attr("close")();
    if (!py::isinstance<py::dict>(loaded)) korali_error("Could not load a Korali state from %s\n", path.c_str());
    // functions cannot be serialised: keep the ones already set on this experiment
    py::dict d = py::reinterpret_borrow<py::dict>(loaded);
    if (_js.contains("Problem") && py::isinstance<py::dict>(_js["Problem"]) && d.contains("Problem")) {
      py::dict oldp = py::reinterpret_borrow<py::dict>(_js["Problem"]), newp = py::reinterpret_borrow<py::dict>(d["Problem"]);
      for (const char* k : {"Objective Function", "Constraints"}) if (oldp.contains(k)) newp[k] = oldp[k];
    }
    if (d.contains("Solver") && py::isinstance<py::dict>(d["Solver"])) {   // .npy side-cars of large N x N arrays (saveState)
      py::dict sj = py::reinterpret_borrow<py::dict>(d["Solver"]);
      py::object os = py::module_::import("os"), np = py::module_::import("numpy");
      const std::string dir = os.attr("path").attr("dirname")(os.attr("path").attr("realpath")(path)).cast<std::string>();
      for (const char* key : {"Covariance Matrix", "Covariance Eigenvector Matrix"}) {
        const std::string fk = std::string(key) + " File";
        if (!sj.contains(fk.c_str())) continue;
        const std::string fname = sj[fk.c_str()].cast<std::string>();
        sj[key] = np.attr("load")(dir + "/" + fname).attr("ravel")().attr("tolist")();
        PyDict_DelItemString(sj.ptr(), fk.c_str());
      }
    }
    _js.clear();
    for (auto kv : d) _js[kv.first] = kv.second;
    reset();
  }

  void log(Verbosity level, const char* fmt, ...) const {
    if (verbosity < level) return;
    va_list ap;
    va_start(ap, fmt);
    printf("[Korali] ");
    vprintf(fmt, ap);
    va_end(ap);
  }

  // Experiment::initialize (experiment.cpp.base:165-206): defaults, seed, setConfiguration (strict), solver creation
  void initialize(const std::vector<int>& devices) {
    reset();
    py::dict js;
    for (auto kv : _js) js[kv.first] = kv.second;   // shallow copy: consumed keys are erased from the copy
    Settings top(js, "Experiment");
    if (!top.has("Solver") || !py::isinstance<py::dict>(js["Solver"])) korali_error(" + Object: [ Experiment ] \n + Key:    ['Solver']\n + Reason: mandatory setting missing\n");
    if (!top.has("Problem") || !py::isinstance<py::dict>(js["Problem"])) korali_error(" + Object: [ Experiment ] \n + Key:    ['Problem']\n + Reason: mandatory setting missing\n");
    if (!top.has("Variables") || !py::isinstance<py::list>(js["Variables"])) korali_error(" + Object: [ Experiment ] \n + Key:    ['Variables']\n + Reason: mandatory setting missing\n");
    py::dict solver_js;
    for (auto kv : py::reinterpret_borrow<py::dict>(top.take("Solver"))) solver_js[kv.first] = kv.second;
    py::dict problem_js = py::reinterpret_borrow<py::dict>(top.take("Problem"));
    py::list variables = py::reinterpret_borrow<py::list>(top.take("Variables"));
    const std::string stype = canon(solver_js.contains("Type") && py::isinstance<py::str>(solver_js["Type"]) ? solver_js["Type"].cast<std::string>() : "");
    const bool tmcmc = stype == "sampler/tmcmc" || stype == "tmcmc";
    if (stype != "optimizer/cmaes" && stype != "cmaes" && stype != "optimizer/dea" && stype != "dea" && stype != "optimizer/mocmaes" && stype != "mocmaes" && !tmcmc)
      korali_error("Solver Type '%s' is not served by korali_b200: only 'Optimizer/CMAES', 'Optimizer/DEA', 'Optimizer/MOCMAES' and 'Sampler/TMCMC' are built (SURVEY.md scope)\n", stype.c_str());
    random_seed = top.uint("Random Seed", 0);
    if (random_seed == 0) random_seed = (uint64_t)std::chrono::system_clock::now().time_since_epoch().count();  // experiment.cpp.base:235-251
    top.boolean("Preserve Random Number Generator States", 0);
    top.boolean("Store Sample Information", 0);
    current_generation = top.uint("Current Generation", 0);
    py::object distributions = py::none();   // the priors of Sampler/TMCMC; the optimizers ignore the key
    if (tmcmc && top.has("Distributions")) distributions = top.take("Distributions");
    for (const char* k : {"Distributions", "Results", "Samples", "Globals", "Run ID", "Timestamp", "Type", "Is Finished"}) if (top.has(k)) top.take(k);
    if (top.has("Console Output")) {
      py::object co = top.take("Console Output");
      if (!py::isinstance<py::dict>(co)) korali_error("'Console Output' is not an object\n");
      py::dict cd;
      for (auto kv : py::reinterpret_borrow<py::dict>(co)) cd[kv.first] = kv.second;
      Settings c(cd, "Experiment['Console Output']");
      const std::string v = c.str("Verbosity", "Normal");
      if (v == "Silent") verbosity = SILENT; else if (v == "Minimal") verbosity = MINIMAL; else if (v == "Normal") verbosity = NORMAL;
      else if (v == "Detailed") verbosity = DETAILED; else korali_error("Unknown Console Output Verbosity '%s'\n", v.c_str());
      console_frequency = c.uint("Frequency", 1);
      c.finish();
    }
    if (top.has("File Output")) {
      py::object fo = top.take("File Output");
      if (!py::isinstance<py::dict>(fo)) korali_error("'File Output' is not an object\n");
      py::dict fd;
      for (auto kv : py::reinterpret_borrow<py::dict>(fo)) fd[kv.first] = kv.second;
      Settings f(fd, "Experiment['File Output']");
      file_enabled = f.boolean("Enabled", 1);
      file_path = f.str("Path", "_korali_result");
      file_frequency = f.uint("Frequency", 1);
      f.boolean("Use Multiple Files", 1);
      if (f.has("Excluded Keys")) f.take("Excluded Keys");
      f.str("Name", "");
      f.finish();
    }
    top.finish();
    if (stype == "optimizer/dea" || stype == "dea") solver = std::make_unique<DEA>();
    else if (stype == "optimizer/mocmaes" || stype == "mocmaes") solver = std::make_unique<MOCMAES>();
    else if (tmcmc) { auto t = std::make_unique<TMCMC>(); t->distributions = distributions; solver = std::move(t); }
    else solver = std::make_unique<CMAES>();
    solver->setConfiguration(solver_js, variables, problem_js, random_seed);   // Normal Generator gets seed S (distribution.cpp.base:36-37)
    solver->initialize(devices);
    solver->restore(current_generation);
    is_finished = false;
  }

  void getConfiguration() {
    py::dict sj;
    solver->getConfiguration(sj);
    _js["Solver"] = sj;
    _js["Current Generation"] = current_generation;
    _js["Random Seed"] = random_seed + 2;   // Normal S, Uniform S+1, counter ends at S+2 (fixture: 790510 -> 790512)
    _js["Is Finished"] = is_finished ? 1 : 0;
    py::list vars = py::reinterpret_borrow<py::list>(_js["Variables"]);
    for (size_t i = 0; i < py::len(vars); i++) {
      py::dict v = py::reinterpret_borrow<py::dict>(vars[i]);
      v["Lower Bound"] = solver->lower[i]; v["Upper Bound"] = solver->upper[i];
    }
  }

  // saveState (experiment.cpp.base:120-148): <Path>/gen%08lu.json written atomically + 'latest' link
  void saveState() {
    py::object os = py::module_::import("os"), json = py::module_::import("json");
    os.attr("makedirs")(file_path, py::arg("exist_ok") = true);
    char name[64];
    snprintf(name, sizeof(name), "gen%08lu.json", (unsigned long)current_generation);
    const std::string target = file_path + "/" + name, aux = target + ".aux";
    py::dict out;
    for (auto kv : _js) out[kv.first] = kv.second;
    if (out.contains("Problem")) {   // callables are not serialisable: the reference stores function indices
      py::dict p;
      for (auto kv : py::reinterpret_borrow<py::dict>(out["Problem"])) {
        if (PyCallable_Check(kv.second.ptr())) p[kv.first] = 0;
        else if (py::isinstance<py::list>(kv.second)) { py::list l; for (auto it : kv.second) l.append(PyCallable_Check(it.ptr()) ? py::object(py::int_(0)) : py::reinterpret_borrow<py::object>(it)); p[kv.first] = l; }
        else p[kv.first] = kv.second;
      }
      out["Problem"] = p;
    }
    // N x N arrays above 2^22 entries do not go through JSON (SURVEY 5.4: 134 MB of text per matrix at N = 4096): they are written
    // as .npy side-cars next to the result file, and the file names them so that loadState finds them again
    if (solver && !solver->sideCars().empty() && out.contains("Solver")) {
      py::object np = py::module_::import("numpy");
      py::dict sj;
      for (auto kv : py::reinterpret_borrow<py::dict>(out["Solver"])) sj[kv.first] = kv.second;
      const size_t n = solver->variableCount();
      for (auto& kf : solver->sideCars()) {
        std::vector<double> flat = solver->array(kf.first.c_str());
        std::string fname = std::string(name) + "." + kf.second + ".npy";
        py::array_t<double> arr({(py::ssize_t)n, (py::ssize_t)n}, flat.data());
        np.attr("save")(file_path + "/" + fname, arr);
        sj[(kf.first + " File").c_str()] = fname;
      }
      out["Solver"] = sj;
    }
    py::object fh = py::module_::import("builtins").attr("open")(aux, "w");
    json.attr("dump")(out, fh);
    fh.attr("close")();
    os.attr("replace")(aux, target);
    const std::string latest = file_path + "/latest";
    if (os.attr("path").attr("lexists")(latest).cast<bool>()) os.attr("remove")(latest);
    os.attr("link")(target, latest);
  }

  bool needsPython() const { return !solver || solver->needsPython(); }

  // Experiment::run (experiment.cpp.base:39-118)
  void run() {
    auto t0 = std::chrono::steady_clock::now();
    if (current_generation == 0 && file_enabled) { getConfiguration(); saveState(); }
    current_generation++;
    solver->termination_criteria.clear();
    while (!solver->checkTermination()) {
      const bool print = console_frequency > 0 && current_generation % console_frequency == 0;
      if (print) {
        log(MINIMAL, "--------------------------------------------------------------------\n");
        log(MINIMAL, "Current Generation: #%zu\n", (size_t)current_generation);
      }
      auto g0 = std::chrono::steady_clock::now();
      solver->runGeneration();
      auto g1 = std::chrono::steady_clock::now();
      if (print && verbosity >= NORMAL) {
        solver->printGeneration([this](int level, const char* line) { log((Verbosity)level, "%s", line); });
        log(DETAILED, "Experiment: 0 - Generation Time: %.3fs\n", std::chrono::duration<double>(g1 - g0).count());
      }
      if (verbosity >= DETAILED) {
        const std::string w = solver->takeWarnings();
        if (!w.empty()) fprintf(stderr, "[Korali] Warning: %s", w.c_str());
      }
      if (file_enabled && file_frequency > 0 && current_generation % file_frequency == 0) { getConfiguration(); saveState(); }
      current_generation++;
      if (PyErr_CheckSignals() != 0) throw py::error_already_set();   // "User requested break."
    }
    auto t1 = std::chrono::steady_clock::now();
    current_generation--;
    is_finished = true;
    // finalize (CMAES.cpp.base:994-1010)
    py::dict results;
    const bool own_finalize = solver->finalize(results, [this](int level, const char* line) { log((Verbosity)level, "%s", line); });
    if (!own_finalize) {
      py::dict best;
      best["F(x)"] = solver->scalar("Best Ever Value");
      best["Parameters"] = solver->array("Best Ever Variables");
      results["Best Sample"] = best;
    }
    _js["Results"] = results;
    if (!own_finalize) {
      log(MINIMAL, "Optimum found: %e\n", solver->scalar("Best Ever Value"));
      log(MINIMAL, "Number of Infeasible Samples: %zu\n", (size_t)solver->scalar("Infeasible Sample Count"));
    }
    getConfiguration();
    if (file_enabled) saveState();
    if (!own_finalize) {
      log(MINIMAL, "--------------------------------------------------------------------\n");
      log(MINIMAL, "%s finished correctly.\n", solver->name());
    }
    for (auto& c : solver->termination_criteria) log(NORMAL, "Termination Criterion Met: %s\n", c.c_str());
    log(NORMAL, "Final Generation: %lu\n", (unsigned long)current_generation);
    log(NORMAL, "Elapsed Time: %.3fs\n", std::chrono::duration<double>(t1 - t0).count());
    reset();
  }
};

// ---- Engine -------------------------------------------------------------------------------------------------------
class Engine : public KoraliJson {
 public:
  // k["Conduit"]: "Type" (Sequential / Concurrent / Distributed dispatch one JSON sample at a time in the reference,
  // conduit.cpp.base:29-88; here they all map onto the batched device conduit "Device", which evaluates the whole population in
  // one launch), "Device" (ordinal of the single GPU) or "Devices" (G, or a list of ordinals: the population is sharded over G
  // GPUs of this process — the reference selects its Distributed conduit the same way, purely from k["Conduit"]).
  std::vector<int> devices() {
    std::vector<int> dev{0};
    if (_js.contains("Conduit") && py::isinstance<py::dict>(_js["Conduit"])) {
      py::dict c = py::reinterpret_borrow<py::dict>(_js["Conduit"]);
      if (c.contains("Type")) {
        const std::string t = canon(c["Type"].cast<std::string>());
        if (t != "device" && t != "sequential" && t != "concurrent" && t != "distributed") korali_error("Unknown Conduit Type '%s'\n", t.c_str());
      }
      if (c.contains("Device")) dev[0] = c["Device"].cast<int>();
      if (c.contains("Devices")) {
        py::object d = c["Devices"];
        dev.clear();
        if (py::isinstance<py::list>(d) || py::isinstance<py::tuple>(d)) for (auto x : d) dev.push_back(x.cast<int>());
        else if (is_number(d)) for (int r = 0; r < d.cast<int>(); r++) dev.push_back(r);
        else korali_error(" + Object: [ Engine ] \n + Key:    ['Conduit']['Devices']\n + Reason: a device count or a list of device ordinals was expected\n");
        if (dev.empty()) korali_error("k['Conduit']['Devices'] names no device\n");
      }
    }
    return dev;
  }
  void run(Experiment& e) {
    reset();
    e.initialize(devices());
    e.run();
  }
  // k.run([e1, e2, ...]) (engine.cpp:98-111: the reference interleaves the experiments by coroutine switches on one core).
  // Here, with k["Conduit"]["Devices"] = G > 1 and device objectives, the experiments run CONCURRENTLY: experiment j on device
  // j mod G, one host thread per device, the GIL released while a generation is on the GPU (results are those of the separate
  // runs: an experiment never spans devices in this mode). Otherwise the experiments run one after the other.
  void runMany(std::vector<Experiment*> es) {
    const std::vector<int> dev = devices();
    const size_t G = dev.size();
    bool parallel = es.size() > 1 && G > 1;
    if (parallel) {
      for (size_t j = 0; j < es.size(); j++) es[j]->initialize({dev[j % G]});
      for (auto* e : es) parallel = parallel && !e->needsPython();
    }
    if (!parallel) {
      for (auto* e : es) { e->initialize(dev); }
      for (auto* e : es) e->run();
      return;
    }
    std::vector<std::string> errors(G);
    {
      py::gil_scoped_release nogil;
      std::vector<std::thread> workers;
      for (size_t g = 0; g < G; g++)
        workers.emplace_back([&, g]() {
          for (size_t j = g; j < es.size() && errors[g].empty(); j += G) {
            py::gil_scoped_acquire gil;
            try { es[j]->run(); }
            catch (py::error_already_set& ex) { errors[g] = ex.what(); }
            catch (std::exception& ex) { errors[g] = ex.what(); }
          }
        });
      for (auto& w : workers) w.join();
    }
    for (auto& e : errors) if (!e.empty()) throw std::runtime_error(e);
  }
};

}  // namespace

PYBIND11_MODULE(_host, m) {
  m.doc() = "korali_b200 host shim: Korali's Engine/Experiment surface for Optimizer/CMAES on libkcma.so";
  py::class_<KoraliJson>(m, "koraliJson")
      .def("__getitem__", &KoraliJson::getItem)
      .def("__setitem__", &KoraliJson::setItem);
  py::class_<Experiment, KoraliJson>(m, "Experiment")
      .def(py::init<>())
      .def("__getitem__", &Experiment::getItem)
      .def("__setitem__", &Experiment::setItem)
      .def("loadState", &Experiment::loadState);
  py::class_<Engine, KoraliJson>(m, "Engine")
      .def(py::init<>())
      .def("__getitem__", &Engine::getItem)
      .def("__setitem__", &Engine::setItem)
      .def("run", &Engine::run)
      .def("run", &Engine::runMany);
}
