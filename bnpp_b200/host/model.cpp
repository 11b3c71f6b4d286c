#include "model.hh"
#include "runtime.hh"
#include "../csrc/elim_order.hpp"

#include <cassert>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <iostream>

namespace bn {

namespace {

struct Stopwatch {
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    double ms() const { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
};

bool has(const std::unordered_set<const Variable*> &s, const Variable *v) { return s.find(v) != s.end(); }

}  // namespace

// ------------------------------------------------------------------------------------------
// Model
// ------------------------------------------------------------------------------------------
Model::Model(std::string name, std::vector<Variable*> &variables, std::vector<Factor*> &factors)
    : _name(name), _variables(variables), _factors(factors)
{
    // The model's tables become resident NOW: creating the CUDA context and uploading the CPTs is
    // loading, not inference -- the reference's `uptime` (steady_clock around each inference call,
    // code/model.cpp:57-64, 258-298) has no counterpart of either.
    gpu::ctx();
    for (const Factor *pf : _factors) pf->device_data();
}

// a Model owns its variables and factors (code/model.cpp:21-29)
Model::~Model()
{
    for (Factor *pf : _factors) delete pf;
    for (Variable *pv : _variables) delete pv;
}

// brute-force joint, what `mn` runs (code/model.cpp:31-49)
Factor Model::joint_distribution() const
{
    Factor f(1.0);
    for (const Factor *pf : _factors) f *= *pf;
    return f;
}

Factor Model::joint_distribution(const std::unordered_map<unsigned,unsigned> &evidence) const
{
    Factor f(1.0);
    for (const Factor *pf : _factors) f *= pf->conditioning(evidence);
    return f;
}

double Model::partition(const std::unordered_map<unsigned,unsigned> &evidence, std::unordered_map<std::string,bool> &options,
                        double &uptime) const
{
    Stopwatch sw;
    double p;
    if (options["variable-elimination"]) p = partition_ve(evidence, options);   // extension: the reference's mn has no VE flag
    else p = joint_distribution(evidence).partition();
    uptime = sw.ms();
    return p;
}

std::vector<const Factor*> Model::marginals(const std::unordered_map<unsigned,unsigned> &evidence,
                                            std::unordered_map<std::string,bool> &options, double &uptime) const
{
    Stopwatch sw;
    std::vector<const Factor*> marg;
    if (options["variable-elimination"]) {
        marg = marginals_ve(evidence, options);
    } else {
        Factor joint = joint_distribution(evidence).normalize();
        for (const Variable *pv : _variables) marg.push_back(new Factor(marginal(pv, joint)));
    }
    uptime = sw.ms();
    return marg;
}

// sum out every other variable, in id order (code/model.cpp:91-101)
Factor Model::marginal(const Variable *v, Factor &joint) const
{
    Factor f = joint;
    for (const Variable *pv : _variables)
        if (pv->id() != v->id()) f = f.sum_out(pv);
    return f;
}

// Bucket elimination of code/model.cpp:348-446 as ONE device plan.  `evidence` replaces the
// conditioned copies of code/model.cpp:283-286 by views of the resident tables.
Factor Model::eliminate(const std::vector<const Variable*> &variables, const std::vector<const Factor*> &factors,
                        const std::unordered_map<unsigned,unsigned> &evidence,
                        std::unordered_map<std::string,bool> &options) const
{
    // variables to eliminate, in the caller's order; observed ones have nothing left to sum
    // (the reference crashes on them when an ordering flag is set, SURVEY A.2 i)
    std::vector<unsigned> ids;
    for (const Variable *pv : variables)
        if (evidence.find(pv->id()) == evidence.end()) ids.push_back(pv->id());

    if (options["min-fill"] || options["weighted-min-fill"] || options["min-degree"]) {
        std::vector<std::vector<unsigned>> scopes;
        for (const Factor *pf : factors) {
            std::vector<unsigned> sc;
            for (uint32_t id : pf->domain().ids())
                if (evidence.find(id) == evidence.end()) sc.push_back(id);
            scopes.push_back(sc);
        }
        std::vector<unsigned> card;
        for (const Variable *pv : _variables) card.push_back(pv->size());
        bnpp::Heuristic h = bnpp::H_MIN_FILL;
        if (options["min-degree"]) h = bnpp::H_MIN_DEGREE;
        else if (options["weighted-min-fill"]) h = bnpp::H_WEIGHTED_MIN_FILL;
        unsigned width = 0;
        ids = bnpp::FastOrderer(scopes, card).ordering(ids, h, width);
        if (options["verbose"]) {
            // same (mis)label as the reference (code/model.cpp:371-379, SURVEY A.2 iii)
            std::cout << ">> Original elimination order (width = " << bnpp::InteractionGraph(scopes, card).order_width(ids) << ")" << std::endl << "  ";
            for (unsigned id : ids) std::cout << " " << id;
            std::cout << std::endl << std::endl;
        }
    }

    std::vector<bnpp_scope> scopes(factors.size());
    std::vector<const double*> tables(factors.size());
    for (size_t i = 0; i < factors.size(); ++i) {
        const Domain &d = factors[i]->domain();
        scopes[i].rank = (int32_t)d.width();
        scopes[i].var_id = d.ids().data();
        scopes[i].card = d.cards().data();
        tables[i] = factors[i]->device_data();
    }
    std::vector<uint32_t> obs_var, obs_val;
    for (const auto &e : evidence) {
        obs_var.push_back(e.first);
        obs_val.push_back(e.second);
    }
    bnpp_ctx *ctx = gpu::ctx();
    bnpp_ve_plan *plan = nullptr;
    gpu::check(bnpp_ve_plan_create(ctx, (int)factors.size(), scopes.data(), (int)obs_var.size(), obs_var.data(),
                                   (int)ids.size(), ids.data(), &plan), "bnpp_ve_plan_create");
    int32_t rank = 0;
    uint32_t rvar[BNPP_MAX_RANK], rcard[BNPP_MAX_RANK];
    gpu::check(bnpp_ve_plan_info(plan, &rank, rvar, rcard, nullptr, nullptr, nullptr, nullptr, nullptr), "bnpp_ve_plan_info");
    std::vector<const Variable*> sc;
    for (int i = 0; i < rank; ++i) sc.push_back(_variables.at(rvar[i]));
    Domain *dom = new Domain(sc);
    double *res = nullptr;
    gpu::check(bnpp_alloc(ctx, (uint64_t)dom->size() + 1, &res), "bnpp_alloc");
    gpu::check(bnpp_ve_plan_run(plan, tables.data(), obs_val.data(), res, res + dom->size()), "bnpp_ve_plan_run");
    bnpp_ve_plan_destroy(plan);
    return Factor::adopt(dom, res);
}

double Model::partition_ve(const std::unordered_map<unsigned,unsigned> &evidence, std::unordered_map<std::string,bool> &options) const
{
    std::vector<const Variable*> variables(_variables.begin(), _variables.end());
    std::vector<const Factor*> factors(_factors.begin(), _factors.end());
    Factor part = eliminate(variables, factors, evidence, options);
    assert(part[0] == part.partition());   // code/model.cpp:288
    return part.partition();
}

// BN::marginals, VE branch (code/model.cpp:320-339).  The reference runs one complete VE pass per
// variable; here all marginals come from ONE two-pass bucket-tree plan on the device
// (bnpp_mar_plan_create) -- the same tables up to rounding.  With -v and an ordering flag the
// reference prints the order of every pass, so that combination keeps the pass-per-variable form.
std::vector<const Factor*> Model::marginals_ve(const std::unordered_map<unsigned,unsigned> &evidence,
                                               std::unordered_map<std::string,bool> &options) const
{
    std::vector<const Factor*> factors(_factors.begin(), _factors.end());
    std::vector<const Factor*> marg;
    const bool heuristic = options["min-fill"] || options["weighted-min-fill"] || options["min-degree"];
    if (options["verbose"] && heuristic) {
        for (const Variable *pv : _variables) {
            std::vector<const Variable*> vars;
            for (const Variable *pv2 : _variables)
                if (pv2 != pv) vars.push_back(pv2);
            marg.push_back(new Factor(eliminate(vars, factors, evidence, options).normalize()));
        }
        return marg;
    }

    std::vector<unsigned> ids;
    for (const Variable *pv : _variables)
        if (evidence.find(pv->id()) == evidence.end()) ids.push_back(pv->id());
    std::vector<unsigned> card;
    for (const Variable *pv : _variables) card.push_back(pv->size());
    if (heuristic) {
        std::vector<std::vector<unsigned>> scopes;
        for (const Factor *pf : factors) {
            std::vector<unsigned> sc;
            for (uint32_t id : pf->domain().ids())
                if (evidence.find(id) == evidence.end()) sc.push_back(id);
            scopes.push_back(sc);
        }
        bnpp::Heuristic h = bnpp::H_MIN_FILL;
        if (options["min-degree"]) h = bnpp::H_MIN_DEGREE;
        else if (options["weighted-min-fill"]) h = bnpp::H_WEIGHTED_MIN_FILL;
        unsigned width = 0;
        ids = bnpp::FastOrderer(scopes, card).ordering(ids, h, width);
    }
    std::vector<bnpp_scope> scopes(factors.size());
    std::vector<const double*> tables(factors.size());
    for (size_t i = 0; i < factors.size(); ++i) {
        const Domain &d = factors[i]->domain();
        scopes[i].rank = (int32_t)d.width();
        scopes[i].var_id = d.ids().data();
        scopes[i].card = d.cards().data();
        tables[i] = factors[i]->device_data();
    }
    std::vector<uint32_t> obs_var, obs_val;
    for (const auto &e : evidence) {
        obs_var.push_back(e.first);
        obs_val.push_back(e.second);
    }
    bnpp_ctx *ctx = gpu::ctx();
    bnpp_ve_plan *plan = nullptr;
    const int nvars = (int)_variables.size();
    gpu::check(bnpp_mar_plan_create(ctx, nvars, card.data(), (int)factors.size(), scopes.data(), (int)obs_var.size(),
                                    obs_var.data(), (int)ids.size(), ids.data(), &plan), "bnpp_mar_plan_create");
    std::vector<uint32_t> off(nvars), size(nvars);
    uint64_t total = 0;
    gpu::check(bnpp_mar_plan_layout(plan, nvars, off.data(), size.data(), &total), "bnpp_mar_plan_layout");
    double *res = nullptr;
    gpu::check(bnpp_alloc(ctx, total + 1, &res), "bnpp_alloc");
    gpu::check(bnpp_ve_plan_run(plan, tables.data(), obs_val.data(), res, nullptr), "bnpp_ve_plan_run");
    std::vector<double> host(total + 1);
    gpu::check(bnpp_download(ctx, host.data(), res, total), "bnpp_download");
    bnpp_free(ctx, res);
    bnpp_ve_plan_destroy(plan);
    for (int v = 0; v < nvars; ++v) {
        if (size[v] == 1 && _variables[v]->size() != 1) {
            marg.push_back(new Factor(1.0));      // observed (or unmentioned) variable: the width-0 factor [1]
            continue;
        }
        std::vector<const Variable*> sc(1, _variables[v]);
        std::vector<double> values(host.begin() + off[v], host.begin() + off[v] + size[v]);
        marg.push_back(new Factor(new Domain(sc), values, 1.0));
    }
    return marg;
}

double Model::mpe(const std::unordered_map<unsigned,unsigned> &evidence, std::unordered_map<std::string,bool> &options,
                  std::vector<unsigned> &assignment, double &uptime) const
{
    Stopwatch sw;
    std::vector<const Factor*> factors(_factors.begin(), _factors.end());
    std::vector<unsigned> ids, card;
    for (const Variable *pv : _variables)
        if (evidence.find(pv->id()) == evidence.end()) ids.push_back(pv->id());
    for (const Variable *pv : _variables) card.push_back(pv->size());
    if (options["min-fill"] || options["weighted-min-fill"] || options["min-degree"]) {
        std::vector<std::vector<unsigned>> scopes;
        for (const Factor *pf : factors) {
            std::vector<unsigned> sc;
            for (uint32_t id : pf->domain().ids())
                if (evidence.find(id) == evidence.end()) sc.push_back(id);
            scopes.push_back(sc);
        }
        bnpp::Heuristic h = bnpp::H_MIN_FILL;
        if (options["min-degree"]) h = bnpp::H_MIN_DEGREE;
        else if (options["weighted-min-fill"]) h = bnpp::H_WEIGHTED_MIN_FILL;
        unsigned width = 0;
        ids = bnpp::FastOrderer(scopes, card).ordering(ids, h, width);
    }
    std::vector<bnpp_scope> scopes(factors.size());
    std::vector<const double*> tables(factors.size());
    for (size_t i = 0; i < factors.size(); ++i) {
        const Domain &d = factors[i]->domain();
        scopes[i].rank = (int32_t)d.width();
        scopes[i].var_id = d.ids().data();
        scopes[i].card = d.cards().data();
        tables[i] = factors[i]->device_data();
    }
    std::vector<uint32_t> obs_var, obs_val;
    for (const auto &e : evidence) {
        obs_var.push_back(e.first);
        obs_val.push_back(e.second);
    }
    bnpp_ctx *ctx = gpu::ctx();
    bnpp_ve_plan *plan = nullptr;
    const int nvars = (int)_variables.size();
    gpu::check(bnpp_mpe_plan_create(ctx, nvars, card.data(), (int)factors.size(), scopes.data(), (int)obs_var.size(),
                                    obs_var.data(), (int)ids.size(), ids.data(), &plan), "bnpp_mpe_plan_create");
    // [value, assignment as uint32 words]: one buffer, one download
    double *res = nullptr;
    gpu::check(bnpp_alloc(ctx, 1 + ((uint64_t)nvars + 1) / 2, &res), "bnpp_alloc");
    gpu::check(bnpp_mpe_plan_run(plan, tables.data(), obs_val.data(), res, reinterpret_cast<uint32_t *>(res + 1)), "bnpp_mpe_plan_run");
    std::vector<double> host(1 + ((size_t)nvars + 1) / 2);
    gpu::check(bnpp_download(ctx, host.data(), res, host.size()), "bnpp_download");
    bnpp_free(ctx, res);
    bnpp_ve_plan_destroy(plan);
    assignment.assign(nvars, 0);
    std::memcpy(assignment.data(), host.data() + 1, sizeof(unsigned) * nvars);
    uptime = sw.ms();
    return host[0];
}

double Model::map(const std::vector<unsigned> &map_vars, const std::unordered_map<unsigned,unsigned> &evidence,
                  std::unordered_map<std::string,bool> &options, std::vector<unsigned> &assignment, double &uptime) const
{
    Stopwatch sw;
    std::vector<const Factor*> factors(_factors.begin(), _factors.end());
    const int nvars = (int)_variables.size();
    std::vector<unsigned> card;
    for (const Variable *pv : _variables) card.push_back(pv->size());
    std::vector<char> in_map(nvars, 0);
    for (unsigned v : map_vars)
        if (v < (unsigned)nvars) in_map[v] = 1;
    std::vector<unsigned> summed, last;
    for (const Variable *pv : _variables) {
        const unsigned id = pv->id();
        if (evidence.find(id) != evidence.end()) continue;
        if (!in_map[id]) summed.push_back(id);
    }
    for (unsigned v : map_vars)
        if (evidence.find(v) == evidence.end()) last.push_back(v);
    std::sort(last.begin(), last.end());
    std::vector<bnpp_scope> scopes(factors.size());
    std::vector<const double*> tables(factors.size());
    for (size_t i = 0; i < factors.size(); ++i) {
        const Domain &d = factors[i]->domain();
        scopes[i].rank = (int32_t)d.width();
        scopes[i].var_id = d.ids().data();
        scopes[i].card = d.cards().data();
        tables[i] = factors[i]->device_data();
    }
    std::vector<uint32_t> obs_var, obs_val;
    for (const auto &e : evidence) {
        obs_var.push_back(e.first);
        obs_val.push_back(e.second);
    }
    std::vector<uint32_t> ids(summed.begin(), summed.end());
    ids.insert(ids.end(), last.begin(), last.end());
    if (options["min-fill"] || options["weighted-min-fill"] || options["min-degree"]) {
        int h = 0;
        if (options["min-degree"]) h = 2;
        else if (options["weighted-min-fill"]) h = 1;
        uint32_t n = 0, width = 0;
        gpu::check(bnpp_elim_order_constrained(nvars, card.data(), (int)factors.size(), scopes.data(), (int)obs_var.size(),
                                               obs_var.data(), (int)summed.size(), summed.data(), (int)last.size(), last.data(),
                                               h, ids.data(), &n, &width), "bnpp_elim_order_constrained");
        ids.resize(n);
    }
    std::vector<uint32_t> mv(map_vars.begin(), map_vars.end());
    bnpp_ctx *ctx = gpu::ctx();
    bnpp_ve_plan *plan = nullptr;
    gpu::check(bnpp_map_plan_create(ctx, nvars, card.data(), (int)factors.size(), scopes.data(), (int)obs_var.size(),
                                    obs_var.data(), (int)mv.size(), mv.data(), (int)ids.size(), ids.data(), &plan),
               "bnpp_map_plan_create");
    // [value, assignment as uint32 words]: one buffer, one download
    double *res = nullptr;
    gpu::check(bnpp_alloc(ctx, 1 + ((uint64_t)nvars + 1) / 2, &res), "bnpp_alloc");
    gpu::check(bnpp_mpe_plan_run(plan, tables.data(), obs_val.data(), res, reinterpret_cast<uint32_t *>(res + 1)), "bnpp_mpe_plan_run");
    std::vector<double> host(1 + ((size_t)nvars + 1) / 2);
    gpu::check(bnpp_download(ctx, host.data(), res, host.size()), "bnpp_download");
    bnpp_free(ctx, res);
    bnpp_ve_plan_destroy(plan);
    assignment.assign(nvars, 0);
    std::memcpy(assignment.data(), host.data() + 1, sizeof(unsigned) * nvars);
    uptime = sw.ms();
    return host[0];
}

// ------------------------------------------------------------------------------------------
// BN
// ------------------------------------------------------------------------------------------
// factor i is the CPT of variable i with scope (child, parents...) -- code/model.cpp:104-120, SURVEY A.6
BN::BN(std::string name, std::vector<Variable*> &variables, std::vector<Factor*> &factors) : Model(name, variables, factors)
{
    for (const Variable *pv : _variables) {
        _children[pv];
        _parents[pv];
    }
    for (size_t i = 0; i < _variables.size() && i < _factors.size(); ++i) {
        const Variable *child = _variables[i];
        const std::vector<const Variable*> scope = _factors[i]->domain().scope();
        for (size_t j = 1; j < scope.size(); ++j) {
            _parents[child].insert(scope[j]);
            _children[scope[j]].insert(child);
        }
    }
}

const std::vector<const Variable*> BN::roots() const
{
    std::vector<const Variable*> r;
    for (const Variable *pv : _variables)
        if (_parents.find(pv)->second.empty()) r.push_back(pv);
    return r;
}

const std::vector<const Variable*> BN::leaves() const
{
    std::vector<const Variable*> r;
    for (const Variable *pv : _variables)
        if (_children.find(pv)->second.empty()) r.push_back(pv);
    return r;
}

double BN::partition(const std::unordered_map<unsigned,unsigned> &evidence, std::unordered_map<std::string,bool> &options,
                     double &uptime) const
{
    Stopwatch sw;
    double p = -1.0;
    if (options["logical-sampling"]) p = logical_sampling(evidence, 0.05, 0.05);
    else if (options["likelihood-weighting"]) p = likelihood_weighting(evidence, 0.05, 0.05);
    else if (options["gibbs-sampling"]) p = gibbs_sampling(evidence, 100000, 10000);
    else p = partition_ve(evidence, options);     // variable elimination by default (code/model.cpp:275-294)
    uptime = sw.ms();
    return p;
}

std::vector<const Factor*> BN::marginals(const std::unordered_map<unsigned,unsigned> &evidence,
                                         std::unordered_map<std::string,bool> &options, double &uptime) const
{
    Stopwatch sw;
    std::vector<const Factor*> marg;
    if (options["sum-product"]) {
        FactorGraph g = sum_product();            // evidence is ignored here, as in the reference (SURVEY A.2 ii)
        for (const Variable *pv : _variables) marg.push_back(new Factor(g.marginal(pv)));
    } else {
        marg = marginals_ve(evidence, options);
    }
    uptime = sw.ms();
    return marg;
}

// joint, then sum out (code/model.cpp:147-202)
Factor BN::query(const std::unordered_set<const Variable*> &target, const std::unordered_set<const Variable*> &evidence,
                 std::unordered_map<std::string,bool> &options, double &uptime) const
{
    Stopwatch sw;
    Factor joint(1.0);
    if (options["bayes-ball"]) {
        std::unordered_set<const Variable*> Np, Ne, F;
        bayes_ball(target, evidence, F, Np, Ne);
        for (const Variable *pv : Np) joint *= *_factors[pv->id()];
        if (options["verbose"]) {
            std::cout << ">> Requisite probability nodes Np:" << std::endl;
            for (const Variable *pv : Np) std::cout << *pv << std::endl;
            std::cout << std::endl << ">> Requisite observation nodes Ne" << std::endl;
            for (const Variable *pv : Ne) std::cout << *pv << std::endl;
            std::cout << std::endl;
        }
    } else {
        joint = joint_distribution();
    }
    Factor f = joint;
    for (const Variable *pv : _variables)
        if (!has(target, pv) && !has(evidence, pv)) f = f.sum_out(pv);
    if (!evidence.empty()) {
        Factor g = f;
        for (const Variable *pv : target) g = g.sum_out(pv);
        f = f.divide(g);
    }
    uptime = sw.ms();
    return f;
}

// code/model.cpp:204-248: evidence is a set of VARIABLES here; the result is the conditional table
Factor BN::query_ve(const std::unordered_set<const Variable*> &target, const std::unordered_set<const Variable*> &evidence,
                    std::unordered_map<std::string,bool> &options, double &uptime) const
{
    Stopwatch sw;
    std::vector<const Variable*> variables;
    std::vector<const Factor*> factors;
    if (options["bayes-ball"]) {
        std::unordered_set<const Variable*> Np, Ne, F;
        bayes_ball(target, evidence, F, Np, Ne);
        // id order instead of the reference's pointer-hash order: same set, reproducible plan
        for (const Variable *pv : _variables) {
            if (!has(Np, pv)) continue;
            if (!has(target, pv) && !has(evidence, pv)) variables.push_back(pv);
            factors.push_back(_factors[pv->id()]);
        }
    } else {
        for (const Variable *pv : _variables) {
            if (!has(target, pv) && !has(evidence, pv)) variables.push_back(pv);
            factors.push_back(_factors[pv->id()]);
        }
    }
    Factor f = variable_elimination(variables, factors, options);
    if (!evidence.empty()) {
        Factor g = f;
        for (const Variable *pv : target) g = g.sum_out(pv);
        f = f.divide(g);
    }
    uptime = sw.ms();
    return f;
}

Factor BN::variable_elimination(std::vector<const Variable*> &variables, std::vector<const Factor*> &factors,
                                std::unordered_map<std::string,bool> &options) const
{
    static const std::unordered_map<unsigned,unsigned> none;
    return eliminate(variables, factors, none, options);
}

// Bayes-ball (Shachter 1998) as used by code/model.cpp:448-537: Np = nodes whose top is
// marked, Ne = observed nodes that were visited.
void BN::bayes_ball(const std::unordered_set<const Variable*> &J, const std::unordered_set<const Variable*> &K,
                    const std::unordered_set<const Variable*> &F, std::unordered_set<const Variable*> &Np,
                    std::unordered_set<const Variable*> &Ne) const
{
    struct Visit { const Variable *node; bool from_child; };
    std::vector<Visit> todo;
    for (const Variable *j : J) todo.push_back({j, true});
    std::unordered_set<const Variable*> visited, top, bottom;
    while (!todo.empty()) {
        const Visit v = todo.back();
        todo.pop_back();
        visited.insert(v.node);
        const bool observed = has(K, v.node);
        bool to_parents = false, to_children = false;
        if (v.from_child) {
            if (!observed) {
                to_parents = true;
                to_children = !has(F, v.node);
            }
        } else {
            to_parents = observed;
            to_children = !observed;
        }
        if (to_parents && top.insert(v.node).second)
            for (const Variable *pa : _parents.at(v.node)) todo.push_back({pa, true});
        if (to_children && bottom.insert(v.node).second)
            for (const Variable *ch : _children.at(v.node)) todo.push_back({ch, false});
    }
    Np.insert(top.begin(), top.end());
    for (const Variable *pv : K)
        if (has(visited, pv)) Ne.insert(pv);
}

// m-separation in the moralised ancestral graph (code/model.cpp:755-835)
bool BN::m_separated(const Variable *v1, const Variable *v2, const std::unordered_set<const Variable*> evidence, bool verbose) const
{
    std::unordered_set<const Variable*> keep(evidence);
    keep.insert(v1);
    keep.insert(v2);
    std::unordered_set<const Variable*> nodes = ancestors(keep);
    nodes.insert(keep.begin(), keep.end());

    std::unordered_map<const Variable*, std::unordered_set<const Variable*>> g;
    for (const Variable *pv : nodes) g[pv];
    for (const Variable *pv : nodes) {
        const std::unordered_set<const Variable*> &pa = _parents.find(pv)->second;
        for (const Variable *p : pa) {
            g[pv].insert(p);
            g[p].insert(pv);
            for (const Variable *q : pa)       // marry the parents
                if (p != q) {
                    g[p].insert(q);
                    g[q].insert(p);
                }
        }
    }
    for (const Variable *e : evidence) {
        g.erase(e);
        for (auto &node : g) node.second.erase(e);
    }
    if (verbose) {
        std::cout << ">> Graph:" << std::endl;
        for (const auto &node : g) {
            std::cout << "variable id=" << node.first->id() << ", neighboors={ ";
            for (const Variable *pv : node.second) std::cout << pv->id() << " ";
            std::cout << "}" << std::endl;
        }
    }
    std::vector<const Variable*> stack(1, v1);
    std::unordered_set<const Variable*> seen;
    while (!stack.empty()) {
        const Variable *v = stack.back();
        stack.pop_back();
        if (v->id() == v2->id()) return false;
        if (!seen.insert(v).second) continue;
        auto it = g.find(v);
        if (it == g.end()) continue;
        for (const Variable *n : it->second)
            if (!has(seen, n)) stack.push_back(n);
    }
    return true;
}

std::unordered_set<const Variable*> BN::markov_blanket(const Variable *v) const
{
    std::unordered_set<const Variable*> mb = parents(v);
    for (const Variable *ch : children(v)) {
        mb.insert(ch);
        for (const Variable *co : parents(ch))
            if (co->id() != v->id()) mb.insert(co);
    }
    return mb;
}

std::unordered_set<const Variable*> BN::markov_independence(const Variable *v) const
{
    std::unordered_set<const Variable*> nd(_variables.begin(), _variables.end());
    nd.erase(v);
    for (const Variable *pv : _parents.find(v)->second) nd.erase(pv);
    for (const Variable *pv : descendants(v)) nd.erase(pv);
    return nd;
}

std::unordered_set<const Variable*> BN::descendants(const Variable *v) const
{
    std::unordered_set<const Variable*> out;
    std::vector<const Variable*> stack(1, v);
    while (!stack.empty()) {
        const Variable *u = stack.back();
        stack.pop_back();
        for (const Variable *ch : _children.find(u)->second)
            if (out.insert(ch).second) stack.push_back(ch);
    }
    return out;
}

std::unordered_set<const Variable*> BN::ancestors(const std::unordered_set<const Variable*> &vars) const
{
    std::unordered_set<const Variable*> out;
    std::vector<const Variable*> stack(vars.begin(), vars.end());
    while (!stack.empty()) {
        const Variable *u = stack.back();
        stack.pop_back();
        for (const Variable *pa : _parents.find(u)->second)
            if (out.insert(pa).second) stack.push_back(pa);
    }
    return out;
}

std::unordered_set<const Variable*> BN::ancestors(const Variable *v) const
{
    std::unordered_set<const Variable*> one;
    one.insert(v);
    return ancestors(one);
}

// BN::sum_product, code/model.cpp:736-753: 10 000 sweeps at most, epsilon 0.001
FactorGraph BN::sum_product(void) const
{
    std::vector<const Variable*> variables(_variables.begin(), _variables.end());
    std::vector<const Factor*> factors(_factors.begin(), _factors.end());
    FactorGraph g(variables, factors);
    g.update(10000, 0.001);
    return g;
}

// ---- stochastic inference (SURVEY 8f row 4): -ls / -lw draw their samples on the GPU; -gs (one sequential chain) stays on the host ----
std::vector<const Factor*> BN::topological_sampling_order() const
{
    std::vector<const Factor*> order;
    std::unordered_set<const Variable*> done;
    while (order.size() < _variables.size()) {
        const size_t before = order.size();
        for (const Variable *pv : _variables) {
            if (has(done, pv)) continue;
            bool ready = true;
            for (const Variable *pa : _parents.find(pv)->second) ready = ready && has(done, pa);
            if (ready) {
                order.push_back(_factors[pv->id()]);
                done.insert(pv);
            }
        }
        if (order.size() == before) break;   // cyclic input: give up rather than spin
    }
    return order;
}

std::unordered_map<unsigned,unsigned> BN::sampling() const
{
    std::unordered_map<unsigned,unsigned> valuation;
    for (const Factor *pf : topological_sampling_order())
        for (const auto &s : pf->sampling(valuation)) valuation[s.first] = s.second;
    return valuation;
}

// The sampler of the C ABI (csrc/sampling.cu): one GPU thread per sample over the resident CPTs.  The seed comes from
// BNPP_SEED (default 1): unlike the reference (std::random_device per draw) a run can be repeated.
namespace {
struct GpuSampler {
    bnpp_sampler *h = nullptr;
    std::vector<uint32_t> ev_var, ev_val;
    uint64_t seed = 1;
    GpuSampler(const BN &bn, const std::vector<Variable*> &variables, const std::vector<Factor*> &factors,
               const std::vector<const Factor*> &order, const std::unordered_map<unsigned,unsigned> &evidence)
    {
        const int n = (int)variables.size();
        std::vector<uint32_t> card(n), ord;
        std::vector<std::vector<uint32_t>> ids(n), cards(n);
        std::vector<bnpp_scope> scopes(n);
        std::vector<const double*> tables(n);
        for (int v = 0; v < n; ++v) {
            card[v] = variables[v]->size();
            const Domain &d = factors[v]->domain();
            for (unsigned i = 0; i < d.width(); ++i) {
                ids[v].push_back(d[i]->id());
                cards[v].push_back(d[i]->size());
            }
            scopes[v] = bnpp_scope{(int32_t)d.width(), ids[v].data(), cards[v].data()};
            tables[v] = factors[v]->device_data();
        }
        for (const Factor *pf : order) ord.push_back(pf->domain()[0]->id());
        gpu::check(bnpp_sampler_create(gpu::ctx(), n, card.data(), scopes.data(), ord.data(), tables.data(), &h), "bnpp_sampler_create");
        for (const auto &e : evidence) {
            ev_var.push_back(e.first);
            ev_val.push_back(e.second);
        }
        if (const char *s = std::getenv("BNPP_SEED")) seed = std::strtoull(s, nullptr, 10);
        (void)bn;
    }
    ~GpuSampler() { bnpp_sampler_destroy(h); }
};
}  // namespace

// BN::logical_sampling, code/model.cpp:540-560
double BN::logical_sampling(const std::unordered_map<unsigned,unsigned> &evidence, double delta, double epsilon) const
{
    const unsigned long M = 3 * std::log(2 / delta) / std::pow(epsilon, 2) * 1 / 0.1;
    GpuSampler g(*this, _variables, _factors, topological_sampling_order(), evidence);
    uint64_t hits = 0;
    gpu::check(bnpp_sampler_logical(g.h, (int)g.ev_var.size(), g.ev_var.data(), g.ev_val.data(), M, g.seed, &hits), "bnpp_sampler_logical");
    return 1.0 * hits / M;
}

// BN::likelihood_weighting, code/model.cpp:620-690 (bounded-variance stopping rule)
double BN::likelihood_weighting(const std::unordered_map<unsigned,unsigned> &evidence, double delta, double epsilon) const
{
    double U = 1.0;
    for (const Factor *pf : _factors) U *= pf->max();
    const double Nstar = 4 * std::log(2 / delta) * (1 + epsilon) / std::pow(epsilon, 2);
    GpuSampler g(*this, _variables, _factors, topological_sampling_order(), evidence);
    double N = 0.0;
    uint64_t M = 0;
    gpu::check(bnpp_sampler_likelihood(g.h, (int)g.ev_var.size(), g.ev_var.data(), g.ev_val.data(), U, Nstar, 1u << 16, 1ull << 34, g.seed,
                                       &N, &M), "bnpp_sampler_likelihood");
    assert(N > 0.0);
    return U * N / M;
}

double BN::gibbs_sampling(const std::unordered_map<unsigned,unsigned> &evidence, long unsigned M, long unsigned burn_in) const
{
    std::vector<Factor*> blanket;
    for (const Factor *pf : _factors) {
        const Variable *X = pf->domain()[0];
        std::unordered_set<const Variable*> mb = markov_blanket(X);
        mb.insert(X);
        Factor joint(1.0);
        for (const Variable *pv : mb) {
            Factor f(*_factors.at(pv->id()));
            for (const Variable *pa : parents(pv))
                if (!has(mb, pa)) f = f.sum_out(pa);
            joint *= f;
        }
        blanket.push_back(new Factor(joint.divide(joint.sum_out(X))));
    }
    std::unordered_map<unsigned,unsigned> valuation;
    for (const Variable *pv : _variables) {
        auto e = evidence.find(pv->id());
        valuation[pv->id()] = e == evidence.end() ? 0 : e->second;
    }
    long unsigned hits = 0;
    for (long unsigned i = 0; i < M + burn_in; ++i) {
        for (const Factor *pf : blanket) {
            valuation.erase(pf->domain()[0]->id());
            for (const auto &s : pf->sampling(valuation)) valuation[s.first] = s.second;
        }
        if (i < burn_in) continue;
        bool ok = true;
        for (const auto &e : evidence) ok = ok && valuation.at(e.first) == e.second;
        hits += ok;
    }
    for (Factor *pf : blanket) delete pf;
    return 1.0 * hits / M;
}

// text of code/model.cpp:924-963
void BN::write(std::ostream &os) const
{
    os << "BAYES:" << std::endl << ">> Variables" << std::endl;
    for (const Variable *pv : _variables) {
        os << *pv << ", " << "parents:{";
        for (const Variable *p : _parents.find(pv)->second) os << " " << p->id();
        os << " }, " << "children:{";
        for (const Variable *c : _children.find(pv)->second) os << " " << c->id();
        os << " }" << std::endl;
    }
    os << std::endl << ">> Factors" << std::endl;
    for (const Factor *pf : _factors) os << *pf << std::endl;
}

std::ostream &operator<<(std::ostream &os, const BN &bn)
{
    bn.write(os);
    return os;
}

// ------------------------------------------------------------------------------------------
// MN
// ------------------------------------------------------------------------------------------
MN::MN(std::string name, std::vector<Variable*> &variables, std::vector<Factor*> &factors) : Model(name, variables, factors)
{
    for (const Variable *pv : _variables) _neighbors[pv];
    for (const Factor *pf : _factors) {
        const std::vector<const Variable*> scope = pf->domain().scope();
        for (const Variable *a : scope)
            for (const Variable *b : scope)
                if (a->id() != b->id()) _neighbors[a].insert(b);
    }
}

void MN::write(std::ostream &os) const
{
    os << "MARKOV:" << std::endl << ">> Variables" << std::endl;
    for (const Variable *pv : _variables) {
        os << *pv << ", " << "neighbors:{";
        for (const Variable *n : _neighbors.find(pv)->second) os << " " << n->id();
        os << " }" << std::endl;
    }
    os << std::endl << ">> Factors" << std::endl;
    for (const Factor *pf : _factors) os << *pf << std::endl;
}

std::ostream &operator<<(std::ostream &os, const MN &mn)
{
    mn.write(os);
    return os;
}

}  // namespace bn
