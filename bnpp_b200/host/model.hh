// bn::Model / bn::BN / bn::MN -- inference drivers.  Public API of reference
// code/model.hh:15-133.  The variable-elimination and sum-product loops run as device
// plans (include/bnpp_b200.h: bnpp_ve_plan_*, bnpp_fg_*); ordering heuristics, bayes-ball
// and the other graph queries stay on the host.
#ifndef BNPP_HOST_MODEL_HH
#define BNPP_HOST_MODEL_HH

#include "variable.hh"
#include "factor.hh"
#include "graph.hh"

#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

namespace bn {

class Model {
public:
    Model(std::string name, std::vector<Variable*> &variables, std::vector<Factor*> &factors);
    virtual ~Model();

    const std::string name() const { return _name; }
    const std::vector<Variable*> &variables() const { return _variables; }
    const std::vector<Factor*>   &factors()   const { return _factors;   }

    Factor joint_distribution() const;
    Factor joint_distribution(const std::unordered_map<unsigned,unsigned> &evidence) const;

    virtual double partition(
        const std::unordered_map<unsigned,unsigned> &evidence,
        std::unordered_map<std::string,bool> &options,
        double &uptime) const;

    virtual std::vector<const Factor*> marginals(
        const std::unordered_map<unsigned,unsigned> &evidence,
        std::unordered_map<std::string,bool> &options,
        double &uptime) const;

    virtual Factor marginal(const Variable *v, Factor &joint) const;

    virtual void write(std::ostream&) const = 0;

    // ---- device-resident variable elimination shared by BN and (as an extension) MN ----
    // VE over `factors` (any resident tables), eliminating `variables` in the given order
    // unless an ordering flag is set; `evidence` is applied as views, never materialised.
    Factor eliminate(
        const std::vector<const Variable*> &variables,
        const std::vector<const Factor*> &factors,
        const std::unordered_map<unsigned,unsigned> &evidence,
        std::unordered_map<std::string,bool> &options) const;
    // PR / MAR by variable elimination for ANY model kind (the reference reaches this for
    // Markov nets only through its library API, SURVEY §8c)
    double partition_ve(const std::unordered_map<unsigned,unsigned> &evidence, std::unordered_map<std::string,bool> &options) const;
    std::vector<const Factor*> marginals_ve(const std::unordered_map<unsigned,unsigned> &evidence, std::unordered_map<std::string,bool> &options) const;
    // MPE (no reference counterpart): the most probable assignment of the unobserved variables given the evidence
    // (assignment[id]; observed variables keep their evidence value) and its value max_x prod_f f(x, e), by
    // max-product variable elimination on the device.  The order follows the -mf / -wmf / -md flags as in
    // partition_ve, else variables in id order.  Ties go to the lowest values.
    double mpe(const std::unordered_map<unsigned,unsigned> &evidence, std::unordered_map<std::string,bool> &options,
               std::vector<unsigned> &assignment, double &uptime) const;
    // Marginal MAP (no reference counterpart): the jointly most probable assignment of the MAP variables `map_vars`
    // given the evidence, every other unobserved variable summed out, and its value max_{x_M} sum_{x_S} prod_f f(x, e)
    // (assignment[id]: MAP variables their decoded value, observed ones their evidence, summed ones BNPP_ASSIGN_SUMMED).
    // The order eliminates the summed variables first: with -mf / -wmf / -md the constrained heuristic order
    // (bnpp_elim_order_constrained), else each group in id order.  Ties go to the lowest values in decode order.
    double map(const std::vector<unsigned> &map_vars, const std::unordered_map<unsigned,unsigned> &evidence,
               std::unordered_map<std::string,bool> &options, std::vector<unsigned> &assignment, double &uptime) const;

protected:
    std::string _name;
    std::vector<Variable*> _variables;
    std::vector<Factor*> _factors;
};

class BN : public Model {
public:
    BN(std::string name, std::vector<Variable*> &variables, std::vector<Factor*> &factors);

    double partition(
        const std::unordered_map<unsigned,unsigned> &evidence,
        std::unordered_map<std::string,bool> &options,
        double &uptime) const;

    std::vector<const Factor*> marginals(
        const std::unordered_map<unsigned,unsigned> &evidence,
        std::unordered_map<std::string,bool> &options,
        double &uptime) const;

    Factor query(
        const std::unordered_set<const Variable*> &target,
        const std::unordered_set<const Variable*> &evidence,
        std::unordered_map<std::string,bool> &options,
        double &uptime) const;

    Factor query_ve(
        const std::unordered_set<const Variable*> &target,
        const std::unordered_set<const Variable*> &evidence,
        std::unordered_map<std::string,bool> &options,
        double &uptime) const;

    Factor variable_elimination(
        std::vector<const Variable*> &variables,
        std::vector<const Factor*> &factors,
        std::unordered_map<std::string,bool> &options) const;

    void bayes_ball(
        const std::unordered_set<const Variable*> &J,
        const std::unordered_set<const Variable*> &K,
        const std::unordered_set<const Variable*> &F,
        std::unordered_set<const Variable*> &Np,
        std::unordered_set<const Variable*> &Ne) const;

    bool m_separated(
        const Variable *v1, const Variable *v2,
        const std::unordered_set<const Variable*> evidence,
        bool verbose=false) const;

    double logical_sampling(const std::unordered_map<unsigned,unsigned> &evidence, double delta, double epsilon) const;
    double likelihood_weighting(const std::unordered_map<unsigned,unsigned> &evidence, double delta, double epsilon) const;
    double gibbs_sampling(const std::unordered_map<unsigned,unsigned> &evidence, long unsigned M, long unsigned burn_in) const;

    FactorGraph sum_product(void) const;

    const std::unordered_set<const Variable*> parents(const Variable *v)  const { return _parents.find(v)->second;  }
    const std::unordered_set<const Variable*> children(const Variable *v) const { return _children.find(v)->second; }

    const std::vector<const Variable*> roots()  const;
    const std::vector<const Variable*> leaves() const;

    std::unordered_set<const Variable*> markov_blanket(const Variable *v)      const;
    std::unordered_set<const Variable*> markov_independence(const Variable *v) const;

    std::unordered_set<const Variable*> descendants(const Variable *v) const;
    std::unordered_set<const Variable*> ancestors(const Variable *v) const;
    std::unordered_set<const Variable*> ancestors(const std::unordered_set<const Variable*> &vars) const;

    void write(std::ostream& os) const;
    friend std::ostream &operator<<(std::ostream &os, const BN &bn);

private:
    std::unordered_map<const Variable*,std::unordered_set<const Variable*>> _parents;
    std::unordered_map<const Variable*,std::unordered_set<const Variable*>> _children;

    std::vector<const Factor*> topological_sampling_order() const;
    std::unordered_map<unsigned,unsigned> sampling() const;
};

class MN : public Model {
public:
    MN(std::string name, std::vector<Variable*> &variables, std::vector<Factor*> &factors);

    const std::unordered_set<const Variable*> neighbors(const Variable *v) const { return _neighbors.find(v)->second; }

    void write(std::ostream& os) const;
    friend std::ostream &operator<<(std::ostream &os, const MN &bn);

private:
    std::unordered_map<const Variable*,std::unordered_set<const Variable*>> _neighbors;
};

}  // namespace bn

#endif
