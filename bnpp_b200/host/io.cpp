#include "io.hh"
#include "uai_parse.hpp"

#include <algorithm>
#include <cmath>
#include <iostream>
#include <vector>

namespace bn {

namespace {

// next whitespace-separated token; a token starting with '#' comments out the rest of its line
// (code/io.cpp:14-23)
bool next_token(std::ifstream &in, std::string &tok)
{
    while (in >> tok) {
        if (tok[0] != '#') return true;
        std::getline(in, tok);
    }
    return false;
}

unsigned next_unsigned(std::ifstream &in)
{
    std::string tok;
    next_token(in, tok);
    return (unsigned)std::stoi(tok);      // at end of file tok is empty and stoi throws, as in the reference (code/io.cpp:25-33)
}

double next_double(std::ifstream &in)
{
    std::string tok;
    next_token(in, tok);
    return std::stod(tok);                // a truncated table is an error, not zeros
}

// Well-formed files: one read, tokens scanned in place (uai_parse.hpp).  false = "not sure": the caller
// re-reads the file with the reference's token-at-a-time reader below.
template <class M>
bool load_fast(std::string &filename, M **model, const char *want, const char *other, int &rc)
{
    std::string buf;
    uai::Parsed p;
    if (!uai::slurp(filename, buf) || !uai::parse_model(buf.data(), buf.size(), p)) return false;
    if (p.type == other) {
        std::cerr << "Error: file " << filename << " is not a " << want << " net." << std::endl;
        rc = -2;
        return true;
    }
    std::vector<Variable*> variables;
    std::vector<Factor*> factors;
    for (unsigned id = 0; id < p.card.size(); ++id) variables.push_back(new Variable(id, p.card[id]));
    for (size_t f = 0; f < p.scopes.size(); ++f) {
        std::vector<const Variable*> scope;
        for (unsigned id : p.scopes[f]) scope.push_back(variables[id]);
        factors.push_back(new Factor(new Domain(scope), p.values[f], p.partition[f]));
    }
    if (p.type == want) *model = new M(filename, variables, factors);
    rc = 0;
    return true;
}

template <class M>
int load(std::string &filename, M **model, const char *want, const char *other)
{
    int rc = 0;
    if (load_fast(filename, model, want, other, rc)) return rc;
    std::ifstream in(filename);
    if (!in.is_open()) {
        std::cerr << "Error: couldn't read file " << filename << std::endl;
        return -1;
    }
    const std::string type = read_file_header(in);
    if (type == other) {
        // checked BEFORE building anything: the reference builds first and leaks (SURVEY A.2 v)
        std::cerr << "Error: file " << filename << " is not a " << want << " net." << std::endl;
        return -2;
    }
    std::vector<Variable*> variables;
    std::vector<Factor*> factors;
    read_variables(in, variables);
    read_factors(in, variables, factors);
    if (type == want) *model = new M(filename, variables, factors);
    return 0;
}

}  // namespace

std::string read_file_header(std::ifstream &in)
{
    std::string tok;
    next_token(in, tok);
    if (tok != "BAYES" && tok != "MARKOV")
        std::cerr << "ERROR! Expected 'BAYES' or 'MARKOV' file header, found: " << tok << std::endl;
    return tok;
}

void read_variables(std::ifstream &in, std::vector<Variable*> &variables)
{
    const unsigned n = next_unsigned(in);
    for (unsigned id = 0; id < n; ++id) variables.push_back(new Variable(id, next_unsigned(in)));
}

// scopes first, then the tables; each factor's partition is summed in file order (code/io.cpp:66-100)
void read_factors(std::ifstream &in, std::vector<Variable*> &variables, std::vector<Factor*> &factors)
{
    const unsigned n = next_unsigned(in);
    std::vector<Domain*> domains;
    for (unsigned i = 0; i < n; ++i) {
        const unsigned width = next_unsigned(in);
        std::vector<const Variable*> scope;
        for (unsigned j = 0; j < width; ++j) scope.push_back(variables[next_unsigned(in)]);
        domains.push_back(new Domain(scope));
    }
    for (unsigned i = 0; i < n; ++i) {
        const unsigned size = next_unsigned(in);
        std::vector<double> values;
        values.reserve(size);
        double partition = 0;
        for (unsigned j = 0; j < size; ++j) {
            values.push_back(next_double(in));
            partition += values.back();
        }
        factors.push_back(new Factor(domains[i], values, partition));
    }
}

int read_uai_model(std::string &filename, BN **model) { return load(filename, model, "BAYES", "MARKOV"); }

int read_uai_model(std::string &filename, MN **model) { return load(filename, model, "MARKOV", "BAYES"); }

// only a leading sample count of exactly 1 is honoured (code/io.cpp:157-180, SURVEY A.2 iv)
int read_uai_evidence(std::string &filename, std::unordered_map<unsigned,unsigned> &evidence)
{
    std::ifstream in(filename);
    if (!in.is_open()) {
        std::cerr << "Error: couldn't read file " << filename << std::endl;
        return -1;
    }
    if (next_unsigned(in) == 1) {
        const unsigned k = next_unsigned(in);
        for (unsigned i = 0; i < k; ++i) {
            const unsigned id = next_unsigned(in);
            evidence[id] = next_unsigned(in);
        }
    }
    return 0;
}

int write_uai_pr(const std::string &filename, double partition)
{
    std::ofstream out(filename);
    if (!out.is_open()) return -1;
    out << "PR" << std::endl << 1 << std::endl << std::log10(partition) << std::endl;
    return out.good() ? 0 : -1;
}

int write_uai_mpe(const std::string &filename, const std::vector<unsigned> &assignment)
{
    std::ofstream out(filename);
    if (!out.is_open()) return -1;
    out << "MPE" << std::endl << 1 << std::endl << assignment.size();
    for (unsigned x : assignment) out << " " << x;
    out << std::endl;
    return out.good() ? 0 : -1;
}

int write_uai_mar(const std::string &filename, const std::vector<const Factor*> &marginals,
                  const std::vector<unsigned> &cardinalities, const std::unordered_map<unsigned,unsigned> &evidence)
{
    std::ofstream out(filename);
    if (!out.is_open()) return -1;
    out << "MAR" << std::endl << 1 << std::endl << marginals.size() << std::endl;
    for (size_t v = 0; v < marginals.size(); ++v) {
        const unsigned card = v < cardinalities.size() ? cardinalities[v] : marginals[v]->size();
        out << card;
        const auto e = evidence.find((unsigned)v);
        if (e != evidence.end() || marginals[v]->size() != card) {
            // observed (BN::marginals / Model::marginals hand back the width-0 factor [1]): the indicator of its value
            for (unsigned i = 0; i < card; ++i) out << ' ' << ((e != evidence.end() && e->second == i) ? 1 : 0);
        } else {
            for (unsigned i = 0; i < card; ++i) out << ' ' << (*marginals[v])[i];
        }
        out << std::endl;
    }
    return out.good() ? 0 : -1;
}

int write_uai_evidence(const std::string &filename, const std::unordered_map<unsigned,unsigned> &evidence)
{
    std::ofstream out(filename);
    if (!out.is_open()) return -1;
    std::vector<std::pair<unsigned,unsigned>> ev(evidence.begin(), evidence.end());
    std::sort(ev.begin(), ev.end());
    out << 1 << std::endl << ev.size();
    for (const auto &e : ev) out << ' ' << e.first << ' ' << e.second;
    out << std::endl;
    return out.good() ? 0 : -1;
}

}  // namespace bn
