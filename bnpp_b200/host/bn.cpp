// `bn` -- Bayesian-network CLI on the B200 factor-algebra library.
// Same flags, prompt commands and text output as the reference tool (code/bn.cpp:63-549);
// everything it prints is computed through bn::BN, i.e. on the GPU.
#include "io.hh"
#include "utils.hh"
#include "model.hh"
#include "graph.hh"
using namespace bn;

#include <cassert>
#include <cstring>
#include <functional>
#include <iostream>
#include <regex>
#include <string>
#include <unordered_map>
#include <vector>
using namespace std;

static unordered_map<string,bool> options;
static vector<string> positional;
static BN *model;
static unordered_map<unsigned,unsigned> evidence;

struct Flag { const char *text; const char *key; const char *help; };
static const Flag kTasks[] = {
    {"-pr", "partition", "solve partition task"},
    {"-mar", "marginals", "solve marginals task"},
    {"-mpe", "mpe", "solve most probable explanation task"},
};
static const Flag kOptions[] = {
    {"-ls", "logical-sampling", "compute partition using logical sampling"},
    {"-lw", "likelihood-weighting", "compute partition using (bounded-variance) likelihood weighting"},
    {"-gs", "gibbs-sampling", "compute partition using gibbs sampling"},
    {"-sp", "sum-product", "compute marginals using sum-product in factor graphs"},
    {"-ve", "variable-elimination", "compute inference using variable elimination"},
    {"-mf", "min-fill", "variable elimination using min-fill heuristic"},
    {"-wmf", "weighted-min-fill", "variable elimination using weighted min-fill heuristic"},
    {"-md", "min-degree", "variable elimination using min-degree heuristic"},
    {"-bb", "bayes-ball", "variable elimination using bayes-ball"},
    {"-h", "help", "display help information"},
    {"-v", "verbose", "verbose"},
};

static void usage(const char *progname)
{
    cout << "usage: " << progname << " /path/to/model.uai [/path/to/evidence.uai.evid TASK] [OPTIONS]" << endl << endl;
    cout << "TASK:" << endl;
    for (const Flag &f : kTasks) cout << f.text << "\t" << f.help << endl;
    cout << endl << "OPTIONS:" << endl;
    for (const Flag &f : kOptions) cout << f.text << "\t" << f.help << endl;
}

static void read_parameters(int argc, char *argv[])
{
    for (const Flag &f : kTasks) options[f.key] = false;
    for (const Flag &f : kOptions) options[f.key] = false;
    for (int i = 1; i < argc; ++i) {
        const string param(argv[i]);
        bool known = false;
        for (const Flag &f : kTasks) if (param == f.text) { options[f.key] = true; known = true; }
        for (const Flag &f : kOptions) if (param == f.text) { options[f.key] = true; known = true; }
        if (known) continue;
        if (param[0] == '-') {
            cerr << "Error: invalid option `" << param << "'." << endl << endl;
            usage(argv[0]);
            exit(-1);
        }
        positional.push_back(param);
    }
}

static void print_evidence(const char *sep)
{
    cout << ">> Evidence:" << endl;
    for (const auto &e : evidence) cout << "Variable = " << e.first << sep << "Value = " << e.second << endl;
    cout << endl;
}

static void execute_partition()
{
    double uptime;
    if (options["verbose"]) cout << ">> Computing partition for evidence ..." << endl;
    const double p = model->partition(evidence, options, uptime);
    cout << ">> Partition = " << p << endl;
    cout << ">> Executed in " << uptime << "ms." << endl << endl;
}

static void execute_mpe()
{
    double uptime;
    vector<unsigned> assignment;
    const double p = model->mpe(evidence, options, assignment, uptime);
    cout << ">> MPE = " << p << endl;
    cout << ">> Assignment =";
    for (unsigned x : assignment) cout << " " << x;
    cout << endl;
    cout << ">> Executed in " << uptime << "ms." << endl << endl;
}

// prompt command `map <id>[, <id>...]`: marginal MAP of those variables under the file's evidence and ordering flags
static void execute_map(const smatch &m)
{
    vector<unsigned> map_vars;
    const string list = m[1];
    const regex id("[0-9]+");
    for (sregex_iterator it(list.begin(), list.end(), id), end; it != end; ++it) map_vars.push_back(stoi(it->str()));
    double uptime;
    vector<unsigned> assignment;
    const double p = model->map(map_vars, evidence, options, assignment, uptime);
    sort(map_vars.begin(), map_vars.end());
    cout << ">> MAP = " << p << endl;
    cout << ">> Assignment =";
    for (unsigned v : map_vars) cout << " " << v << "=" << assignment[v];
    cout << endl;
    cout << ">> Executed in " << uptime << "ms." << endl << endl;
}

static void execute_marginals()
{
    double uptime;
    vector<const Factor*> marginals = model->marginals(evidence, options, uptime);
    cout << ">> Marginals:" << endl;
    for (const Factor *pf : marginals) {
        cout << *pf << endl;
        delete pf;
    }
    if (options["verbose"] && !evidence.empty()) print_evidence(", ");
    cout << ">> Executed in " << uptime << "ms." << endl << endl;
}

static string strip_spaces(const string &s)
{
    string o;
    for (char c : s) if (!isspace((unsigned char)c)) o += c;
    return o;
}

static void execute_query(const smatch &m)
{
    const string target = strip_spaces(m[1]), given = strip_spaces(m[3]);
    unordered_set<const Variable*> target_vars, evidence_vars;
    parse_vars_set(model, target, target_vars);
    if (!given.empty()) parse_vars_set(model, given, evidence_vars);
    double uptime;
    Factor q;
    if (options["variable-elimination"]) q = model->query_ve(target_vars, evidence_vars, options, uptime);
    else q = model->query(target_vars, evidence_vars, options, uptime);
    cout << (given.empty() ? "P(" + target + ") =" : "P(" + target + "|" + given + ") =") << endl;
    cout << q;
    cout << ">> Executed in " << uptime << "ms." << endl << endl;
}

static void execute_independence(const smatch &m)
{
    const Variable *a = model->variables()[stoi(m[1])];
    const Variable *b = model->variables()[stoi(m[2])];
    unordered_set<const Variable*> given;
    const string e = m[4];
    if (!e.empty()) parse_vars_set(model, strip_spaces(e), given);
    cout << (model->m_separated(a, b, given, options["verbose"]) ? "true" : "false") << endl << endl;
}

static void print_ids(const char *title, const vector<const Variable*> &vars)
{
    cout << title;
    for (const Variable *pv : vars) cout << " " << pv->id();
    cout << endl << endl;
}

static void execute_blanket(const smatch &m)
{
    const unsigned index = stoi(m[1]);
    assert(index < model->variables().size());
    const unordered_set<const Variable*> mb = model->markov_blanket(model->variables()[index]);
    print_ids(">> Markov blanket:", vector<const Variable*>(mb.begin(), mb.end()));
}

static void execute_width()
{
    vector<const Variable*> vars(model->variables().begin(), model->variables().end());
    vector<const Factor*> factors(model->factors().begin(), model->factors().end());
    Graph g(vars, factors);
    cout << endl;
    cout << ">> Original elimination order          (width = " << g.order_width(vars) << ")" << endl;
    if (options["verbose"]) {
        cout << "  ";
        for (const Variable *pv : vars) cout << " " << pv->id();
        cout << endl << endl;
    }
    struct { const char *key; const char *label; } rows[] = {
        {"min-degree", ">> Min-degree elimination order        (width = "},
        {"min-fill", ">> Min-fill elimination order          (width = "},
        {"weighted-min-fill", ">> Weighted min-fill elimination order (width = "},
    };
    for (int r = 0; r < 3; ++r) {
        unordered_map<string,bool> o;
        o[rows[r].key] = true;
        unsigned width = 0;
        const vector<unsigned> ids = g.ordering(vars, width, o);
        cout << rows[r].label << width << ")" << endl;
        if (options["verbose"]) {
            cout << "  ";
            for (unsigned id : ids) cout << " " << id;
            cout << endl;
            if (r < 2) cout << endl;
        }
    }
    cout << endl;
}

static void execute_stats()
{
    const vector<Variable*> &variables = model->variables();
    const vector<Factor*> &factors = model->factors();
    unsigned nroots = 0, nleaves = 0, nalone = 0, maxcard = 0, maxparents = 0, maxchildren = 0, nparams = 0;
    for (const Variable *pv : variables) {
        const unsigned np = model->parents(pv).size(), nc = model->children(pv).size();
        maxcard = max(maxcard, pv->size());
        nroots += np == 0;
        nleaves += nc == 0;
        nalone += np == 0 && nc == 0;
        maxparents = max(maxparents, np);
        maxchildren = max(maxchildren, nc);
    }
    double minprob = 1.0, maxprob = 0.0, maxpartition = 0.0;
    for (const Factor *pf : factors) {
        nparams += pf->size() - 1;
        maxpartition = max(maxpartition, pf->partition());
        for (unsigned i = 0; i < pf->size(); ++i) {
            minprob = min(minprob, (*pf)[i]);
            maxprob = max(maxprob, (*pf)[i]);
        }
    }
    cout << ">> Stats (" << model->name() << ")" << endl;
    cout << ">> variables = " << variables.size() << ", factors = " << factors.size() << endl;
    cout << ">> roots = " << nroots << ", leaves = " << nleaves << ", disconnected = " << nalone << endl;
    cout << ">> max number of parents = " << maxparents << ", max number of children = " << maxchildren << endl;
    cout << ">> max domain size = " << maxcard << endl;
    cout << ">> number of parameters = " << nparams << endl;
    cout << ">> lowest probability = " << minprob << ", highest probability = " << maxprob << endl;
    cout << ">> max partition = " << maxpartition << endl << endl;
}

static void print_help()
{
    cout << endl << "COMMANDS:" << endl << endl;
    cout << "query <target> [ | evidence]  to compute a (conditional) distribution" << endl;
    cout << "ind   <target> [ | evidence]  to check an independence assertion" << endl;
    cout << "stats                         to get summary information about the model" << endl;
    cout << "roots                         to get the list of root nodes" << endl;
    cout << "leaves                        to get the list of leaf nodes" << endl;
    cout << "blanket <var>                 to get the markov blanket of var" << endl;
    cout << "width                         to get elimination order width for ordering heuristics" << endl;
    cout << "help                          to display this information" << endl;
    cout << "quit                          to exit the prompt" << endl << endl;
}

static void prompt()
{
    struct Command { regex pattern; function<void(const smatch &)> run; };
    const vector<Command> commands = {
        {regex("query ([^\\|]+)\\s*(\\|\\s*(.*))?"), execute_query},
        {regex("ind ([0-9]+)\\s*,\\s*([0-9]+)\\s*(\\|\\s*([0-9]+(\\s*,\\s*[0-9]+)*))?"), execute_independence},
        {regex("stats"), [](const smatch &) { execute_stats(); }},
        {regex("roots"), [](const smatch &) { print_ids(">> Roots:", model->roots()); }},
        {regex("leaves"), [](const smatch &) { print_ids(">> Leaves:", model->leaves()); }},
        {regex("blanket\\s*([0-9]+)"), execute_blanket},
        {regex("width"), [](const smatch &) { execute_width(); }},
        {regex("map\\s+([0-9]+(\\s*,\\s*[0-9]+)*)"), execute_map},
        {regex("help"), [](const smatch &) { print_help(); }},
    };
    const regex quit("quit");
    cout << ">> Query prompt: (type a command or 'help' to list all commands)" << endl;
    while (cin) {
        cout << "? ";
        string line;
        getline(cin, line);
        if (regex_match(line, quit)) break;
        smatch m;
        bool done = false;
        for (const Command &c : commands)
            if (regex_match(line, m, c.pattern)) {
                c.run(m);
                done = true;
                break;
            }
        if (!done) cout << "Error: not a valid query." << endl << endl;
    }
}

int main(int argc, char *argv[])
{
    if (argc < 2) {
        usage(argv[0]);
        exit(1);
    }
    read_parameters(argc, argv);
    if (options["help"]) {
        usage(argv[0]);
        return 0;
    }
    string model_filename = positional[0];
    if (options["verbose"]) cout << ">> Reading file " << model_filename << " ..." << endl;
    if (read_uai_model(model_filename, &model)) return -1;
    if (options["verbose"]) cout << *model << endl;
    if (positional.size() > 1) {
        string evidence_filename = positional[1];
        if (options["verbose"]) cout << ">> Reading file " << evidence_filename << " ..." << endl;
        if (read_uai_evidence(evidence_filename, evidence)) return -2;
        if (options["verbose"] && !evidence.empty()) print_evidence(",\t");
    }
    if (options["partition"] || options["marginals"] || options["mpe"]) {
        if (options["partition"]) execute_partition();
        if (options["marginals"]) execute_marginals();
        if (options["mpe"]) execute_mpe();
    } else {
        prompt();
    }
    delete model;
    return 0;
}
