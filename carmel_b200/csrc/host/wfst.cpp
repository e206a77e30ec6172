// wfst.cpp -- weights, alphabets, WFST text reader / writer, reduce, corpus reader (host side).
#include <algorithm>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>

#include "carmel_host.hpp"

namespace cb {

static const double kLn10 = 2.30258509299404568402;

// ---- weights ---------------------------------------------------------------------------------------
bool parse_weight(const char* b, double& out) {  // legal forms: weight.h:18-27
  const char* end = b + std::strlen(b);
  char* e;
  if (b == end) return false;
  if (end - b > 2 && b[0] == 'e' && b[1] == '^') {
    out = std::strtod(b + 2, &e);
    return e == end;
  }
  if (end - b > 3 && b[0] == '1' && b[1] == '0' && b[2] == '^') {
    out = std::strtod(b + 3, &e) * kLn10;
    return e == end;
  }
  const double d = std::strtod(b, &e);
  if (e == b) return false;
  if (e == end) {
    out = d > 0 ? std::log(d) : kNegInf;
    return true;
  }
  if (!std::strcmp(e, "ln")) {
    out = d;
    return true;
  }
  if (!std::strcmp(e, "log")) {
    out = d * kLn10;
    return true;
  }
  return false;
}

static std::string fmt(double d, int prec) {
  std::ostringstream o;
  o.precision(prec);
  o << d;
  return o.str();
}

std::string format_weight(double w, WeightFormat const& f) {
  if (!(w > kNegInf)) return "0";
  const bool fits = w < 82. && w > -82.;  // weight.h:112,266
  if ((f.thresh == WeightFormat::SOMETIMES && fits) || f.thresh == WeightFormat::NEVER) return fmt(std::exp(w), 15);
  if (f.base == WeightFormat::LN) return fmt(w, 15) + "ln";
  if (f.base == WeightFormat::LOG10) return fmt(w / kLn10, 15) + "log";
  return "e^" + fmt(w, 15);
}

std::string format_base2(double w) { return "2^" + fmt(w / std::log(2.), 6); }

double ln_add(double a, double b) {
  if (!(a > kNegInf)) return b;
  if (!(b > kNegInf)) return a;
  const double d = a - b;
  if (d > 36.) return a;
  if (d < -36.) return b;
  return d < 0 ? b + std::log1p(std::exp(d)) : a + std::log1p(std::exp(-d));
}

double ln_sub(double a, double b) {
  if (!(b > kNegInf)) return a;
  const double rd = b - a;
  if (rd >= 0) return kNegInf;
  if (rd < -36.) return a;
  return a + std::log1p(-std::exp(rd));
}

// ---- alphabet --------------------------------------------------------------------------------------
Alphabet::Alphabet() {
  index_of("*e*");  // 0 = epsilon, 1 = wildcard (graehl/shared/arc.h:45-46)
  index_of("*w*");
}
uint32_t Alphabet::index_of(std::string const& s) {
  auto it = idx.find(s);
  if (it != idx.end()) return it->second;
  const uint32_t i = (uint32_t)names.size();
  names.push_back(s);
  idx.emplace(s, i);
  return i;
}
int Alphabet::find(std::string const& s) const {
  auto it = idx.find(s);
  return it == idx.end() ? -1 : (int)it->second;
}

// ---- tokenizer shared by the WFST and corpus readers (wfstio.cc:95-150) ---------------------------
struct Scanner {
  std::istream& in;
  explicit Scanner(std::istream& i) : in(i) {}
  // next non-blank character without consuming it; 0 at end of input
  char peek() {
    char c;
    if (!(in >> c)) return 0;
    in.unget();
    return c;
  }
  bool take(char want) {
    char c;
    return (in >> c) && c == want;
  }
  bool token(std::string& out) {
    out.clear();
    char c;
    if (!(in >> c)) return false;
    if (c == '(' || c == ')') return false;
    out.push_back(c);
    if (c == '"') {  // quoted: up to the next unescaped quote
      bool esc = false;
      for (char s; in.get(s);) {
        out.push_back(s);
        if (s == '"' && !esc) return true;
        esc = (s == '\\') ? !esc : false;
      }
      return false;
    }
    if (c == '*') {  // *special* symbols are case-folded
      for (char s; in.get(s);) {
        if (s == '*') {
          out.push_back(s);
          return true;
        }
        out.push_back((char)std::tolower((unsigned char)s));
      }
      return false;
    }
    for (char s; in.get(s);) {
      if (s == ' ' || s == '\t' || s == '\n') break;
      if (s == '!' || s == ')') {
        in.unget();
        break;
      }
      out.push_back(s);
    }
    if (out.size() > 1 && out.back() == '\r') out.pop_back();
    return true;
  }
  void skip_comments() {
    for (;;) {
      char c = peek();
      if (c != '%') return;
      std::string rest;
      std::getline(in, rest);
    }
  }
};

// ---- WFST -----------------------------------------------------------------------------------------
Wfst::Wfst() {
  alph[0] = std::make_shared<Alphabet>();
  alph[1] = std::make_shared<Alphabet>();
}
size_t Wfst::num_arcs() const {
  size_t n = 0;
  for (auto const& s : states) n += s.size();
  return n;
}
std::string Wfst::state_name(uint32_t i) const {
  if (named && i < state_names.size()) return state_names[i];
  return std::to_string(i);
}
void Wfst::arc_offsets(std::vector<uint32_t>& off) const {
  off.resize(states.size() + 1);
  off[0] = 0;
  for (size_t s = 0; s < states.size(); ++s) off[s + 1] = off[s] + (uint32_t)states[s].size();
}

// Grammar (carmel/doc/FORMATS:50-98):  final  ( src ( dst [in [out]] [weight] [!|!N] ) ... ) ...
// with optional extra nesting "(dst (in out w) (in out w))".
bool Wfst::read(std::istream& is, bool always_named) {
  Scanner sc(is);
  Alphabet &ain = *alph[0], &aout = *alph[1];
  valid = false;
  named = true;
  sc.skip_comments();
  std::string final_name, tok, tok2, tok3;
  if (!sc.token(final_name)) return false;
  if (!always_named) {
    named = !std::all_of(final_name.begin(), final_name.end(), [](char c) { return std::isdigit((unsigned char)c); });
  }
  auto state_index = [&](std::string const& name, uint32_t& out) -> bool {
    if (!named) {  // wfstio.cc:313-327: integer state names are indices
      char* e;
      const unsigned long v = std::strtoul(name.c_str(), &e, 10);
      if (name.empty() || *e) return false;
      if (v >= states.size()) states.resize(v + 1);
      out = (uint32_t)v;
      return true;
    }
    auto it = state_idx.find(name);
    if (it == state_idx.end()) {
      it = state_idx.emplace(name, (uint32_t)state_names.size()).first;
      state_names.push_back(name);
      states.emplace_back();
    }
    out = it->second;
    return true;
  };
  if (!named && !state_index(final_name, final_state)) return false;

  auto at_end_of_arc = [&](char c) { return c == ')' || c == '!'; };
  // one "[in [out]] [weight] [!group]" body; the opening parenthesis (if any) is already consumed
  auto read_arc_body = [&](uint32_t src, uint32_t dst) -> bool {
    Arc a{kEps, kEps, dst, 0., kNoGroup};
    char c = sc.peek();
    if (!c) return false;
    if (!at_end_of_arc(c)) {
      if (!sc.token(tok)) return false;
      if (!(c = sc.peek())) return false;
      if (at_end_of_arc(c)) {  // "weight" or "symbol"
        if (!parse_weight(tok.c_str(), a.ln_w)) {
          a.in = ain.index_of(tok);
          a.out = aout.index_of(tok);
          a.ln_w = 0;
        }
      } else {
        a.in = ain.index_of(tok);
        if (!sc.token(tok2)) return false;
        if (!(c = sc.peek())) return false;
        if (at_end_of_arc(c)) {  // "iosymbol weight" or "in out"
          if (parse_weight(tok2.c_str(), a.ln_w))
            a.out = aout.index_of(tok);
          else {
            a.out = aout.index_of(tok2);
            a.ln_w = 0;
          }
        } else {  // "in out weight"
          a.out = aout.index_of(tok2);
          if (!sc.token(tok3) || !parse_weight(tok3.c_str(), a.ln_w)) return false;
          if (!(c = sc.peek()) || !at_end_of_arc(c)) return false;
        }
      }
    }
    if (sc.peek() == '!') {
      sc.take('!');
      c = sc.peek();
      if (std::isdigit((unsigned char)c)) {
        unsigned g;
        if (!(is >> g)) return false;
        a.group = g;
      } else
        a.group = kLocked;
    }
    states[src].push_back(a);
    return true;
  };

  for (;;) {
    sc.skip_comments();
    char c = sc.peek();
    if (!c) break;
    if (!sc.take('(')) return false;
    uint32_t src, dst;
    if (!sc.token(tok) || !state_index(tok, src)) return false;
    for (;;) {  // destinations
      c = sc.peek();
      if (!c) return false;
      if (c == ')') break;
      const bool dest_paren = (c == '(');
      if (dest_paren) sc.take('(');
      if (!sc.token(tok) || !state_index(tok, dst)) return false;
      for (;;) {  // arcs to this destination
        c = sc.peek();
        if (!c) return false;
        const bool arc_paren = (c == '(');
        if (arc_paren) sc.take('(');
        if (!read_arc_body(src, dst)) return false;
        if (!arc_paren) break;
        if (!sc.take(')')) return false;
        if (sc.peek() == ')') break;
      }
      if (!dest_paren) break;
      if (!sc.take(')')) return false;
    }
    if (!sc.take(')')) return false;
  }
  if (!named) {
    valid = final_state < states.size();
    return valid;
  }
  auto it = state_idx.find(final_name);
  if (it == state_idx.end()) {
    std::cout << "\nFinal state named " << final_name << " not found.\n";
    return false;
  }
  final_state = it->second;
  valid = true;
  return true;
}

bool Wfst::read_file(std::string const& path, bool always_named) {
  std::ifstream f(path);
  return f && read(f, always_named);
}

void Wfst::write(std::ostream& os, bool full, bool onearc, bool include_zero, WeightFormat const& wf) const {
  if (!valid) return;  // wfstio.cc:594-625
  os << state_name(final_state);
  for (uint32_t s = 0; s < num_states(); ++s) {
    if (!onearc) os << "\n(" << state_name(s);
    for (Arc const& a : states[s]) {
      if (!include_zero && !(a.ln_w > kNegInf)) continue;
      if (onearc) os << "\n(" << state_name(s);
      os << " (" << state_name(a.dest);
      if (full || a.in || a.out) {
        std::string const &il = alph[0]->names[a.in], &ol = alph[1]->names[a.out];
        os << ' ' << il;
        if (full || il != ol) os << ' ' << ol;
      }
      if (full || a.group != kNoGroup || a.ln_w != 0.) os << ' ' << format_weight(a.ln_w, wf);
      if (a.group != kNoGroup) {
        os << '!';
        if (a.group != kLocked) os << a.group;
      }
      os << ')';
      if (onearc) os << ')';
    }
    if (!onearc) os << ')';
  }
  os << '\n';
}

// Keep only states both reachable from the start and co-reachable from the final state, preserving
// relative order; then drop *e*:*e* self loops (fst.cc:468-545, state.h:280-289).
void Wfst::reduce() {
  if (!valid) {
    states.clear();
    return;
  }
  const uint32_t n = num_states();
  std::vector<uint32_t> roff(n + 1, 0), rsrc;
  for (auto const& st : states)
    for (Arc const& a : st) ++roff[a.dest + 1];
  for (uint32_t i = 0; i < n; ++i) roff[i + 1] += roff[i];
  rsrc.resize(roff[n]);
  {
    std::vector<uint32_t> cur(roff.begin(), roff.end() - 1);
    for (uint32_t s = 0; s < n; ++s)
      for (Arc const& a : states[s]) rsrc[cur[a.dest]++] = s;
  }
  std::vector<char> fwd(n, 0), bwd(n, 0);
  std::vector<uint32_t> stack{0};
  fwd[0] = 1;
  while (!stack.empty()) {
    const uint32_t s = stack.back();
    stack.pop_back();
    for (Arc const& a : states[s])
      if (!fwd[a.dest]) {
        fwd[a.dest] = 1;
        stack.push_back(a.dest);
      }
  }
  stack.push_back(final_state);
  bwd[final_state] = 1;
  while (!stack.empty()) {
    const uint32_t s = stack.back();
    stack.pop_back();
    for (uint32_t k = roff[s]; k < roff[s + 1]; ++k)
      if (!bwd[rsrc[k]]) {
        bwd[rsrc[k]] = 1;
        stack.push_back(rsrc[k]);
      }
  }
  std::vector<uint32_t> renum(n);
  uint32_t kept = 0;
  for (uint32_t i = 0; i < n; ++i) renum[i] = (fwd[i] && bwd[i]) ? kept++ : ~0u;
  if (!~renum[final_state] || !~renum[0]) {
    valid = false;
    states.clear();
    return;
  }
  if (kept != n) {
    std::vector<std::vector<Arc>> ns(kept);
    std::vector<std::string> nn;
    for (uint32_t i = 0; i < n; ++i) {
      if (!~renum[i]) continue;
      auto& dst = ns[renum[i]];
      for (Arc a : states[i])
        if (~renum[a.dest]) {
          a.dest = renum[a.dest];
          dst.push_back(a);
        }
      if (named && i < state_names.size()) nn.push_back(state_names[i]);
    }
    states.swap(ns);
    if (named) {
      state_names.swap(nn);
      state_idx.clear();
      for (uint32_t i = 0; i < state_names.size(); ++i) state_idx.emplace(state_names[i], i);
    }
    final_state = renum[final_state];
  }
  for (uint32_t s = 0; s < num_states(); ++s) {
    auto& st = states[s];
    st.erase(std::remove_if(st.begin(), st.end(), [s](Arc const& a) { return a.in == kEps && a.out == kEps && a.dest == s; }),
             st.end());
  }
}

// ---- corpus ----------------------------------------------------------------------------------------
void Corpus::count() {
  n_pairs = 0;
  total_weight = n_input = n_output = 0;
  for (auto const& e : examples) {
    n_input += e.in.size();
    n_output += e.out.size();
    total_weight += e.weight;
    ++n_pairs;
  }
}

static void symbols_of_line(std::string const& line, Alphabet& a, std::vector<uint32_t>& out) {
  std::istringstream is(line);
  Scanner sc(is);
  std::string t;
  while (sc.token(t)) out.push_back(a.index_of(t));
}

// optional weight line (first char a digit, '-', '.' or 'e'), input line, output line (train.cc:985-1025)
void Corpus::read(std::istream& in, Wfst& x) {
  std::string line;
  while (std::getline(in, line)) {
    Example e;
    const char c0 = line.empty() ? 0 : line[0];
    if (std::isdigit((unsigned char)c0) || c0 == '-' || c0 == '.' || c0 == 'e') {
      std::istringstream w(line);
      if (!(w >> e.weight)) {
        std::cerr << "Bad training example weight: " << line << std::endl;
        continue;
      }
      if (!std::getline(in, line)) break;
    }
    symbols_of_line(line, *x.alph[0], e.in);
    if (!std::getline(in, line)) {
      if (!e.in.empty()) std::cerr << "Incomplete input/output training pair: " << line << std::endl;
      break;
    }
    symbols_of_line(line, *x.alph[1], e.out);
    examples.push_back(std::move(e));
  }
  count();
}

void Corpus::read_strings(std::istream& in, Wfst& x, int tape) {
  std::string line;
  while (std::getline(in, line)) {
    Example e;
    symbols_of_line(line, *x.alph[tape], tape ? e.out : e.in);
    examples.push_back(std::move(e));
  }
  count();
}

}  // namespace cb
