// Teuchos::ParameterList stand-in + XML reader for the subset used by testSuite/*.xml
// (<ParameterList name>, <Parameter name type value/>; types bool/int/double/string).
// `get(name, default)` stores the default like Teuchos does: the reference relies on that
// (e.g. src/HYMLS_BasePartitioner.cpp:139-141, 237-243).
#pragma once
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace hymls {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

class ParameterList {
 public:
  enum Kind { BOOL, INT, DOUBLE, STRING };
  struct Value {
    Kind kind = INT;
    bool b = false;
    long long i = 0;
    double d = 0;
    std::string s;
  };

  bool isParameter(const std::string& n) const { return vals_.count(n) != 0; }
  Kind kindOf(const std::string& n) const { return vals_.at(n).kind; }  // the parameter must exist
  bool isSublist(const std::string& n) const { return subs_.count(n) != 0; }
  ParameterList& sublist(const std::string& n) {
    auto it = subs_.find(n);
    if (it == subs_.end()) {
      order_.push_back(n);
      it = subs_.emplace(n, std::make_shared<ParameterList>()).first;
    }
    return *it->second;
  }
  const ParameterList* sublistPtr(const std::string& n) const {
    auto it = subs_.find(n);
    return it == subs_.end() ? nullptr : it->second.get();
  }

  int get(const std::string& n, int def);
  bool get(const std::string& n, bool def);
  double get(const std::string& n, double def);
  std::string get(const std::string& n, const char* def);
  std::string get(const std::string& n, const std::string& def) { return get(n, def.c_str()); }

  void set(const std::string& n, int v);
  void set(const std::string& n, bool v);
  void set(const std::string& n, double v);
  void set(const std::string& n, const char* v);

  ParameterList deepCopy() const;
  std::vector<std::string> parameterNames() const;
  std::vector<std::string> sublistNames() const;

  static ParameterList fromXml(const std::string& xml);
  // Teuchos XML of the list (writeParameterListToXmlOStream): entries in insertion order, sublists nested
  std::string toXml(const std::string& name = "HYMLS", int indent = 0) const;

 private:
  Value& slot(const std::string& n) {
    if (!vals_.count(n)) order_.push_back(n);
    return vals_[n];
  }
  std::map<std::string, Value> vals_;
  std::map<std::string, std::shared_ptr<ParameterList>> subs_;
  std::vector<std::string> order_;
};

}  // namespace hymls
