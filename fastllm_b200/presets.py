"""config.json presets of the BASELINE.json models (sizes only), as the adapters' ConfigFile (llama.rs:17-29 etc.)."""
from .models import BertConfig, ConfigFile, LlamaWithConfig, MistralWithConfig, MixtralWithConfig, QwenWithConfig

# TinyLlama-1.1B-Chat: the shape llama.rs:125-145 hard-codes for its cache
TINYLLAMA = (LlamaWithConfig, ConfigFile(2048, 5632, 32000, 22, 32, 4, 1e-5, 10000.0, 2048))
# Mistral-7B-v0.1
MISTRAL_7B = (MistralWithConfig, ConfigFile(4096, 14336, 32000, 32, 32, 8, 1e-5, 10000.0, 32768, 4096))
# Qwen2.5-7B (adapter passes sliding_window.unwrap_or(4096), qwen.rs:49)
QWEN25_7B = (QwenWithConfig, ConfigFile(3584, 18944, 152064, 28, 28, 4, 1e-6, 1000000.0, 32768, None))

# Mixtral-8x7B-v0.1: Mistral-7B dims, 8 experts, top-2, rope theta 1e6 (no reference path; candle-transformers mixtral.rs)
MIXTRAL_8X7B = (MixtralWithConfig, ConfigFile(4096, 14336, 32000, 32, 32, 8, 1e-5, 1000000.0, 32768, 4096, num_local_experts=8,
                                              num_experts_per_tok=2))

PRESETS = {"tinyllama": TINYLLAMA, "mistral7b": MISTRAL_7B, "qwen25_7b": QWEN25_7B, "mixtral8x7b": MIXTRAL_8X7B}

# Mean-pooled BERT sentence encoders (MiniLMModel): all-MiniLM-L6-v2 (head_dim 32), and the BERT-base / -large shapes of e5 and gte
# (head_dim 64)
MINILM_L6 = BertConfig(384, 12, 6, 1536, 512, 1e-12, 30522)
BERT_BASE = BertConfig(768, 12, 12, 3072, 512, 1e-12, 30522)
BERT_LARGE = BertConfig(1024, 16, 24, 4096, 512, 1e-12, 30522)
BERT_PRESETS = {"minilm_l6": MINILM_L6, "bert_base": BERT_BASE, "bert_large": BERT_LARGE}
